"""Generate the golden vectors under tests/golden/ by running the REAL reference.

Run in the authoring container only (the reference tree is not available on the GPU box):

    PYTHONPATH=oracle/_shim:/root/reference python tests/golden/make_golden.py

`oracle/_shim` provides the three import shims the reference needs offline (package metadata,
`natsort`, `h5py`; SURVEY.md Appendix B).  Every fixture stores the inputs next to the reference's
outputs, all produced on CPU in float32 by deepinv v0.4.1 through its public API.  The fixtures pin
(1) the oracle restatement (tests/test_oracle_golden.py, CPU) and (2) the CUDA kernels
(tests/test_gpu_golden.py, `-m gpu`).
"""
from __future__ import annotations

import sys
import warnings
from pathlib import Path

import numpy as np
import torch

warnings.filterwarnings("ignore")
import deepinv as dinv  # noqa: E402  (the real reference)
from deepinv.optim import ADMM, HQS, PGD, FISTA  # noqa: E402
from deepinv.optim.data_fidelity import L2  # noqa: E402
from deepinv.optim.prior import PnP  # noqa: E402
from deepinv.physics import MRI, Blur, BlurFFT, MultiCoilMRI, Tomography  # noqa: E402
from deepinv.physics.generator import RandomMaskGenerator  # noqa: E402

OUT = Path(__file__).resolve().parent
assert dinv.__version__ == "0.4.1", dinv.__version__


PART_BYTES = 800_000  # raw array bytes beyond which a fixture is split over two files: each stays under 1 MB compressed


def save(name, **arrays):
    conv = {}
    for k, v in arrays.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        conv[k] = np.asarray(v)
    parts = [{}, {}]
    if sum(v.nbytes for v in conv.values()) > PART_BYTES:  # largest first, each into the lighter half; the second -> more/
        for k in sorted(conv, key=lambda k: -conv[k].nbytes):
            parts[sum(v.nbytes for v in parts[0].values()) > sum(v.nbytes for v in parts[1].values())][k] = conv[k]
    else:
        parts[0] = conv
    np.savez_compressed(OUT / f"{name}.npz", **parts[0])
    more = OUT / "more" / f"{name}.npz"
    if parts[1]:
        more.parent.mkdir(exist_ok=True)
        np.savez_compressed(more, **parts[1])
    else:
        more.unlink(missing_ok=True)
    print(f"{name}: {len(conv)} arrays, {sum(v.nbytes for v in conv.values()) / 1024:.0f} KiB")


def g(seed):
    return torch.Generator().manual_seed(seed)


def mri_fixtures():
    for tag, (B, H, W), kind in [("mri_16x12_full", (2, 16, 12), "full"), ("mri_32x32_lines", (3, 32, 32), "lines"),
                                 ("mri_17x11_odd", (2, 17, 11), "full"), ("mri_20x24_shared", (2, 20, 24), "shared")]:
        x = torch.randn(B, 2, H, W, generator=g(1))
        if kind == "lines":
            mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
        elif kind == "shared":
            mask = (torch.rand(1, 1, H, W, generator=g(2)) > 0.6).float()
        else:
            mask = (torch.rand(B, 2, H, W, generator=g(2)) > 0.5).float()
        phys = MRI(mask=mask, img_size=(2, H, W))
        y = phys.A(x)
        z = torch.randn(B, 2, H, W, generator=g(3))
        save(tag, x=x, mask=phys.mask, y=y, At=phys.A_adjoint(y), AtA=phys.A_adjoint_A(x), AAt=phys.A_A_adjoint(y),
             z=z, prox=phys.prox_l2(z, y, 0.7), dagger=phys.A_dagger(y), Vt=phys.V_adjoint(x), V=phys.V(x),
             At_mag=phys.A_adjoint(y, mag=True), gamma=np.float32(0.7))


def dynamic_fixtures():
    """SURVEY §8(f) item 3: DynamicMRI / SequentialMRI (mri.py:499-695)"""
    from deepinv.physics import DynamicMRI, SequentialMRI

    B, T, H, W = 2, 3, 16, 12
    x = torch.randn(B, 2, T, H, W, generator=g(1))
    z = torch.randn(B, 2, T, H, W, generator=g(3))
    for tag, mask in [("dynmri_batched", RandomMaskGenerator((2, T, H, W), acceleration=4, rng=g(0)).step(B)["mask"]),
                      ("dynmri_shared_thw", (torch.rand(T, H, W, generator=g(2)) > 0.5).float())]:
        phys = DynamicMRI(mask=mask, img_size=(2, T, H, W))
        y = phys.A(x)
        save(tag, x=x, mask_in=mask, mask=phys.mask, y=y, At=phys.A_adjoint(y), At_mag=phys.A_adjoint(y, mag=True),
             AtA=phys.A_adjoint_A(x), z=z, prox=phys.prox_l2(z, y, 0.7), dagger=phys.A_dagger(y), gamma=np.float32(0.7))
    # sequential: T disjoint line sets of one static image
    xs = torch.randn(B, 2, H, W, generator=g(4))
    cols = torch.randperm(W, generator=g(5))
    mask = torch.zeros(T, H, W)
    for t in range(T):
        mask[t, :, cols[t::T][:3]] = 1
    mask = mask[None, None].expand(B, 2, T, H, W).contiguous()  # the reference needs the mask batch to equal x's
    phys = SequentialMRI(mask=mask, img_size=(2, T, H, W))
    y = phys.A(xs)
    save("seqmri_lines", x=xs, mask_in=mask, mask=phys.mask, y=y, At=phys.A_adjoint(y),
         At_keep=phys.A_adjoint(y, keep_time_dim=True), dagger=phys.A_dagger(y))


def down_fixtures():
    """SURVEY §8(f) item 3: Downsampling (blur.py:15-440) and the filter constructors it uses"""
    from deepinv.physics import Downsampling
    from deepinv.physics import functional as dF

    save("filters", gaussian=dF.gaussian_blur(sigma=(2.0, 2.0)), gaussian_aniso=dF.gaussian_blur(sigma=(1.0, 2.5), angle=30.0),
         bilinear2=dF.bilinear_filter(2), bicubic2=dF.bicubic_filter(2), bicubic4=dF.bicubic_filter(4),
         sinc2=dF.sinc_filter(2, length=8), sinc3=dF.sinc_filter(3, length=12))
    B, C, H, W = 2, 3, 24, 32
    x = torch.rand(B, C, H, W, generator=g(21))
    z = torch.rand(B, C, H, W, generator=g(22))
    for tag, filt, factor, pad in [("down_gauss_f2_circular", "gaussian", 2, "circular"), ("down_bicubic_f4_circular", "bicubic", 4, "circular"),
                                   ("down_none_f2_circular", None, 2, "circular"), ("down_bilinear_f2_valid", "bilinear", 2, "valid"),
                                   ("down_sinc_f2_reflect", "sinc", 2, "reflect")]:
        phys = Downsampling(img_size=(C, H, W), filter=filt, factor=factor, padding=pad)
        y = phys.A(x)
        v = torch.rand(*y.shape, generator=g(23))
        arrs = dict(x=x, y=y, v=v, At=phys.A_adjoint(v), factor=np.int32(factor))
        if pad == "circular" and filt is not None:
            arrs.update(z=z, prox=phys.prox_l2(z, y, 1.5), gamma=np.float32(1.5))
        save(tag, **arrs)


def combine_fixtures():
    """§8(b): `__mul__` (composition) and `stack` of operators on the path"""
    from deepinv.physics import Downsampling

    B, C, H, W = 2, 1, 24, 32
    x = torch.rand(B, C, H, W, generator=g(31))
    z = torch.rand(B, C, H, W, generator=g(32))
    filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.5))
    blur = Blur(filter=filt, padding="circular")
    down = Downsampling(img_size=(C, H, W), filter="bilinear", factor=2, padding="circular")
    comp = down * blur  # y = down(blur(x))
    y = comp.A(x)
    v = torch.rand(*y.shape, generator=g(33))
    save("combine_down_blur", x=x, filt=filt, y=y, v=v, At=comp.A_adjoint(v), z=z, prox=comp.prox_l2(z, y, 2.0),
         gamma=np.float32(2.0))
    Bm, Hm, Wm = 2, 16, 20
    xm = torch.randn(Bm, 2, Hm, Wm, generator=g(34))
    zm = torch.randn(Bm, 2, Hm, Wm, generator=g(35))
    m1 = (torch.rand(Bm, 2, Hm, Wm, generator=g(36)) > 0.6).float()
    m2 = RandomMaskGenerator((2, Hm, Wm), acceleration=4, rng=g(0)).step(Bm)["mask"]
    st = MRI(mask=m1, img_size=(2, Hm, Wm)).stack(MRI(mask=m2, img_size=(2, Hm, Wm)))
    ys = st.A(xm)
    save("combine_stack_mri", x=xm, m1=m1, m2=m2, y0=ys[0], y1=ys[1], At=st.A_adjoint(ys), z=zm,
         prox=st.prox_l2(zm, ys, 0.9), gamma=np.float32(0.9), dagger=st.A_dagger(ys))


def maskgen_fixtures():
    """§8(f) item 4: the LAW of the reference's mask generators (inclusion frequencies, equispaced pattern set)"""
    from deepinv.physics.generator import EquispacedMaskGenerator, GaussianMaskGenerator

    W, N = 64, 6000
    out = {}
    for tag, cls, acc in [("random4", RandomMaskGenerator, 4), ("gauss4", GaussianMaskGenerator, 4), ("gauss8", GaussianMaskGenerator, 8)]:
        gen = cls((2, 8, W), acceleration=acc, rng=g(0))
        m = gen.step(N)["mask"]
        out[f"freq_{tag}"] = m[:, 0, 0].mean(0)
        out[f"count_{tag}"] = m[:, 0, 0].sum(-1).unique()
    out["n_rows"] = np.int64(N)
    gen = EquispacedMaskGenerator((2, 6, 8, W), acceleration=4, rng=g(0))
    pats = torch.unique(gen.step(200)["mask"][:, 0, :, 0], dim=0)  # (n_offsets, T, W)
    out["equi_patterns"] = pats
    save("maskgen_stats", **out)
    from deepinv.physics.generator import MotionBlurGenerator

    mb = MotionBlurGenerator((31, 31), rng=g(0))  # cfg5's PSF generator, seed 0
    save("motionblur_psf", filt=mb.step(3)["filter"], filt_l=mb.step(2, sigma=0.4, l=0.5, seed=7)["filter"])


def mri3d_fixture():
    B, D, H, W = 2, 6, 8, 12
    x = torch.randn(B, 2, D, H, W, generator=g(41))
    z = torch.randn(B, 2, D, H, W, generator=g(42))
    mask = (torch.rand(B, 1, D, H, W, generator=g(43)) > 0.5).float()
    phys = MRI(mask=mask, img_size=(2, D, H, W), three_d=True)
    y = phys.A(x)
    save("mri3d_6x8x12", x=x, mask_in=mask, mask=phys.mask, y=y, At=phys.A_adjoint(y), AtA=phys.A_adjoint_A(x), z=z,
         prox=phys.prox_l2(z, y, 0.7), dagger=phys.A_dagger(y), Vt=phys.V_adjoint(x), gamma=np.float32(0.7))


def multicoil_fixtures():
    B, N, H, W = 2, 3, 16, 20
    x = torch.randn(B, 2, H, W, generator=g(1))
    maps = torch.randn(B, N, H, W, generator=g(4), dtype=torch.complex64)
    maps = maps / maps.abs().pow(2).sum(1, keepdim=True).sqrt()
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
    phys = MultiCoilMRI(mask=mask, coil_maps=maps, img_size=(2, H, W))
    y = phys.A(x)
    save("mcmri_16x20", x=x, mask=phys.mask, maps_re=maps.real, maps_im=maps.imag, y=y, At=phys.A_adjoint(y),
         At_rss=phys.A_adjoint(y, rss=True))
    # shared (batch-1) maps, CG pseudo-inverse
    maps1 = maps[:1]
    phys = MultiCoilMRI(mask=torch.ones(H, W), coil_maps=maps1, img_size=(2, H, W))
    y = phys.A(x)
    save("mcmri_shared_dagger", x=x, mask=phys.mask, maps_re=maps1.real, maps_im=maps1.imag, y=y, At=phys.A_adjoint(y),
         dagger=phys.A_dagger(y))


def tomo_fixtures():
    for tag, W, nang, circle in [("tomo_16_a8", 16, 8, False), ("tomo_24_a10_circle", 24, 10, True), ("tomo_32_a12", 32, 12, False)]:
        x = torch.randn(2, 1, W, W, generator=g(5))
        phys = Tomography(angles=nang, img_width=W, circle=circle, normalize=False)
        y = phys.A(x)
        v = torch.randn(*y.shape, generator=g(6))
        physb = Tomography(angles=nang, img_width=W, circle=circle, normalize=False, adjoint_via_backprop=False)
        save(tag, x=x, angles=phys.angles, y=y.contiguous(), v=v, At=phys.A_adjoint(v), fbp=phys.A_dagger(y, fbp=True),
             At_irad=physb.A_adjoint(v), fbp_irad=physb.A_dagger(y, fbp=True), filt=phys.iradon.filter(y))
    # normalised operator: operator_norm comes from a seeded power iteration + global RNG -> stored
    torch.manual_seed(0)
    W, nang = 16, 8
    phys = Tomography(angles=nang, img_width=W, normalize=True)
    x = torch.randn(1, 1, W, W, generator=g(7))
    y = phys.A(x)
    save("tomo_16_norm", x=x, angles=phys.angles, operator_norm=phys.operator_norm, y=y.contiguous(), At=phys.A_adjoint(y),
         fbp=phys.A_dagger(y, fbp=True), dagger=phys.A_dagger(y))


def fanbeam_fixtures():
    """§8(f) item 3: fan-beam Tomography (functional/radon.py:16-52; tomography.py fan_beam=True)"""
    for tag, W, circle, fp in [("fan_24_default", 24, False, None),
                               ("fan_20_circle_custom", 20, True, {"n_detector_pixels": 37, "detector_spacing": 0.31,
                                                                   "source_radius": 40.0, "detector_radius": 25.0})]:
        x = torch.randn(2, 1, W, W, generator=g(51))
        phys = Tomography(angles=9, img_width=W, circle=circle, fan_beam=True, fan_parameters=fp, normalize=False)
        y = phys.A(x)
        v = torch.randn(*y.shape, generator=g(52))
        save(tag, x=x, angles=phys.angles, y=y.contiguous(), v=v, At=phys.A_adjoint(v), fbp=phys.A_dagger(y, fbp=True))


def blur_fixtures():
    B, C, H, W = 2, 2, 17, 19
    x = torch.rand(B, C, H, W, generator=g(8))
    for hw in [(3, 3), (4, 4), (5, 3), (6, 5)]:
        filt = torch.rand(1, 1, *hw, generator=g(9))
        filt = filt / filt.sum()
        for pad in ["valid", "circular", "replicate", "reflect", "constant"]:
            phys = Blur(filter=filt, padding=pad)
            y = phys.A(x)
            v = torch.rand(*y.shape, generator=g(10))
            if pad == "circular" and 2 in hw:
                continue
            save(f"blur_{hw[0]}x{hw[1]}_{pad}", x=x, filt=filt, y=y, v=v, At=phys.A_adjoint(v))
    # per-sample, per-channel filters
    filt = torch.rand(B, C, 5, 5, generator=g(11))
    phys = Blur(filter=filt, padding="reflect")
    y = phys.A(x)
    save("blur_5x5_perbc_reflect", x=x, filt=filt, y=y, v=y, At=phys.A_adjoint(y))
    # CG prox on a circular blur
    filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.0))
    phys = Blur(filter=filt, padding="circular")
    y = phys.A(x)
    z = torch.rand(B, C, H, W, generator=g(12))
    save("blur_gauss_circular_prox", x=x, filt=filt, y=y, z=z, prox=phys.prox_l2(z, y, 2.0), gamma=np.float32(2.0),
         dagger=phys.A_dagger(y))


def blurfft_fixtures():
    for tag, (B, C, H, W), sig in [("blurfft_64_cfg1", (1, 1, 64, 64), 2.0), ("blurfft_18x20", (2, 3, 18, 20), 1.0),
                                   ("blurfft_15x16_odd", (2, 1, 15, 16), 1.0)]:
        x = torch.randn(B, C, H, W, generator=g(13))
        filt = dinv.physics.functional.gaussian_blur(sigma=(sig, sig))
        phys = BlurFFT(img_size=(C, H, W), filter=filt)
        y = phys.A(x)
        z = torch.randn(B, C, H, W, generator=g(14))
        save(tag, x=x, filt=filt, y=y, At=phys.A_adjoint(y), prox=phys.prox_l2(z, y, 1.5), z=z, gamma=np.float32(1.5),
             dagger=phys.A_dagger(y), mask=phys.mask, angle_re=phys.angle.real, angle_im=phys.angle.imag,
             Vt=phys.V_adjoint(x), Ut=phys.U_adjoint(x), AtA=phys.A_adjoint_A(x))
    # one filter PER SAMPLE (what MotionBlurGenerator.step(batch_size=B) hands out), with and without a channel dimension
    for tag, (B, C, H, W), fshape in [("blurfft_persample", (3, 2, 12, 14), (3, 1, 5, 5)), ("blurfft_persample_c", (2, 3, 10, 12), (2, 3, 3, 3))]:
        x = torch.randn(B, C, H, W, generator=g(33))
        filt = torch.rand(*fshape, generator=g(34)) + 0.1
        filt = filt / filt.sum(dim=(-2, -1), keepdim=True)
        phys = BlurFFT(img_size=(C, H, W), filter=filt)
        y = phys.A(x)
        z = torch.randn(B, C, H, W, generator=g(35))
        save(tag, x=x, filt=filt, y=y, At=phys.A_adjoint(y), prox=phys.prox_l2(z, y, 1.5), z=z, gamma=np.float32(1.5),
             dagger=phys.A_dagger(y), mask=phys.mask, angle_re=phys.angle.real, angle_im=phys.angle.imag,
             Vt=phys.V_adjoint(x), Ut=phys.U_adjoint(x), AtA=phys.A_adjoint_A(x))


def tiny_drunet(cin):
    torch.manual_seed(0)
    return dinv.models.DRUNet(in_channels=cin, out_channels=cin, nc=(8, 16, 32, 64), nb=2, pretrained=None).eval()


def tiny_dncnn(cin):
    torch.manual_seed(0)
    return dinv.models.DnCNN(in_channels=cin, out_channels=cin, depth=5, nf=8, pretrained=None).eval()


def sd_arrays(model, prefix):
    """state_dict entries of a fixture; the seed-0 tiny 2-channel DRUNet is stored once (drunet_tiny.npz) and referenced"""
    sd = model.state_dict()
    ref = OUT / "drunet_tiny.npz"
    if ref.exists():
        base = dict(np.load(ref))
        if (OUT / "more" / ref.name).exists():
            base.update(np.load(OUT / "more" / ref.name))
        keys = {f"sd__{k.replace('.', '__')}" for k in sd}
        if keys == {k for k in base if k.startswith("sd__")} and all(
                np.array_equal(base[f"sd__{k.replace('.', '__')}"], v.numpy()) for k, v in sd.items()):
            return {"sd_from": np.array("drunet_tiny")}
    return {f"{prefix}{k.replace('.', '__')}": v for k, v in sd.items()}


def model_fixtures():
    den = tiny_drunet(2)
    x = torch.randn(2, 2, 32, 40, generator=g(15))
    with torch.no_grad():
        out = den(x, 0.05)
        sig = torch.tensor([0.03, 0.1])
        out_b = den(x, sig)
        xs = torch.randn(1, 2, 20, 36, generator=g(16))  # needs the replicate-pad path
        out_s = den(xs, 0.05)
    save("drunet_tiny", x=x, out=out, sig=sig, out_b=out_b, xs=xs, out_s=out_s,
         **{f"sd__{k.replace('.', '__')}": v for k, v in den.state_dict().items()})
    dn = tiny_dncnn(1)
    x = torch.randn(2, 1, 24, 28, generator=g(17))
    with torch.no_grad():
        out = dn(x, 0.1)
    save("dncnn_tiny", x=x, out=out, **sd_arrays(dn, "sd__"))


def optim_fixtures():
    # cfg2 in miniature: MRI 32x32, 4x line mask, PnP-PGD + DRUNet
    B, H, W = 2, 32, 32
    x = torch.randn(B, 2, H, W, generator=g(1))
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
    phys = MRI(mask=mask, img_size=(2, H, W))
    y = phys(x)
    den = tiny_drunet(2)
    with torch.no_grad():
        pgd = PGD(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=4, early_stop=False)
        out_pgd = pgd(y, phys)
        pgd2 = PGD(data_fidelity=L2(), prior=PnP(den), max_iter=3, early_stop=False,
                   params_algo={"stepsize": 0.8, "g_param": 0.05, "lambda": 1.0, "beta": 0.9})
        out_pgd2 = pgd2(y, phys)
        hqs = HQS(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=3, early_stop=False)
        out_hqs = hqs(y, phys)
        admm = ADMM(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=3, early_stop=False)
        out_admm = admm(y, phys)
        fista = FISTA(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=3, early_stop=False)
        out_fista = fista(y, phys)
    save("optim_mri_tiny", x=x, mask=phys.mask, y=y, pgd=out_pgd, pgd_relax=out_pgd2, hqs=out_hqs, admm=out_admm,
         fista=out_fista, **sd_arrays(den, "sd__"))
    # cfg5 in miniature: circular Blur (CG prox) + DnCNN, PnP-ADMM
    B, C, H, W = 2, 1, 24, 28
    x = torch.rand(B, C, H, W, generator=g(18))
    filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.0))
    phys = Blur(filter=filt, padding="circular")
    y = phys(x)
    dn = tiny_dncnn(1)
    with torch.no_grad():
        admm = ADMM(data_fidelity=L2(), prior=PnP(dn), stepsize=1.0, sigma_denoiser=0.05, max_iter=3, early_stop=False)
        out = admm(y, phys)
    save("optim_blur_tiny", x=x, filt=filt, y=y, admm=out, **sd_arrays(dn, "sd__"))


def optim2_fixtures():
    """SURVEY §8(f) item 1: DRS, GD (explicit + RED priors), DPIR — same miniature MRI problem as optim_mri_tiny"""
    from deepinv.optim import DPIR, DRS, GD
    from deepinv.optim.prior import RED, Tikhonov

    B, H, W = 2, 32, 32
    x = torch.randn(B, 2, H, W, generator=g(1))
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
    phys = MRI(mask=mask, img_size=(2, H, W))
    y = phys(x)
    den = tiny_drunet(2)
    kw = dict(data_fidelity=L2(), early_stop=False)
    with torch.no_grad():
        drs = DRS(prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=3, **kw)(y, phys)
        drs_relax = DRS(prior=PnP(den), max_iter=3, g_first=True,
                        params_algo={"stepsize": 0.7, "g_param": 0.05, "lambda": 1.0, "beta": 0.8}, **kw)(y, phys)
        gd_tik = GD(prior=Tikhonov(), stepsize=0.5, lambda_reg=0.1, max_iter=4, **kw)(y, phys)
        gd_red = GD(prior=RED(den), stepsize=0.5, lambda_reg=0.3, sigma_denoiser=0.05, max_iter=3, **kw)(y, phys)
        dpir = DPIR(sigma=0.05, denoiser=den)(y, phys)
        # the same recipe on a non-decomposable operator: circular Blur -> CG prox inside HQS
        xb = torch.rand(2, 2, 24, 32, generator=g(18))
        filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.0))
        physb = Blur(filter=filt, padding="circular")
        yb = physb(xb)
        dpir_blur = DPIR(sigma=0.05, denoiser=den)(yb, physb)
    save("optim2_mri_tiny", x=x, mask=phys.mask, y=y, drs=drs, drs_relax=drs_relax, gd_tik=gd_tik, gd_red=gd_red,
         dpir=dpir, xb=xb, filt=filt, yb=yb, dpir_blur=dpir_blur, **sd_arrays(den, "sd__"))


def _grads(model, names=None):
    out = {}
    for k, p_ in model.named_parameters():
        if p_.grad is not None and (names is None or any(n in k for n in names)):
            out["grad__" + k.replace(".", "__")] = p_.grad.detach().clone()
    return out


def train_fixtures():
    """SURVEY §8(f) item 2: gradients of unfolded / deep-equilibrium models from the real reference (one backward each)"""
    from deepinv.optim import GD
    from deepinv.optim.prior import Tikhonov
    from deepinv.unfolded import unfolded_builder

    B, H, W = 2, 32, 32
    x = torch.randn(B, 2, H, W, generator=g(1))
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
    phys = MRI(mask=mask, img_size=(2, H, W))
    y = phys(x)
    # (1) unfolded PGD, 2 iterations, trainable stepsize + sigma + DRUNet weights
    den = tiny_drunet(2).train()
    model = unfolded_builder("PGD", params_algo={"stepsize": [1.0, 0.8], "g_param": [0.05, 0.03], "lambda": 1.0},
                             trainable_params=["stepsize", "g_param"], data_fidelity=L2(), prior=PnP(den), max_iter=2)
    out = model(y, phys)
    loss = ((out - x) ** 2).mean()
    loss.backward()
    save("train_unfolded_pgd_mri", x=x, mask=phys.mask, y=y, out=out, loss=loss, **sd_arrays(den, "sd__"), **_grads(model))
    # (2) deep equilibrium: PGD, 6 forward iterations, 8 backward fixed-point sweeps
    den = tiny_drunet(2).train()
    from deepinv.optim import DEQConfig
    deq = PGD(data_fidelity=L2(), prior=PnP(den), stepsize=0.9, sigma_denoiser=0.05, max_iter=6, early_stop=False,
              DEQ=DEQConfig(max_iter_backward=8), trainable_params=["stepsize"])
    out = deq(y, phys)
    loss = ((out - x) ** 2).mean()
    loss.backward()
    save("train_deq_pgd_mri", out=out, loss=loss, **_grads(deq))
    # (3) DEQ with an explicit prior (cheap enough for the CPU host-logic test): GD + Tikhonov, trainable stepsize / lambda
    deq2 = GD(data_fidelity=L2(), prior=Tikhonov(), stepsize=0.5, lambda_reg=0.2, max_iter=10, early_stop=False,
              DEQ=DEQConfig(max_iter_backward=12), trainable_params=["stepsize", "lambda"])
    out = deq2(y, phys)
    loss = ((out - x) ** 2).mean()
    loss.backward()
    save("train_deq_gd_tikhonov", out=out, loss=loss, **_grads(deq2))
    # (4) unfolded ADMM on a non-decomposable operator: circular Blur, CG prox with implicit-differentiation backward
    Bb, C, Hb, Wb = 2, 1, 24, 28
    xb = torch.rand(Bb, C, Hb, Wb, generator=g(18))
    filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.0))
    physb = Blur(filter=filt, padding="circular")
    yb = physb(xb)
    dn = tiny_dncnn(1).train()
    modelb = unfolded_builder("ADMM", params_algo={"stepsize": [1.0, 1.2], "g_param": 0.05, "lambda": 1.0, "beta": 1.0},
                              trainable_params=["stepsize"], data_fidelity=L2(), prior=PnP(dn), max_iter=2)
    out = modelb(yb, physb)
    loss = ((out - xb) ** 2).mean()
    loss.backward()
    save("train_unfolded_admm_blur", x=xb, filt=filt, y=yb, out=out, loss=loss, **sd_arrays(dn, "sd__"), **_grads(modelb))


def anderson_fixtures():
    """Anderson-accelerated fixed-point loops (fixed_point.py:117-260) from the real reference"""
    from deepinv.optim import GD, AndersonAccelerationConfig
    from deepinv.optim.prior import Tikhonov

    B, H, W = 2, 32, 32
    x = torch.randn(B, 2, H, W, generator=g(1))
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(B)["mask"]
    phys = MRI(mask=mask, img_size=(2, H, W))
    y = phys(x)
    den = tiny_drunet(2)
    with torch.no_grad():
        pgd = PGD(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=4, early_stop=False,
                  anderson_acceleration=True)(y, phys)
        gd = GD(data_fidelity=L2(), prior=Tikhonov(), stepsize=0.5, lambda_reg=0.2, max_iter=12, early_stop=False,
                anderson_acceleration=AndersonAccelerationConfig(history_size=3, beta=1.0, eps=1e-3))(y, phys)
    from deepinv.optim import BacktrackingConfig

    with torch.no_grad():
        gd_bt = GD(data_fidelity=L2(), prior=Tikhonov(), stepsize=2.5, lambda_reg=0.2, max_iter=8, early_stop=False,
                   backtracking=BacktrackingConfig(gamma=0.1, eta=0.5, max_iter=20))
        out_bt = gd_bt(y, phys)
        pgd_bt = PGD(data_fidelity=L2(), prior=Tikhonov(), stepsize=3.0, lambda_reg=0.5, max_iter=10, early_stop=False,
                     backtracking=True)
        out_pgd_bt = pgd_bt(y, phys)
    from deepinv.optim import PDCP

    with torch.no_grad():
        cp = PDCP(data_fidelity=L2(), prior=Tikhonov(), lambda_reg=0.3, stepsize=0.6, stepsize_dual=0.8, max_iter=6, early_stop=False)(y, phys)
        cp_g = PDCP(data_fidelity=L2(), prior=Tikhonov(), lambda_reg=0.3, stepsize=0.6, stepsize_dual=0.8, max_iter=6, early_stop=False,
                    g_first=True, K=phys.A, K_adjoint=phys.A_adjoint)(y, phys)
    save("optim_pdcp", cp=cp, cp_gfirst=cp_g)
    save("optim_anderson", x=x, mask=phys.mask, y=y, pgd=pgd, gd=gd, gd_bt=out_bt,
         gd_bt_step=np.float32(gd_bt.params_algo["stepsize"][0]), pgd_bt=out_pgd_bt,
         pgd_bt_step=np.float32(pgd_bt.params_algo["stepsize"][0]), **sd_arrays(den, "sd__"))


def ddrm_fixture():
    B, H, W = 2, 32, 32
    x = torch.randn(B, 2, H, W, generator=g(1)) * 0.3
    mask = RandomMaskGenerator((2, H, W), acceleration=4, rng=g(0)).step(1)["mask"]  # batch-1 mask (diffusion.py:173)
    phys = MRI(mask=mask, img_size=(2, H, W), noise_model=dinv.physics.GaussianNoise(sigma=0.02, rng=g(3)))
    y = phys(x)
    den = tiny_drunet(2)
    sigmas = np.linspace(1, 0, 5)
    noises = [torch.randn(B, 2, H, W, generator=g(100 + t)) for t in range(len(sigmas))]
    it = iter(noises)
    orig = torch.randn_like
    torch.randn_like = lambda t, **kw: next(it).to(t)
    try:
        model = dinv.sampling.DDRM(denoiser=den, sigmas=sigmas)
        out = model(y, phys)
    finally:
        torch.randn_like = orig
    save("ddrm_mri_tiny", x=x, mask=phys.mask, y=y, sigmas=sigmas, noises=torch.stack(noises), out=out,
         sigma_noise=np.float32(0.02), **sd_arrays(den, "sd__"))


def inpainting_fixture():
    """DDRM on Inpainting (the reference's own sampling test, tests/test_sampling.py:147-195) with a recorded noise sequence"""
    from deepinv.physics import Denoising, Inpainting

    B, H, W = 2, 32, 32
    x = torch.rand(B, 2, H, W, generator=g(71))
    mask = (torch.rand(1, 2, H, W, generator=g(72)) > 0.4).float()
    phys = Inpainting(img_size=(2, H, W), mask=mask, noise_model=dinv.physics.GaussianNoise(sigma=0.05, rng=g(73)))
    y = phys(x)
    den = tiny_drunet(2)
    sigmas = np.linspace(1, 0, 5)
    noises = [torch.randn(B, 2, H, W, generator=g(300 + t)) for t in range(len(sigmas))]
    it = iter(noises)
    orig = torch.randn_like
    torch.randn_like = lambda t, **kw: next(it).to(t)
    try:
        out = dinv.sampling.DDRM(denoiser=den, sigmas=sigmas)(y, phys)
        it = iter(noises)
        out_den = dinv.sampling.DDRM(denoiser=den, sigmas=sigmas)(y, Denoising(dinv.physics.GaussianNoise(sigma=0.05)))
    finally:
        torch.randn_like = orig
    save("ddrm_inpainting_tiny", x=x, mask=mask, y=y, sigmas=sigmas, noises=torch.stack(noises), out=out, out_denoising=out_den,
         At=phys.A_adjoint(y), prox=phys.prox_l2(x, y, 0.8), sigma_noise=np.float32(0.05), **sd_arrays(den, "sd__"))


def diffpir_fixture():
    """DiffPIR (sampling/diffusion.py:227-513) on a circular blur with a recorded noise sequence"""
    B, H, W = 2, 32, 32
    x = torch.rand(B, 1, H, W, generator=g(61))
    filt = dinv.physics.functional.gaussian_blur(sigma=(1.0, 1.0))
    phys = BlurFFT(img_size=(1, H, W), filter=filt, noise_model=dinv.physics.GaussianNoise(sigma=0.03, rng=g(62)))
    y = phys(x)
    den = tiny_drunet(1)
    noises = [torch.randn(B, 1, H, W, generator=g(200 + t)) for t in range(8)]
    it = iter(noises)
    orig = torch.randn_like
    torch.randn_like = lambda t, **kw: next(it).to(t)
    try:
        out = dinv.sampling.DiffPIR(den, L2(), sigma=0.03, max_iter=6, zeta=0.3, lambda_=7.0)(y, phys)
    finally:
        torch.randn_like = orig
    save("diffpir_blurfft_tiny", x=x, filt=filt, y=y, noises=torch.stack(noises), out=out, sigma_noise=np.float32(0.03),
         **sd_arrays(den, "sd__"))


def fastmri_fixture():
    """a synthetic HDF5-shaped fastMRI volume (h5py is absent here: the arrays ARE the file content) and what the reference's
    own code makes of every slice: MRIMixin.from_torch_complex (datasets/fastmri.py:475-478) and MRISliceTransform.__call__
    (:719-749) with a file mask / a scalar normalisation"""
    from deepinv.datasets.fastmri import MRISliceTransform
    from deepinv.physics.mri import MRIMixin

    gen = np.random.default_rng(0)
    D, N, H, W = 3, 2, 8, 6
    ks = (gen.standard_normal((D, N, H, W)) + 1j * gen.standard_normal((D, N, H, W))).astype(np.complex64)
    rss = gen.random((D, 4, 4)).astype(np.float32)
    mask = np.array([1, 0, 1, 1, 0, 1], dtype=np.float32)
    ks1 = (gen.standard_normal((2, 6, 6)) + 1j * gen.standard_normal((2, 6, 6))).astype(np.complex64)
    out = dict(vol_kspace=ks, vol_rss=rss, vol_mask=mask, vol1_kspace=ks1, acs=np.int64(2))
    mix = MRIMixin()
    for d in range(D):
        k = mix.from_torch_complex(torch.from_numpy(ks[d]).unsqueeze(0)).squeeze(0)
        t, k2, p = MRISliceTransform()(torch.from_numpy(rss[d]).unsqueeze(0), k, mask=torch.as_tensor(mask), seed="x", metadata={})
        out[f"k_{d}"], out[f"t_{d}"], out[f"m_{d}"] = k2, t, p["mask"]
        _, k3, _ = MRISliceTransform(normalize=2.0)(None, k, seed="x", metadata={})
        out[f"kn_{d}"] = k3
    for d in range(2):
        out[f"k1_{d}"] = mix.from_torch_complex(torch.from_numpy(ks1[d]).unsqueeze(0)).squeeze(0)
    save("fastmri_synth", **out)


def callers_fixture():
    """what the reference's own callers compute on the inputs of optim_mri_tiny / ddrm_mri_tiny / blur_gauss_circular_prox:
    PGD / HQS, DDRM with a closed-form toy denoiser and the least-squares solvers (optim/linear) — the yardsticks of
    tests/test_reference_callers_dropin.py"""
    from deepinv.optim import HQS
    from deepinv.optim.linear import least_squares

    out = {}
    o = np.load(OUT / "optim_mri_tiny.npz")
    y, mask = torch.from_numpy(o["y"]), torch.from_numpy(o["mask"])
    phys = MRI(mask=mask, img_size=(2, 32, 32))
    toy = lambda v, s: v * (1.0 - float(s))
    with torch.no_grad():
        out["pgd"] = PGD(data_fidelity=L2(), prior=PnP(tiny_drunet(2)), stepsize=1.0, sigma_denoiser=0.05, max_iter=2,
                         early_stop=False)(y, phys)
        out["hqs_toy"] = HQS(data_fidelity=L2(), prior=PnP(toy), stepsize=0.8, sigma_denoiser=0.05, max_iter=3,
                             early_stop=False)(y, phys)
    d = np.load(OUT / "ddrm_mri_tiny.npz")
    sig = float(d["sigma_noise"])
    physd = MRI(mask=torch.from_numpy(d["mask"]), img_size=(2, 32, 32), noise_model=dinv.physics.GaussianNoise(sigma=sig))
    it = iter(list(torch.from_numpy(d["noises"])))
    orig = torch.randn_like
    torch.randn_like = lambda t, **kw: next(it).to(t)
    try:
        out["ddrm_toy"] = dinv.sampling.DDRM(denoiser=lambda v, s: v * (1.0 / (1.0 + float(s))), sigmas=d["sigmas"])(
            torch.from_numpy(d["y"]), physd)
    finally:
        torch.randn_like = orig
    b = {k: torch.from_numpy(v) for k, v in np.load(OUT / "blur_gauss_circular_prox.npz").items()}
    gam = float(b["gamma"])
    circ, valid = Blur(filter=b["filt"], padding="circular"), Blur(filter=b["filt"], padding="valid")

    def ls(p, y_, z, gamma, solver, max_iter, tol, normal=True):
        kw = dict(AAT=p.A_A_adjoint, ATA=p.A_adjoint_A) if normal else {}
        return least_squares(p.A, p.A_adjoint, y_, z=z, init=z, gamma=gamma, parallel_dim=[0], max_iter=max_iter, tol=tol,
                             solver=solver, **kw)

    yv = valid.A(b["z"])
    out["valid_y"] = yv
    for solver in ("CG", "BiCGStab"):
        out[f"ls_{solver}"] = ls(circ, b["y"], b["z"], gam, solver, 25, 1e-5)
    out["ls_valid_BiCGStab"] = ls(valid, yv, b["z"], gam, "BiCGStab", 25, 1e-5)
    yl = valid.A(b["z"]) + 0.01 * torch.randn(valid.A(b["z"]).shape, generator=g(0))
    out["lsqr_y"] = yl
    out["lsqr_gamma2"] = ls(valid, yl, b["x"], 2.0, "lsqr", 30, 1e-6, normal=False)
    out["lsqr_gamma_batched"] = ls(valid, yl, b["x"], torch.tensor([0.5, 3.0]), "lsqr", 30, 1e-6, normal=False)
    out["minres_valid"] = ls(valid, yv, b["x"], 2.0, "minres", 30, 1e-6)
    out["minres_circular"] = ls(circ, b["y"], b["z"], 2.0, "minres", 15, 1e-6)
    save("reference_callers", **out)


if __name__ == "__main__":
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["mri", "multicoil", "tomo", "blur", "blurfft", "model", "optim", "ddrm", "optim2", "train", "dynamic", "down", "combine", "maskgen", "mri3d", "fan", "anderson", "diffpir", "inpainting", "fastmri", "callers"]
    table = {"mri": mri_fixtures, "multicoil": multicoil_fixtures, "tomo": tomo_fixtures, "blur": blur_fixtures,
             "blurfft": blurfft_fixtures, "model": model_fixtures, "optim": optim_fixtures, "ddrm": ddrm_fixture,
             "optim2": optim2_fixtures, "train": train_fixtures,
             "dynamic": dynamic_fixtures, "down": down_fixtures,
             "combine": combine_fixtures, "maskgen": maskgen_fixtures,
             "mri3d": mri3d_fixture, "fan": fanbeam_fixtures, "anderson": anderson_fixtures,
             "diffpir": diffpir_fixture, "inpainting": inpainting_fixture, "fastmri": fastmri_fixture,
             "callers": callers_fixture}
    for w in which:
        table[w]()
