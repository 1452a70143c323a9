"""The drop-in boundary against the reference's callers (SURVEY §8(b) "Callers"): deepinv_b200's optimisers, least-squares
solvers and DDRM sampler on its operator / denoiser classes reproduce what deepinv v0.4.1's own PGD, HQS, DDRM and
optim/linear solvers compute on the reference's classes, and the package's unfolded model trains under the reference Trainer's
supervised step.  The reference results are stored in tests/golden/reference_callers.npz (tests/golden/make_golden.py,
`callers`).  The kernels are the host-emulated SIMT kernels (tests/emul), injected like in tests/test_host_logic_emul.py;
nothing here is a product path."""
import pytest
import torch

import parity_cases as P
from conftest import load_golden, rel_err

DEV = torch.device("cpu")


@pytest.fixture(autouse=True)
def emul_backend(monkeypatch):
    from emul_util import emul_lib

    from deepinv_b200 import ops

    lib = emul_lib()

    def check(rc):
        assert rc == 0, lib.dinvk_last_error()

    monkeypatch.setattr(ops, "_require_cuda", lambda *ts: torch.device("cpu"))
    monkeypatch.setattr(ops, "_stream", lambda dev: None)
    monkeypatch.setattr(ops, "get_lib", lambda: lib)
    monkeypatch.setattr(ops, "check", check)
    ops._ws_cache.clear()
    yield
    ops._ws_cache.clear()


def test_dropin_pgd_and_hqs_match_the_reference_on_mri_and_denoiser():
    """deepinv_b200 PGD / HQS (L2.grad, L2.prox, PnP.prox) on its MRI and DRUNet == the reference's PGD / HQS on the reference's own
    MRI and DRUNet (same weights).  Two PGD iterations with the real denoiser, HQS with a closed-form toy denoiser: keeps the
    emulated run short."""
    import deepinv_b200 as dinv
    from deepinv_b200.optim import HQS, L2, PGD, PnP

    g = load_golden("optim_mri_tiny")
    want = load_golden("reference_callers")
    den = P.load_model(dinv.models.DRUNet, g, DEV, in_channels=2, out_channels=2, nc=(8, 16, 32, 64), nb=2)
    phys = dinv.physics.MRI(mask=g["mask"], img_size=(2, 32, 32), device=DEV)
    toy = lambda v, s: v * (1.0 - float(s))
    with torch.no_grad():
        pgd = PGD(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=0.05, max_iter=2, early_stop=False)
        hqs = HQS(data_fidelity=L2(), prior=PnP(toy), stepsize=0.8, sigma_denoiser=0.05, max_iter=3, early_stop=False)
        assert rel_err(pgd(g["y"], phys), want["pgd"]) < 1e-5
        assert rel_err(hqs(g["y"], phys), want["hqs_toy"]) < 1e-5


def test_dropin_least_squares_reproduces_the_reference_prox_on_blur():
    """deepinv_b200 least_squares (CG) on its Blur.A, A_adjoint, A_adjoint_A == the reference's prox_l2 of the same Blur"""
    import deepinv_b200 as dinv

    g = load_golden("blur_gauss_circular_prox")
    phys = dinv.physics.Blur(filter=g["filt"], padding="circular", device=DEV)
    out = dinv.optim.least_squares(phys, g["y"], z=g["z"], init=g["z"], gamma=float(g["gamma"]), solver="CG", max_iter=50, tol=1e-4)
    assert rel_err(out, g["prox"]) < 1e-4


def test_dropin_ddrm_matches_the_reference_on_mri():
    """deepinv_b200 DDRM on its MRI (U_adjoint / V / V_adjoint / mask) == the reference's DDRM (sampling/diffusion.py:149-224) on
    the reference's MRI: recorded noise draws, closed-form toy denoiser"""
    import deepinv_b200 as dinv

    g = load_golden("ddrm_mri_tiny")
    toy = lambda v, s: v * (1.0 / (1.0 + float(s)))
    phys = dinv.physics.MRI(mask=g["mask"], img_size=(2, 32, 32), device=DEV,
                            noise_model=dinv.physics.GaussianNoise(sigma=float(g["sigma_noise"])))
    out = dinv.sampling.DDRM(denoiser=toy, sigmas=g["sigmas"].numpy())(g["y"], phys, noises=list(g["noises"]))
    assert rel_err(out, load_golden("reference_callers")["ddrm_toy"]) < 1e-5


def test_supervised_training_trains_dropin_unfolded_model():
    """the reference Trainer's supervised step (training/trainer.py: online measurements y = physics(x), SupLoss = MSE, Adam)
    on deepinv_b200's unfolded PGD and MRI: the supervised loss goes down over the epochs, every parameter is updated and the
    PSNR of the trained reconstructions is finite"""
    import deepinv_b200 as dinv
    from deepinv_b200.optim import L2, Tikhonov
    from deepinv_b200.unfolded import unfolded_builder

    torch.manual_seed(0)
    N, H, W = 8, 16, 16
    x = torch.randn(N, 2, H, W)
    mask = (torch.rand(1, 1, 1, W) > 0.5).float().expand(1, 2, H, W).contiguous()
    phys = dinv.physics.MRI(mask=mask, img_size=(2, H, W), device=DEV)
    model = unfolded_builder("PGD", params_algo={"stepsize": [0.5, 0.5], "g_param": None, "lambda": [0.3, 0.3]},
                             trainable_params=["stepsize", "lambda"], data_fidelity=L2(), prior=Tikhonov(), max_iter=2)
    batches = list(x.split(4))

    def sup_loss():
        with torch.no_grad():
            return float(sum(((model(phys(xb), phys) - xb) ** 2).mean() for xb in batches))

    before, p0 = sup_loss(), [p.detach().clone() for p in model.parameters()]
    opt = torch.optim.Adam(model.parameters(), lr=1e-1)
    model.train()
    for _ in range(3):
        for xb in batches:
            opt.zero_grad(set_to_none=True)
            loss = ((model(phys(xb), phys) - xb) ** 2).mean()
            loss.backward()
            opt.step()
    assert sup_loss() < before
    assert all(not torch.equal(a, b) for a, b in zip(p0, model.parameters()))
    with torch.no_grad():
        psnr = [float(-10 * torch.log10(((model(phys(xb), phys) - xb) ** 2).mean())) for xb in batches]
    assert all(v == v and abs(v) < float("inf") for v in psnr)


@pytest.mark.parametrize("solver", ["CG", "BiCGStab"])
def test_least_squares_solvers_match_the_reference_solvers(solver):
    """deepinv_b200.optim.least_squares (CG / BiCGStab on the kernels) == the reference's least_squares with the same solver on the
    same operator: same iterates, same stopping rule"""
    import deepinv_b200 as dinv

    g = load_golden("blur_gauss_circular_prox")
    ref = load_golden("reference_callers")
    phys = dinv.physics.Blur(filter=g["filt"], padding="circular", device=DEV)
    gam = float(g["gamma"])
    want = ref[f"ls_{solver}"]
    got = dinv.optim.least_squares(phys, g["y"], z=g["z"], init=g["z"], gamma=gam, solver=solver, max_iter=25, tol=1e-5)
    # CG: regularised normal equations, well conditioned.  BiCGStab on this square operator: the UNregularised deblurring system
    # A x = y (see below) — 40 iterations of it amplify the round-off differences of the inner products to a few 1e-4
    assert rel_err(got, want) < (2e-5 if solver == "CG" else 2e-3)
    if solver == "CG":
        assert rel_err(got, g["prox"]) < 1e-3  # the fixture was produced with tol = 1e-4 (LinearPhysics default)
    else:  # complete system: the reference gives BiCGStab A x = y itself (gamma, z unused) — so does the drop-in
        assert rel_err(phys.A(got), g["y"]) < 1e-3
        valid = dinv.physics.Blur(filter=g["filt"], padding="valid", device=DEV)   # rectangular: normal equations with gamma
        yv = ref["valid_y"]
        assert rel_err(valid.A(g["z"]), yv) < 1e-5
        got_v = dinv.optim.least_squares(valid, yv, z=g["z"], init=g["z"], gamma=gam, solver=solver, max_iter=25, tol=1e-5)
        assert rel_err(got_v, ref["ls_valid_BiCGStab"]) < 2e-5


def test_lsqr_matches_the_reference_lsqr_on_a_rectangular_operator():
    """deepinv_b200.optim.lsqr (Golub-Kahan on the kernels) vs the reference's lsqr (optim/linear/lsqr.py) on the valid-padding
    Blur (rectangular): damped problem with a warm start, and the plain pseudo-inverse"""
    import deepinv_b200 as dinv

    g = load_golden("blur_gauss_circular_prox")
    ref = load_golden("reference_callers")
    phys = dinv.physics.Blur(filter=g["filt"], padding="valid", device=DEV)
    y = ref["lsqr_y"]  # A z + 0.01 * N(0, 1) (seed 0), with the reference's A
    for gam, want, batched in ((2.0, ref["lsqr_gamma2"], False), (torch.tensor([0.5, 3.0]), ref["lsqr_gamma_batched"], True)):
        got = dinv.optim.least_squares(phys, y, z=g["x"], init=g["x"], gamma=gam, solver="lsqr", max_iter=30, tol=1e-6)
        assert rel_err(got, want) < 1e-4, batched
    cg = dinv.optim.least_squares(phys, y, z=g["x"], init=g["x"], gamma=2.0, solver="CG", max_iter=60, tol=1e-6)
    assert rel_err(dinv.optim.least_squares(phys, y, z=g["x"], gamma=2.0, solver="lsqr", max_iter=60, tol=1e-7), cg) < 1e-3


def test_minres_matches_the_reference_minres():
    """deepinv_b200.optim.minres vs the reference's minres (optim/linear/minres.py): the symmetric system (A^T A + I/gamma) x = b of a
    rectangular operator through least_squares, and a symmetric complete operator handed over as A x = y"""
    import deepinv_b200 as dinv

    g = load_golden("blur_gauss_circular_prox")
    ref = load_golden("reference_callers")
    valid = dinv.physics.Blur(filter=g["filt"], padding="valid", device=DEV)
    y = ref["valid_y"]
    got = dinv.optim.least_squares(valid, y, z=g["x"], init=g["x"], gamma=2.0, solver="minres", max_iter=30, tol=1e-6)
    assert rel_err(got, ref["minres_valid"]) < 1e-4
    circ = dinv.physics.Blur(filter=g["filt"], padding="circular", device=DEV)  # symmetric filter: A = A^T, complete system
    got = dinv.optim.least_squares(circ, g["y"], z=g["z"], init=g["z"], gamma=2.0, solver="minres", max_iter=15, tol=1e-6)
    assert rel_err(got, ref["minres_circular"]) < 2e-3  # unregularised deblurring: see the BiCGStab case above
