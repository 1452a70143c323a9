#!/usr/bin/env python
"""bench.py — the BASELINE.json workloads on B200, one JSON line per run.

    python bench.py --gpus 1 --steps 10 --warmup 3                 # cfg2 (default): PnP-PGD iterations/s, MRI 256x256 + DRUNet
    python bench.py --impl reference --steps 2 --warmup 1          # the reference's CPU path (oracle port) on the host cores
    torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU, batch sharded (weak scaling)
    python bench.py --config cfg3|cfg4|cfg5 ...                    # the other BASELINE.json workloads (see CONFIGS)
    python bench.py --scaling strong --gpus N                      # cfg2 with the GLOBAL batch of 64 split over N ranks
    python bench.py --dump-outputs DIR ...                         # also write the last timed step's result as DIR/x_hat.npy

cfg2 (the configuration the metric is quoted on): one "step" = one PnP-PGD iteration over the whole batch — fused L2 data
step z = x - gamma (A^T A x - A^T y), then x = DRUNet(z, sigma) — through the package's public optimiser API
(deepinv_b200.optim.PGD.single_iteration).  The denoiser runs at precision="tc32h" (3 x FP16 split operands on tcgen05:
22-bit operands, fp32-grade: whole-network error < 1e-5 against the fp32 reference; "tc32" = the TF32 variant); the line also carries the error of the TIMED
configuration's K-iteration result against the fp32 CUDA-core path and against the oracle (`parity`), the throughput of the
fp32 CUDA-core path (`value_fp32`) and of the bf16 tensor-core path with ITS error (`bf16`), per-operator roofline
fractions with full-size errors against the oracle (`operators`), `cpu_baseline`, clocks sampled during the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

SIGMA_DEN = 0.05
STEPSIZE = 1.0
DRUNET_GFLOP_PER_IMAGE = 277.40  # SURVEY Appendix A.12 (C=2, 256x256)

CONFIGS = {
    "cfg2": {"workload": "MRI 4x Cartesian-mask 256x256, PnP-PGD + DRUNet, batch=64 per GPU", "batch": 64, "H": 256, "W": 256,
             "metric": "pnp_pgd_iterations_per_s", "unit": "it/s"},
    "cfg3": {"workload": "Tomography Radon 512x512, 180 angles, FBP + 5-iteration unfolded ADMM (DnCNN prior), batch=32 per GPU",
             "batch": 32, "H": 512, "W": 512, "metric": "fbp_unfolded_admm_reconstructions_per_s", "unit": "batches/s"},
    "cfg4": {"workload": "MRI 8x random-mask 320x320, DDRM sampler steps + DRUNet (single-coil SVD) and multi-coil (8 coils) A/A^T, "
                         "batch=32 per GPU", "batch": 32, "H": 320, "W": 320, "metric": "ddrm_steps_per_s", "unit": "it/s"},
    "cfg5": {"workload": "Blur deconvolution 1024x1024 motion-PSF (BlurFFT), PnP-ADMM + DnCNN, batch=32 per GPU", "batch": 32,
             "H": 1024, "W": 1024, "metric": "pnp_admm_iterations_per_s", "unit": "it/s"},
}
REF_SAMPLE = 16  # images of the 64 the CPU arm runs per step
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs budget over all arrays


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """`--dump-outputs`: each array as <out_dir>/<name>.npy in float32, so that two builds can be compared output for output.
    An array larger than its share of DUMP_BYTES is replaced by a fixed seeded sample of its elements (flat, in index order):
    the same positions on every run."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    cap = (DUMP_BYTES // len(arrays) - 4096) // 4  # elements per array (4096 bytes of room for the .npy header)
    for name, t in arrays.items():
        a = t.detach().float()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.flatten()[idx.to(a.device)]
        np.save(d / f"{name}.npy", a.cpu().numpy())


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def cartesian_mask(batch: int, h: int, w: int, accel: int, seed: int) -> torch.Tensor:
    """the package's RandomMaskGenerator — the law of deepinv/physics/generator/mri.py:136-196 (fully sampled centre band,
    uniformly random further columns, constant along H) — drawn on the host so that both arms see the same masks"""
    from deepinv_b200.physics.generator import RandomMaskGenerator

    gen = RandomMaskGenerator(img_size=(2, h, w), acceleration=accel, rng=torch.Generator().manual_seed(seed), device="cpu")
    return gen.step(batch_size=batch)["mask"].contiguous()


def host_info() -> dict:
    logical = os.cpu_count() or 1
    physical = None
    try:
        cores = set()
        phys, core = None, None
        for line in Path("/proc/cpuinfo").read_text().splitlines():
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
                cores.add((phys, core))
        physical = len(cores) or None
    except OSError:
        pass
    try:
        affinity = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        affinity = logical
    return {"logical": logical, "physical": physical, "usable": affinity}


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """`nvidia-smi -lms 20` running from before the warm-up; every sample carries the driver's timestamp, so the samples that
    fall INSIDE a host-side window (the timed region, or — when that is shorter than a few sampler periods — a replay of the
    same workload right after it) can be picked out afterwards."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    @staticmethod
    def now():
        import datetime

        return datetime.datetime.now()

    def stop(self, windows) -> dict:
        """windows: list of (label, t_begin, t_end) in preference order; the first one holding >= 3 samples is reported"""
        import datetime

        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = []
        for r in Path(self.f.name).read_text().strip().splitlines():
            c = [v.strip() for v in r.split(",")]
            if len(c) < 9:
                continue
            try:
                rows.append((datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f"), c))
            except ValueError:
                continue
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        pick, label = rows, "whole run (no sample inside the windows)"
        for lab, t0, t1 in windows:
            inside = [rc for rc in rows if t0 <= rc[0] <= t1]
            if len(inside) >= 3:
                pick, label = inside, lab
                break
        cols = [c for _, c in pick]
        sm = sorted(float(c[1]) for c in cols)
        reasons = set()
        for c in cols:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if c[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(cols[0][2]), "power_w_max": max(float(c[3]) for c in cols),
                "samples": len(cols), "window": label, "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the reference's CPU path (cfg2)
# ---------------------------------------------------------------------------------------------
_cpu_state = {}


def cpu_pgd_iteration_seconds(sample_batch: int, threads: int) -> float:
    """ONE PnP-PGD iteration of the oracle (torch-CPU restatement of the reference path) on `sample_batch` images, seconds"""
    from oracle import ref_ops as R

    torch.set_num_threads(threads)
    key = sample_batch
    if key not in _cpu_state:
        torch.manual_seed(0)
        import deepinv_b200 as dinv

        den = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None)  # parameter container only (random init, seed 0)
        sd = {k: v.detach() for k, v in den.state_dict().items()}
        c = CONFIGS["cfg2"]
        x = torch.randn(sample_batch, 2, c["H"], c["W"])
        mask = cartesian_mask(sample_batch, c["H"], c["W"], 4, seed=0)
        y = R.mri_A(x, mask)
        with torch.no_grad():
            xk = R.mri_At(y, mask)
        _cpu_state[key] = (sd, mask, y, xk)
    sd, mask, y, xk = _cpu_state[key]
    with torch.no_grad():
        t0 = time.perf_counter()
        grad = R.mri_AtA(xk, mask) - R.mri_At(y, mask)          # data_fidelity.py:335-336
        z = xk - STEPSIZE * grad                                  # pgd.py:137-139
        xk = R.drunet_forward(z, SIGMA_DEN, sd)                   # prior.py:99-109 -> drunet.py:212-263
        dt = time.perf_counter() - t0
    _cpu_state[key] = (sd, mask, y, xk)
    return dt


def best_cpu_threads() -> tuple[int, dict]:
    """torch's default is all logical cores; MKL-DNN convolutions on a handful of images do not always scale to 100+ threads,
    so the CPU arm tries a few thread counts ONCE on a 4-image probe and keeps the fastest (all timings reported)"""
    ncpu = host_info()["usable"]
    cands = sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True)
    tried = {}
    for th in cands:
        cpu_pgd_iteration_seconds(4, th)  # (first call also builds the inputs)
        tried[th] = cpu_pgd_iteration_seconds(4, th)
    best = min(tried, key=tried.get)
    return best, {str(k): round(v, 3) for k, v in tried.items()}


def binding_roofline(kernel: str, ms: float, gflop_alg: float, bytes_alg: float, hbm_gbs: float, tensor_peak: float, traffic,
                     peak_source: str, executed_factor: float = 1.0) -> dict:
    """roofline object of the bench line for one kernel launch: `achieved` = ALGORITHMIC bytes (or flops) / measured time against the
    roofline that BINDS the algorithmic work — max(flops / tensor peak, bytes / HBM peak) —, both fractions printed, plus the
    tensor-pipe view of the executed MMAs (`executed_factor` narrow MMAs per algorithmic product: 3 for the split-operand kernels)"""
    t_tensor, t_hbm = gflop_alg / tensor_peak, bytes_alg / 1e6 / hbm_gbs          # ms
    gbs, tfl = bytes_alg / 1e6 / ms, gflop_alg / ms
    bound = "tensor" if t_tensor >= t_hbm else "hbm"
    r = {"bound": bound, "kernel": kernel,
         "achieved": tfl if bound == "tensor" else gbs, "peak": tensor_peak if bound == "tensor" else hbm_gbs,
         "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": (tfl / tensor_peak) if bound == "tensor" else (gbs / hbm_gbs),
         "traffic": traffic,
         "binding": f"max(algorithmic flops / tensor peak = {t_tensor * 1e3:.0f} us, algorithmic bytes / HBM peak = {t_hbm * 1e3:.0f} us)",
         "frac_hbm": gbs / hbm_gbs, "frac_tensor_algorithmic": tfl / tensor_peak,
         "peak_source": peak_source, "us_per_launch": ms * 1e3, "algorithmic_gflop_per_launch": gflop_alg,
         "algorithmic_bytes_per_launch": bytes_alg, "algorithmic_TFLOPs": tfl}
    if executed_factor != 1.0:
        r["tensor_pipe"] = {"executed_mma_gflop_per_launch": executed_factor * gflop_alg, "executed_TFLOPs": executed_factor * tfl,
                            "frac_of_peak": executed_factor * tfl / tensor_peak, "peak_TFLOPs": tensor_peak,
                            "what": f"{executed_factor:g} narrow MMAs per fp32-grade product (hi*hi, hi*lo, lo*hi): the tensor pipe is this busy, "
                                    "the algorithmic work is what `achieved` counts"}
    return r


def bench_config(cfg: str, world: int, scaling: str) -> dict:
    c = CONFIGS[cfg]
    per_gpu = c["batch"] // world if scaling == "strong" else c["batch"]
    workload = c["workload"]
    if scaling == "strong" and world > 1:   # the SAME batch split over the ranks: say so in the workload name
        workload = workload.replace(f"batch={c['batch']} per GPU", f"batch={c['batch']} in total ({per_gpu} per GPU)")
    return {"workload": workload, "global_batch": per_gpu * world, "parallelism": f"dp{world}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config != "cfg2":
        print(json.dumps({"impl": "reference", "unavailable": f"the CPU arm is implemented for cfg2 (the metric's configuration); got {args.config}"}))
        return
    c = CONFIGS["cfg2"]
    threads, tried = best_cpu_threads()
    for _ in range(max(args.warmup, 0)):
        cpu_pgd_iteration_seconds(REF_SAMPLE, threads)
    ts = [cpu_pgd_iteration_seconds(REF_SAMPLE, threads) for _ in range(max(args.steps, 1))]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"x_hat": _cpu_state[REF_SAMPLE][3]})
    t = sum(ts) / len(ts)
    scale = c["batch"] / REF_SAMPLE
    value = 1.0 / (t * scale)  # every rank's shard is 64 images; at N GPUs the CPU host runs N shards one after another: N x work, N x time
    hi = host_info()
    line = {
        "impl": "reference", "metric": c["metric"], "value": value, "unit": c["unit"], "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * t, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config("cfg2", args.gpus, args.scaling),
        "sample": {"images_per_step": REF_SAMPLE, "of": c["batch"], "scale_to_full_step": scale,
                   "note": "ms_per_step is the MEASURED wall time of one PnP-PGD iteration on the sample; value = 1 / (ms_per_step * scale)"},
        "host_cores": hi,
        "cpu_baseline": {"value": value, "unit": c["unit"], "cores": threads, "kind": "port",
                         "host_cores_logical": hi["logical"], "host_cores_physical": hi["physical"], "threads_tried_s_per_4_images": tried,
                         "sample": f"one PnP-PGD iteration of the oracle (torch-CPU restatement of the reference path) on {REF_SAMPLE} of "
                                   f"the {c['batch']} images per step (measured, then scaled x{scale:g} per image); {threads} threads "
                                   f"(fastest of {sorted(map(int, tried))} on a 4-image probe)"},
        "e2e": {"value": value, "unit": c["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# B200 arm helpers
# ---------------------------------------------------------------------------------------------
def time_cuda(fn, iters: int, warmup: int = 3) -> float:
    """average milliseconds per call, CUDA events on the current stream"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def graph_time(calls, replays: int = 20) -> float:
    """ms per call: the calls (one per operand set) are captured into ONE CUDA graph and replayed"""
    for c in calls:
        c()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for c in calls:
            c()
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        for c in calls:
            c()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (replays * len(calls))


def rel(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm())


def dist_max(ms: float, dev, world: int) -> float:
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


# ---------------------------------------------------------------------------------------------
# operators of the other configurations: time, roofline fraction, full-size error against the oracle (rank 0)
# ---------------------------------------------------------------------------------------------
def operator_report(dev, peaks, with_oracle: bool) -> list[dict]:
    import deepinv_b200 as dinv
    from oracle import ref_ops as R

    out = []
    hbm = peaks["hbm_gbs"]

    def add(name, ms, mb=None, gflop=None, err=None, note=None):
        d = {"op": name, "ms": ms}
        if mb is not None:
            d.update(algorithmic_MB=mb, GBps=mb / ms, frac_hbm=mb / ms / hbm)
        if gflop is not None:
            d.update(algorithmic_gflop=gflop, TFLOPs=gflop / ms)
        if err is not None:
            d["rel_err_vs_oracle_full_size"] = err
        if note:
            d["note"] = note
        out.append(d)

    g = torch.Generator(device=dev).manual_seed(11)
    with torch.no_grad():
        # ---- cfg3: Tomography 512x512, 180 angles, batch 32 ------------------------------------------
        B, W, A = 32, 512, 180
        p = dinv.physics.Tomography(angles=A, img_width=W, normalize=False, device=dev)
        x = torch.rand(B, 1, W, W, device=dev, generator=g)
        y = p.A(x)
        mb = (B * W * W + B * p.P * A) * 4 / 1e6
        gflop = B * A * p.P * p.P * 14 / 1e9
        e, n = {}, {}
        if with_oracle:  # one image at full size on the host: the reference's rotate-and-sum Radon, its autograd transpose, its FBP
            xc = x[:1].cpu()
            theta = torch.linspace(0, 180, A + 1)[:-1]
            yc = R.tomography_A(xc, theta, circle=False)
            th64 = theta.double()
            y64 = R.tomography_A(xc.double(), th64, circle=False)
            # beyond ~1e-5 the oracle's own fp32 sampling grid is the limit at this size: the fp64 yardstick says how far the
            # kernel and the reference's fp32 evaluation each are from the exact operator
            yard = lambda got, r32, r64: f"vs fp64 evaluation: kernel {rel(got, r64):.1e}, reference fp32 {rel(r32, r64):.1e}"
            e["A"] = rel(y[:1], yc)
            n["A"] = yard(y[:1], yc, y64)
            at32 = R.tomography_At(yc, theta, W, circle=False)
            e["At"] = rel(p.A_adjoint(yc.to(dev)), at32)
            n["At"] = yard(p.A_adjoint(yc.to(dev)), at32, R.tomography_At(yc.double(), th64, W, circle=False))
            f32 = R.tomography_fbp(yc, theta, W, circle=False)
            e["fbp"] = rel(p.A_dagger(yc.to(dev), fbp=True), f32)
            n["fbp"] = yard(p.A_dagger(yc.to(dev), fbp=True), f32, R.tomography_fbp(yc.double(), th64, W, circle=False))
        add("Tomography.A 32x512^2, 180 angles (cfg3)", time_cuda(lambda: p.A(x), 5, 2), mb, gflop, e.get("A"), n.get("A"))
        add("Tomography.A_adjoint (exact transpose)", time_cuda(lambda: p.A_adjoint(y), 5, 2), mb, gflop, e.get("At"), n.get("At"))
        add("Tomography.A_dagger(fbp=True)", time_cuda(lambda: p.A_dagger(y, fbp=True), 5, 2), mb + 2 * B * p.P * A * 4 / 1e6, None, e.get("fbp"),
            n.get("fbp"))
        del x, y, p
        # ---- cfg4: MultiCoilMRI 32 x 8 coils x 320x320 -------------------------------------------------
        B, N, H, W = 32, 8, 320, 320
        x = torch.randn(B, 2, H, W, device=dev, generator=g)
        maps = torch.view_as_complex(torch.randn(1, N, H, W, 2, device=dev, generator=g))
        maps = maps / maps.abs().pow(2).sum(1, keepdim=True).sqrt()
        mask = cartesian_mask(B, H, W, 8, seed=5).to(dev)
        p = dinv.physics.MultiCoilMRI(mask=mask, coil_maps=maps, img_size=(2, H, W), device=dev)
        y = p.A(x)
        mb = (B * 2 * H * W + B * 2 * N * H * W + N * H * W * 2) * 4 / 1e6
        e = {}
        if with_oracle:
            yc = R.mcmri_A(x[:2].cpu(), mask[:2].cpu(), maps.cpu())
            e["A"] = rel(y[:2], yc)
            e["At"] = rel(p.A_adjoint(y)[:2], R.mcmri_At(yc, mask[:2].cpu(), maps.cpu()))
        add("MultiCoilMRI.A 32x8x320^2 (cfg4)", time_cuda(lambda: p.A(x), 10, 2), mb, None, e.get("A"))
        add("MultiCoilMRI.A_adjoint", time_cuda(lambda: p.A_adjoint(y), 10, 2), mb, None, e.get("At"))
        del x, y, p, maps
        # ---- cfg5: Blur / BlurFFT 32 x 1024x1024, 31x31 PSF -------------------------------------------------
        B, H, W, k = 32, 1024, 1024, 31
        x = torch.rand(B, 1, H, W, device=dev, generator=g)
        f = torch.rand(1, 1, k, k, device=dev, generator=g)
        f /= f.sum()
        img = B * H * W * 4 / 1e6
        gf = 2 * k * k * B * H * W / 1e9
        pc = dinv.physics.Blur(filter=f, padding="circular", device=dev)
        pf = dinv.physics.BlurFFT(img_size=(1, H, W), filter=f, device=dev)
        y = pc.A(x)
        e = {}
        if with_oracle:
            xc, fc = x[:2].cpu(), f.cpu()
            yc = R.blur_A(xc, fc, "circular")
            e["A"] = rel(y[:2], yc)
            e["At"] = rel(pc.A_adjoint(y[:2]), R.blur_At(yc, fc, "circular", H, W))
            fm, fang = R.blurfft_params(fc, (1, H, W))
            e["fA"] = rel(pf.A(x[:2]), R.blurfft_A(xc, fm, fang, (1, H, W)))
            e["fAt"] = rel(pf.A_adjoint(y[:2]), R.blurfft_At(yc, fm, fang, (1, H, W)))
        add("Blur.A 32x1024^2, 31x31, circular (cfg5)", time_cuda(lambda: pc.A(x), 5, 2), 2 * img, gf, e.get("A"))
        add("Blur.A_adjoint", time_cuda(lambda: pc.A_adjoint(y), 5, 2), 2 * img, gf, e.get("At"))
        add("BlurFFT.A 32x1024^2 (cfg5)", time_cuda(lambda: pf.A(x), 10, 2), 2 * img, None, e.get("fA"))
        add("BlurFFT.A_adjoint", time_cuda(lambda: pf.A_adjoint(y), 10, 2), 2 * img, None, e.get("fAt"))
    return out


def safe_operator_report(dev, peaks, with_oracle):
    try:
        return operator_report(dev, peaks, with_oracle)
    except Exception as exc:  # noqa: BLE001  (the headline must not die on an auxiliary table)
        return [{"op": "operator report failed", "error": f"{type(exc).__name__}: {exc}"}]


# ---------------------------------------------------------------------------------------------
# cfg2: PnP-PGD + DRUNet on MRI 256x256
# ---------------------------------------------------------------------------------------------
def run_cfg2(args, world, rank, dev, peaks):
    import torch.distributed as dist

    import deepinv_b200 as dinv
    from deepinv_b200.optim import L2, PGD, PnP

    c = CONFIGS["cfg2"]
    H, W = c["H"], c["W"]
    BATCH = c["batch"] // world if args.scaling == "strong" else c["batch"]
    shard0 = rank * BATCH if args.scaling == "strong" else 0  # strong: this rank's slice of ONE global batch
    torch.manual_seed(0)
    den = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision=args.precision).to(dev).eval()
    if args.scaling == "strong":
        gen = torch.Generator().manual_seed(1234)
        x_true = torch.randn(c["batch"], 2, H, W, generator=gen)[shard0: shard0 + BATCH].contiguous()
        mask = cartesian_mask(c["batch"], H, W, 4, seed=0)[shard0: shard0 + BATCH].contiguous()
    else:
        gen = torch.Generator().manual_seed(1234 + rank)
        x_true = torch.randn(BATCH, 2, H, W, generator=gen)
        mask = cartesian_mask(BATCH, H, W, 4, seed=rank)
    physics = dinv.physics.MRI(mask=mask.to(dev), img_size=(2, H, W), device=dev)
    x_pin = x_true.pin_memory()
    with torch.no_grad():
        y = physics.A(x_pin.to(dev, non_blocking=True))
    y_pin = y.cpu().pin_memory()
    algo = PGD(data_fidelity=L2(), prior=PnP(den), stepsize=STEPSIZE, sigma_denoiser=SIGMA_DEN, max_iter=args.steps, early_stop=False)
    lib = dinv.get_lib()

    def iteration(X, it):
        return algo.single_iteration(X, it, y, physics)

    graphed = None
    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        clocks.start()  # from before the warm-up: the sampler needs ~100 ms to deliver its first line
    with torch.no_grad():
        X0 = algo.init_iterate_fn(y, physics)
        x_init = X0["est"][0].clone()
        X = X0
        for it in range(args.warmup):
            X = iteration(X, it)
        if not args.no_graph:
            try:  # replay the same public-API iteration from a CUDA graph (no Python / ctypes launch path in the loop)
                from deepinv_b200.optim import GraphedIteration

                graphed = GraphedIteration(algo, y, physics, X=X)
                graphed.run(args.warmup)
            except Exception as exc:  # noqa: BLE001
                print(f"bench.py: CUDA-graph capture unavailable ({exc}); timing the eager loop", file=sys.stderr)
                graphed = None
        # the timed region starts from the reference's initial iterate (A^T y), so that its result IS the K-iteration
        # reconstruction the parity block checks
        if graphed is not None:
            graphed.load(x_init)
        else:
            X = {"est": (x_init.clone(), x_init.clone()), "aty": X0.get("aty")}
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches0 = lib.dinvk_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if os.environ.get("DINVK_BENCH_PROFILE"):  # `ncu --profile-from-start off`: only the timed region is captured
            torch.cuda.profiler.start()
        t_w0 = ClockSampler.now()
        e0.record()
        if graphed is not None:
            x_hat = graphed.run(args.steps)
        else:
            for it in range(args.steps):
                X = iteration(X, it)
            x_hat = X["est"][0]
        gathered = None
        if world > 1:  # the only collective of the path: gather the final reconstructions (SURVEY §8e)
            gathered = torch.empty(world * BATCH, 2, H, W, device=dev)
            dist.all_gather_into_tensor(gathered, x_hat.contiguous())
        e1.record()
        torch.cuda.synchronize()
        t_w1 = ClockSampler.now()
        if os.environ.get("DINVK_BENCH_PROFILE"):
            torch.cuda.profiler.stop()
        ms_total = e0.elapsed_time(e1)
        x_hat = x_hat.clone()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"x_hat": gathered if gathered is not None else x_hat})
        launches = lib.dinvk_launch_count() - launches0
        if graphed is not None:
            launches = graphed.launches_per_step * args.steps
        windows = [("timed region", t_w0, t_w1)]
        if rank == 0 and ms_total < 400.0:
            n_probe = max(1, int(1000.0 / max(ms_total / args.steps, 1e-3)))
            t_p0 = ClockSampler.now()
            if graphed is not None:
                graphed.run(n_probe)
            else:
                Xp = X
                for it in range(n_probe):
                    Xp = iteration(Xp, it)
            torch.cuda.synchronize()
            windows.append(("same workload replayed (untimed) for ~1 s right after the timed region", t_p0, ClockSampler.now()))
        clk = clocks.stop(windows) if rank == 0 else None
        ms_total = dist_max(ms_total, dev, world)
        ms_step = ms_total / args.steps
        images_per_step = BATCH * world
        value = (images_per_step / c["batch"]) * 1000.0 / ms_step  # iterations/s in units of 64-image batches

        # ---- strong scaling: the gathered batch must equal what ONE GPU computes for the whole global batch ---------------
        shard_check = None
        if args.verify_shards and world > 1 and args.scaling == "strong":
            if rank == 0:
                gen1 = torch.Generator().manual_seed(1234)
                xg = torch.randn(c["batch"], 2, H, W, generator=gen1)
                mg = cartesian_mask(c["batch"], H, W, 4, seed=0)
                pg = dinv.physics.MRI(mask=mg.to(dev), img_size=(2, H, W), device=dev)
                yg = pg.A(xg.to(dev))
                Xg = algo.init_iterate_fn(yg, pg)
                for it in range(args.steps):
                    Xg = algo.single_iteration(Xg, it, yg, pg)
                ref_all = Xg["est"][0]
                shard_check = {"torch_equal": bool(torch.equal(gathered, ref_all)), "max_abs_diff": float((gathered - ref_all).abs().max()),
                               "what": f"all_gather of {world} shards of {BATCH} images vs the same {c['batch']} images on rank 0 alone, "
                                       f"{args.steps} iterations (kernels are batch-independent and deterministic)"}
                del pg, yg, Xg, ref_all
            dist.barrier()

        # ---- e2e: host buffers in, host buffer out, every step ------------------------------------
        xh = x_hat.cpu().pin_memory()
        out_pin = torch.empty(xh.shape, dtype=xh.dtype, pin_memory=True)

        def e2e_step():
            xd = xh.to(dev, non_blocking=True)
            yd = y_pin.to(dev, non_blocking=True)
            Xn = algo.single_iteration({"est": (xd, xd), "aty": None}, 0, yd, physics)
            out_pin.copy_(Xn["est"][0], non_blocking=True)

        n_e2e = max(4, min(args.steps, 10))
        e2e_mode = "eager, one stream"
        pipe = None
        if not args.no_graph:
            try:
                from deepinv_b200.optim import HostStreamedIteration

                pipe = HostStreamedIteration(algo, physics, xh, y_pin, dev)
                e2e_mode = "3-stream pipeline over 2 device slots, CUDA-graph compute"
            except Exception as exc:  # noqa: BLE001
                print(f"bench.py: host-streamed pipeline unavailable ({exc}); timing the eager e2e step", file=sys.stderr)
        if pipe is not None:
            def e2e_run(n):
                for _ in range(n):
                    pipe.submit(xh, y_pin, out_pin)
                pipe.drain()

            e2e_run(2)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            e2e_run(n_e2e)
            f1.record()
            torch.cuda.synchronize()
            ms_e2e = f0.elapsed_time(f1) / n_e2e
        else:
            ms_e2e = time_cuda(e2e_step, n_e2e, warmup=1)
        ms_e2e = dist_max(ms_e2e, dev, world)
        h2d = xh.numel() * 4 + y_pin.numel() * 4
        d2h = out_pin.numel() * 4

        # ---- rank 0: parity of the timed configuration, other precisions, rooflines, operators -------------------
        parity = roof = ops_report = den_report = fp32_report = bf16_report = other_report = None
        if rank == 0 and not args.lean:
            from deepinv_b200 import ops as dops
            from oracle import ref_ops as R

            nchk = min(4, BATCH)

            def run_precision(prec, nimg, steps):
                """the same K iterations from the same initial iterate with another denoiser precision, first `nimg` images"""
                torch.manual_seed(0)
                d2 = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision=prec).to(dev).eval()
                d2.load_state_dict(den.state_dict())
                ph = dinv.physics.MRI(mask=mask[:nimg].to(dev), img_size=(2, H, W), device=dev)
                al = PGD(data_fidelity=L2(), prior=PnP(d2), stepsize=STEPSIZE, sigma_denoiser=SIGMA_DEN, max_iter=steps, early_stop=False)
                Xq = {"est": (x_init[:nimg].clone(), x_init[:nimg].clone()), "aty": None}
                for it in range(steps):
                    Xq = al.single_iteration(Xq, it, y[:nimg], ph)
                return Xq["est"][0]

            parity = {"what": f"K={args.steps}-iteration PnP-PGD result of the TIMED configuration (denoiser precision {args.precision})",
                      "tolerance_north_star": 1e-5}
            ref32 = run_precision("fp32", nchk, args.steps)
            parity["rel_l2_vs_fp32_cuda_core_path"] = {"images": nchk, "err": rel(x_hat[:nchk], ref32)}
            # everything that runs the oracle on the host cores belongs to the N = 1 line (the other ranks would wait for minutes)
            use_oracle = (not args.no_cpu_baseline) and world == 1
            if not use_oracle:
                parity["rel_l2_vs_oracle"] = None if args.no_cpu_baseline else "in the N = 1 line (host oracle runs are not repeated at N > 1)"
            if use_oracle:
                k_or = min(args.steps, 20)
                sd = {k: v.detach().cpu() for k, v in den.state_dict().items()}
                mc, yc = mask[:2].cpu(), y[:2].cpu()
                t0 = time.perf_counter()
                xo = x_init[:2].cpu()
                for _ in range(k_or):  # the oracle's loop body (pgd.py:137-168) from the same initial iterate
                    grad = R.mri_AtA(xo, mc) - R.mri_At(yc, mc)
                    xo = R.drunet_forward(xo - STEPSIZE * grad, SIGMA_DEN, sd)
                xk = x_hat[:2] if k_or == args.steps else run_precision(args.precision, 2, k_or)
                parity["rel_l2_vs_oracle"] = {"images": 2, "iterations": k_or, "err": rel(xk, xo), "oracle_s": time.perf_counter() - t0}
            # fp32 CUDA-core path: short run on the full batch -> value_fp32
            torch.manual_seed(0)
            d32 = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision="fp32").to(dev).eval()
            d32.load_state_dict(den.state_dict())
            al32 = PGD(data_fidelity=L2(), prior=PnP(d32), stepsize=STEPSIZE, sigma_denoiser=SIGMA_DEN, max_iter=2, early_stop=False)
            Xf = {"est": (x_init.clone(), x_init.clone()), "aty": None}
            Xf = al32.single_iteration(Xf, 0, y, physics)
            ms32 = time_cuda(lambda: al32.single_iteration(Xf, 0, y, physics), 2, warmup=0)
            fp32_report = {"value": (BATCH / c["batch"]) * 1000.0 / ms32, "unit": "it/s", "ms_per_step": ms32, "steps": 2,
                           "what": "the same iteration with the fp32 CUDA-core denoiser (precision='fp32'), eager, this rank's batch"}
            del d32, al32, Xf
            other_report = None
            if args.precision in ("tc32", "tc32h"):  # the other fp32-grade format, same iteration, eager
                oprec = "tc32" if args.precision == "tc32h" else "tc32h"
                torch.manual_seed(0)
                dox = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision=oprec).to(dev).eval()
                dox.load_state_dict(den.state_dict())
                alo = PGD(data_fidelity=L2(), prior=PnP(dox), stepsize=STEPSIZE, sigma_denoiser=SIGMA_DEN, max_iter=2, early_stop=False)
                Xo = {"est": (x_init.clone(), x_init.clone()), "aty": None}
                Xo = alo.single_iteration(Xo, 0, y, physics)
                mso = time_cuda(lambda: alo.single_iteration(Xo, 0, y, physics), 3, warmup=1)
                xo_k = run_precision(oprec, nchk, args.steps)
                other_report = {"precision": oprec, "value": (BATCH / c["batch"]) * 1000.0 / mso, "unit": "it/s", "ms_per_step": mso,
                                "rel_l2_of_K_iteration_result_vs_fp32_path": rel(xo_k, ref32), "images": nchk,
                                "what": "tc32 = 3 x TF32 (any fp32 range), tc32h = 3 x FP16 (|activations| < 65504, loud overflow); eager loop"}
                del dox, alo, Xo
            if args.precision != "bf16":
                torch.manual_seed(0)
                d16 = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision="bf16").to(dev).eval()
                d16.load_state_dict(den.state_dict())
                al16 = PGD(data_fidelity=L2(), prior=PnP(d16), stepsize=STEPSIZE, sigma_denoiser=SIGMA_DEN, max_iter=args.steps, early_stop=False)
                Xb = {"est": (x_init.clone(), x_init.clone()), "aty": None}
                Xb = al16.single_iteration(Xb, 0, y, physics)
                ms16 = time_cuda(lambda: al16.single_iteration(Xb, 0, y, physics), 5, warmup=1)
                x16 = run_precision("bf16", nchk, args.steps)
                bf16_report = {"value": (BATCH / c["batch"]) * 1000.0 / ms16, "unit": "it/s", "ms_per_step": ms16,
                               "rel_l2_of_K_iteration_result_vs_fp32_path": rel(x16, ref32), "images": nchk,
                               "what": "opt-in precision='bf16' (bf16 operands, fp32 accumulate), eager loop; NOT parity-grade"}
                del d16, al16, Xb
            z = x_hat
            ms_den = time_cuda(lambda: den(z, SIGMA_DEN), max(2, min(args.steps, 5)), warmup=1)
            tflops = DRUNET_GFLOP_PER_IMAGE * BATCH / ms_den
            den_report = {"what": "whole DRUNet forward (%s path)" % args.precision, "ms": ms_den,
                          "algorithmic_gflop": DRUNET_GFLOP_PER_IMAGE * BATCH, "TFLOPs_fp32_equivalent": tflops}
            # dominant kernel: the 64 -> 64 3x3 body convolution at full resolution (ResBlock form: + residual)
            C = 64
            gflop_k = 2.0 * BATCH * H * W * C * 9 * C / 1e9
            traffic = None
            tp = ROOT / "profiles" / "top_kernel_traffic.json"
            if tp.exists():
                tj = json.loads(tp.read_text())
                traffic = tj.get(args.precision, {}).get("dram_bytes_per_launch") if isinstance(tj.get(args.precision), dict) else None
                if traffic is None and args.precision == "bf16":
                    traffic = tj.get("dram_bytes_per_launch")
            if args.precision in ("tc32", "tc32h"):
                from deepinv_b200.models.tc_engine import _pack3x3_slab_tc32

                fmt = 1 if args.precision == "tc32h" else 0
                xa = dops.nchw_to_split16(torch.randn(BATCH, C, H, W, device=dev).abs_(), fmt)
                ra = dops.nchw_to_split16(torch.randn(BATCH, C, H, W, device=dev), fmt)
                wa = _pack3x3_slab_tc32(torch.randn(C, C, 3, 3, device=dev) / (3 * C ** 0.5), fmt)
                ms_k = time_cuda(lambda: dops.conv_tc32_slab(xa, wa, C, res=ra), 10, warmup=3)
                bytes_k = 3 * BATCH * H * W * C * 2 * xa.element_size() + wa.numel() * wa.element_size()
                # tf32: K = 8 per instruction on the pipe that does K = 16 in bf16 / fp16 -> half the measured bf16 rate
                tf32_peak = peaks["bf16_tflops"] / (1 if fmt else 2)
                roof = binding_roofline(
                    f"conv_tc32_slab_kernel<{'FmtF16' if fmt else 'FmtTF32'}>: 3x3 conv 64->64, 64x256x256, 3 x "
                    f"{'FP16' if fmt else 'TF32'} -> fp32 (TMEM + register drain), + residual",
                    ms_k, gflop_k, bytes_k, peaks["hbm_gbs"], tf32_peak, traffic,
                    peaks["source"] + (": HBM copy rate; tensor = bf16 burst (kind::f16 runs at the bf16 rate)" if fmt else
                                       ": HBM copy rate; tensor = bf16 burst / 2 (dense tf32 rate of the same pipe)"), executed_factor=3.0)
                del xa, ra, wa
            elif args.precision == "bf16":
                xa = torch.randn(BATCH, H, W, C, device=dev).to(torch.bfloat16)
                ra = torch.randn(BATCH, H, W, C, device=dev).to(torch.bfloat16)
                wa = (torch.randn(C, 9 * C, device=dev) / (3 * C ** 0.5)).to(torch.bfloat16)
                ms_k = time_cuda(lambda: dops.conv3x3_bf16(xa, wa, res=ra), 20, warmup=3)
                bytes_k = 3 * BATCH * H * W * C * 2 + C * 9 * C * 2
                roof = binding_roofline("conv_tc_halo_kernel<64,...>: 3x3 conv 64->64, 64x256x256, bf16 -> fp32 TMEM, +residual", ms_k, gflop_k,
                                        bytes_k, peaks["hbm_gbs"], peaks["bf16_tflops"], traffic,
                                        peaks["source"] + ": HBM copy rate; tensor = bf16 burst (kernel timed alone)")
                del xa, ra, wa
            else:
                roof = {"bound": "tensor", "kernel": "DRUNet convolutions (fp32 CUDA-core path, whole forward)", "achieved": tflops,
                        "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": tflops / peaks["bf16_tflops_sustained"],
                        "traffic": None, "peak_source": peaks["source"] + " bf16 sustained"}
            # MRI operators: each one captured into a CUDA graph that walks SETS disjoint operand sets (> L2 in total)
            SETS = 6
            img_mb = BATCH * 2 * H * W * 4 / 1e6
            gen2 = torch.Generator(device=dev).manual_seed(7)
            sets = []
            for i in range(SETS):
                xs = torch.randn(BATCH, 2, H, W, device=dev, generator=gen2)
                ms_ = cartesian_mask(BATCH, H, W, 4, seed=100 + i).to(dev)
                ps = dinv.physics.MRI(mask=ms_, img_size=(2, H, W), device=dev)
                ys = ps.A(xs)
                sets.append((ps, xs, ys, ps.A_adjoint(ys)))
            errs = {}
            if use_oracle:  # full batch against the oracle on the host (one set)
                ps, xs, ys, atys = sets[0]
                mc = ps.mask.cpu()
                yc = R.mri_A(xs.cpu(), mc)
                errs["A"] = rel(ys, yc)
                errs["At"] = rel(atys, R.mri_At(yc, mc))
                errs["step"] = rel(ps.normal_step(xs, atys, STEPSIZE), xs.cpu() - STEPSIZE * (R.mri_AtA(xs.cpu(), mc) - atys.cpu()))
            cases = [
                ("MRI.A (2-D FFT + mask)", lambda p, x, y, aty: p.A(x), 2 * img_mb, "A"),
                ("MRI.A_adjoint (mask + 2-D iFFT)", lambda p, x, y, aty: p.A_adjoint(y), 2 * img_mb, "At"),
                ("PGD data step x-g(AtAx-Aty), line mask (1 pass)", lambda p, x, y, aty: p.normal_step(x, aty, STEPSIZE), 3 * img_mb, "step"),
                ("MRI.prox_l2, line mask (1 pass)", lambda p, x, y, aty: p.prox_l2(x, y, 1.0), 3 * img_mb, None),
            ]
            ops_report = []
            for name, fn, mb, ek in cases:
                ms = graph_time([(lambda st=st, fn=fn: fn(*st)) for st in sets])
                gbs = mb / ms
                d = {"op": name, "ms": ms, "algorithmic_MB": mb, "GBps": gbs, "frac_hbm": gbs / peaks["hbm_gbs"],
                     "timing": f"CUDA graph over {SETS} disjoint operand sets (> L2), 20 replays"}
                if ek in errs:
                    d["rel_err_vs_oracle_full_size"] = errs[ek]
                ops_report.append(d)
            del sets
            if not args.no_operators:
                ops_report += safe_operator_report(dev, peaks, with_oracle=use_oracle)

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not args.lean:
            threads, tried = best_cpu_threads()
            cpu_pgd_iteration_seconds(REF_SAMPLE, threads)
            t = cpu_pgd_iteration_seconds(REF_SAMPLE, threads)
            hi = host_info()
            cpu = {"value": 1.0 / (t * c["batch"] / REF_SAMPLE), "unit": "it/s", "cores": threads, "kind": "port",
                   "host_cores_logical": hi["logical"], "host_cores_physical": hi["physical"], "threads_tried_s_per_4_images": tried,
                   "sample": f"one PnP-PGD iteration of the oracle on {REF_SAMPLE} of the {c['batch']} images ({t:.2f} s measured, second of "
                             f"two runs), scaled x{c['batch'] / REF_SAMPLE:g} per image; {threads} threads (fastest on a 4-image probe)"}
        dtype = {"tc32h": "f32 (3 x FP16 split-operand tensor-core GEMMs: 22-bit operands, fp32 accumulate) + f32 operators",
                 "tc32": "f32 (3 x TF32 split-operand tensor-core GEMMs, fp32 accumulate) + f32 operators",
                 "bf16": "bf16 denoiser GEMMs (fp32 accumulate) + f32 operators", "fp32": "f32"}[args.precision]
        line = {
            "metric": c["metric"], "value": value, "unit": c["unit"], "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": bench_config("cfg2", world, args.scaling),
            "details": {"denoiser_precision": args.precision, "cuda_graph": graphed is not None, "images_per_gpu": BATCH,
                        "l2_policy": "per-step working set (>= 1 GB of activations) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": (images_per_step / c["batch"]) * 1000.0 / ms_e2e, "unit": c["unit"], "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": n_e2e, "mode": e2e_mode},
            "gpu_launches": int(launches),
            "clocks": clk,
            "shard_check": shard_check,
            "parity": parity,
            "value_fp32": fp32_report,
            "other_fp32_grade_format": other_report,
            "bf16": bf16_report,
            "roofline": roof,
            "denoiser": den_report,
            "operators": ops_report,
            "cpu_baseline": cpu,
        }
    return line


# ---------------------------------------------------------------------------------------------
# cfg3 / cfg4 / cfg5
# ---------------------------------------------------------------------------------------------
def timed_steps(step, steps, warmup, dev, world):
    import torch.distributed as dist

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = ClockSampler.now()
    e0.record()
    out = None
    for _ in range(steps):
        out = step()
    if world > 1 and out is not None:
        gathered = torch.empty((world * out.shape[0], *out.shape[1:]), device=dev, dtype=out.dtype)
        dist.all_gather_into_tensor(gathered, out.contiguous())
        out = gathered
    e1.record()
    torch.cuda.synchronize()
    t1 = ClockSampler.now()
    return dist_max(e0.elapsed_time(e1), dev, world) / steps, out, (t0, t1)


def run_other(args, world, rank, dev, peaks):
    import deepinv_b200 as dinv
    from deepinv_b200.optim import ADMM, L2, PnP

    c = CONFIGS[args.config]
    B, H, W = c["batch"], c["H"], c["W"]
    lib = dinv.get_lib()
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    torch.manual_seed(0)
    extra = {}
    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        clocks.start()
    with torch.no_grad():
        if args.config == "cfg3":
            from deepinv_b200.unfolded import unfolded_builder

            physics = dinv.physics.Tomography(angles=180, img_width=W, normalize=True, device=dev)
            den = dinv.models.DnCNN(in_channels=1, out_channels=1, depth=7, nf=64, pretrained=None, precision=args.precision).to(dev).eval()
            model = unfolded_builder("ADMM", params_algo={"stepsize": 1.0, "g_param": 0.05, "lambda": 1.0, "beta": 1.0},
                                     trainable_params=[], data_fidelity=L2(), prior=PnP(den), max_iter=5,
                                     custom_init=lambda y, p: {"est": (p.A_dagger(y, fbp=True), p.A_dagger(y, fbp=True))}).to(dev).eval()
            x = torch.rand(B, 1, H, W, device=dev, generator=gen)
            y = physics.A(x)
            step = lambda: model(y, physics)
            h2d, d2h = y.numel() * 4, x.numel() * 4
            y_pin, out_pin = y.cpu().pin_memory(), torch.empty(x.shape, pin_memory=True)

            def e2e():
                out_pin.copy_(model(y_pin.to(dev, non_blocking=True), physics), non_blocking=True)
        elif args.config == "cfg4":
            from deepinv_b200.sampling import DDRM

            mask = cartesian_mask(1, H, W, 8, seed=3).to(dev)
            physics = dinv.physics.MRI(mask=mask, img_size=(2, H, W), device=dev)
            physics.noise_model = dinv.physics.GaussianNoise(sigma=0.02) if hasattr(dinv.physics, "GaussianNoise") else physics.noise_model
            den = dinv.models.DRUNet(in_channels=2, out_channels=2, pretrained=None, precision=args.precision).to(dev).eval()
            nsig = 4
            sampler = DDRM(den, sigmas=torch.linspace(1, 0.02, nsig).tolist())
            x = torch.randn(B, 2, H, W, device=dev, generator=gen)
            y = physics.A(x)
            step_full = lambda: sampler(y, physics)
            step = step_full
            extra["ddrm_steps_per_call"] = nsig
            h2d, d2h = y.numel() * 4, x.numel() * 4
            y_pin, out_pin = y.cpu().pin_memory(), torch.empty(x.shape, pin_memory=True)

            def e2e():
                out_pin.copy_(sampler(y_pin.to(dev, non_blocking=True), physics), non_blocking=True)
        else:  # cfg5
            from deepinv_b200.physics.generator import MotionBlurGenerator

            psf = MotionBlurGenerator((31, 31), device="cpu", rng=torch.Generator().manual_seed(2)).step(batch_size=1)["filter"].to(dev)
            physics = dinv.physics.BlurFFT(img_size=(1, H, W), filter=psf, device=dev)
            den = dinv.models.DnCNN(in_channels=1, out_channels=1, depth=20, nf=64, pretrained=None, precision=args.precision).to(dev).eval()
            algo = ADMM(data_fidelity=L2(), prior=PnP(den), stepsize=1.0, sigma_denoiser=SIGMA_DEN, max_iter=args.steps, early_stop=False)
            x = torch.rand(B, 1, H, W, device=dev, generator=gen)
            y = physics.A(x)
            X = algo.init_iterate_fn(y, physics)
            state = {"X": X}

            def step():
                state["X"] = algo.single_iteration(state["X"], 0, y, physics)
                return state["X"]["est"][0]

            h2d, d2h = y.numel() * 4 + x.numel() * 4, x.numel() * 4
            y_pin, x_pin, out_pin = y.cpu().pin_memory(), x.cpu().pin_memory(), torch.empty(x.shape, pin_memory=True)

            def e2e():
                xd, yd = x_pin.to(dev, non_blocking=True), y_pin.to(dev, non_blocking=True)
                Xn = algo.single_iteration({"est": (xd, xd.clone()), "aty": None}, 0, yd, physics)
                out_pin.copy_(Xn["est"][0], non_blocking=True)

        n0 = lib.dinvk_launch_count()
        ms_step, out, win = timed_steps(step, args.steps, args.warmup, dev, world)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"x_hat": out})
        launches = lib.dinvk_launch_count() - n0 - (0)
        launches = int(launches * args.steps / (args.steps + 0))
        ms_e2e = dist_max(time_cuda(e2e, max(2, min(args.steps, 5)), warmup=1), dev, world)
        clk = clocks.stop([("timed region", win[0], win[1])]) if rank == 0 else None
    per_step_units = extra.get("ddrm_steps_per_call", 1)
    value = world * per_step_units * 1000.0 / ms_step
    if rank != 0:
        return None
    return {
        "metric": c["metric"], "value": value, "unit": c["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"f32 ({args.precision} denoiser GEMMs)" if args.precision in ("tc32", "tc32h") else args.precision, "data": "synthetic",
        "config": bench_config(args.config, world, "weak"),
        "details": {"denoiser_precision": args.precision, "eager_loop": True, **extra},
        "e2e": {"value": world * per_step_units * 1000.0 / ms_e2e, "unit": c["unit"], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clk,
        "roofline": None, "cpu_baseline": None,
    }


def run_b200(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (deepinv_b200 has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ.pop("NCCL_DEBUG")  # keep stdout to the one JSON line (NCCL prints its version banner there at VERSION / WARN)
        dist.init_process_group("nccl", device_id=dev)
    peaks = measured_peaks()
    if args.config == "cfg2":
        line = run_cfg2(args, world, rank, dev, peaks)
    else:
        line = run_other(args, world, rank, dev, peaks)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", default=os.environ.get("DINVK_BENCH_PRECISION", "tc32h"), choices=["fp32", "bf16", "tc32", "tc32h"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip everything that runs the oracle on the host")
    ap.add_argument("--no-operators", action="store_true", help="skip the cfg3/cfg4/cfg5 operator table")
    ap.add_argument("--no-graph", action="store_true", help="time the eager Python loop instead of CUDA-graph replays")
    ap.add_argument("--verify-shards", action="store_true", help="strong scaling: compare the gathered result with rank 0 computing the whole batch")
    ap.add_argument("--lean", action="store_true", help="skip the rank-0 extras (parity, other precisions, rooflines, operators, CPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the reconstruction of the last one as DIR/x_hat.npy "
                                                          "(float32; a fixed seeded sample of it beyond 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
