import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
GOLDEN = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def load_golden(name: str) -> dict:
    """npz fixture -> dict of torch tensors; keys `sd__a__b` are collected into a state_dict under 'sd'.  A fixture too large for
    one file (every stored file stays under 1 MB) continues in golden/more/<name>.npz."""
    z = dict(np.load(GOLDEN / f"{name}.npz"))
    more = GOLDEN / "more" / f"{name}.npz"
    if more.exists():
        z.update(np.load(more))
    out, sd = {}, {}
    for k in z:
        if k == "sd_from":  # the state_dict lives in another fixture (the seed-0 tiny DRUNet is shared by several cases)
            sd = dict(load_golden(str(z[k]))["sd"])
            continue
        t = torch.from_numpy(np.asarray(z[k]))
        if k.startswith("sd__"):
            sd[k[4:].replace("__", ".")] = t
        else:
            out[k] = t
    if sd:
        out["sd"] = sd
    return out


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """relative L2 error of a against the reference b"""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


@pytest.fixture(scope="session")
def golden():
    return load_golden


def golden_names(prefix: str):
    return sorted(p.stem for p in GOLDEN.glob(f"{prefix}*.npz"))
