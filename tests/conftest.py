import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# what the reference (openai/gym 0.26.2) returned in the comparisons of the *_reference* tests
# (oracle/gen_reference_golden.py)
REFERENCE_GOLDEN = os.path.join(GOLDEN, "reference")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def golden_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and f != "rng_kat.npz")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = {k: z[k] for k in z.files}
    g["env_id"] = str(g["env_id"])
    g["N"], g["T"] = int(g["N"]), int(g["T"])
    g["seed"] = (int(g["seed_hi"]) << 64) | int(g["seed_lo"])
    mes = int(g["max_episode_steps"])
    g["max_episode_steps"] = None if mes < 0 else mes
    g["bounds"] = None if np.isnan(g["bounds"]).any() else tuple(float(b) for b in g["bounds"])
    g["param0"] = None if np.isnan(g["param0"]) else float(g["param0"])
    return g


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle
    oracle.build()
    return oracle


def load_reference_golden(name):
    z = np.load(os.path.join(REFERENCE_GOLDEN, name + ".npz"))
    return {k: (str(z[k]) if z[k].dtype.kind == "U" and z[k].ndim == 0 else z[k]) for k in z.files}


def have_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
