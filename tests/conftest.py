import gzip
import json
import os
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
MPS_DIR = os.path.join(GOLDEN, "mps")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)")
    config.addinivalue_line("markers", "slow: larger sizes")


_INFLATED = tempfile.TemporaryDirectory(prefix="cuopt_b200_mps_")  # removed when the session ends


def mps_path(rel: str, tmp_dir=None) -> str:
    """Path of a fixture under tests/golden/mps (gz files are inflated to a temp file: the tree may be read-only)."""
    p = os.path.join(MPS_DIR, rel)
    if os.path.exists(p):
        return p
    gz = p + ".gz"
    if os.path.exists(gz):
        out_dir = tmp_dir or _INFLATED.name
        os.makedirs(out_dir, exist_ok=True)
        out = os.path.join(out_dir, os.path.basename(p))
        if not os.path.exists(out):
            with open(out, "wb") as f:
                f.write(gzip.open(gz).read())
        return out
    raise FileNotFoundError(rel)


def load_golden(name: str):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def pins():
    return load_golden("reference_pins.json")


@pytest.fixture(scope="session")
def simplex_golden():
    return load_golden("simplex_golden.json")


def has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:  # noqa: BLE001
        return os.path.exists("/dev/nvidia0")


def problem_arrays(p):
    """Ranged-form numpy arrays of a capi.Problem (what the solver sees)."""
    off, idx, val = p.constraint_matrix()
    m = p.num_constraints
    clb, cub = p.constraint_lower_bounds(), p.constraint_upper_bounds()
    if m and np.isnan(clb).all():  # sense form
        sense = np.frombuffer(p.constraint_sense(), np.uint8)
        rhs = p.rhs()
        clb = np.where(sense == ord("L"), -np.inf, rhs)
        cub = np.where(sense == ord("G"), np.inf, rhs)
    return dict(offsets=off, indices=idx, values=val, c=p.objective_coefficients(), var_lb=p.variable_lower_bounds(),
                var_ub=p.variable_upper_bounds(), con_lb=clb, con_ub=cub, maximize=p.objective_sense == -1,
                objective_offset=p.objective_offset)
