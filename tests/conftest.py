"""Shared fixtures.  `-m "not gpu"` runs everywhere (oracle vs goldens, host logic, C-ABI symbols,
gloo world-size-2 sharding); `-m gpu` needs a B200 and calls the CUDA library through its C ABI."""
import pathlib
import sys
import warnings

import numpy as np
import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

DATA = ROOT / "tests" / "data"
GOLDEN = ROOT / "tests" / "golden"
CASES = sorted(p.stem for p in DATA.glob("*.cnf"))

# tolerances of BASELINE.json north_star: exit waves rel-L2 <= 1e-5, intensities <= 1e-4
TOL_WAVE = 1e-5
TOL_INTENSITY = 1e-4


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def live_reference_missing(harness) -> bool:
    """True when the reference build (oracle/_ref/ref_harness, made from the reference's sources by
    oracle/Makefile) is absent; the test then says so in the warnings summary of the run."""
    if harness.exists():
        return False
    warnings.warn(f"live reference comparison not run: {harness.name} is not built (make -C oracle REF=<sources>)")
    return True


def rel_l2(a, b):
    a = np.asarray(a).astype(np.complex128).ravel()
    b = np.asarray(b).astype(np.complex128).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture(scope="session")
def orc():
    import fdes_oracle
    return fdes_oracle


@pytest.fixture(scope="session")
def qorc(orc):
    import qsc_oracle
    return qsc_oracle


@pytest.fixture(scope="session")
def fb():
    import fdes_b200
    return fdes_b200


def golden(case):
    f = GOLDEN / f"{case}.npz"
    if not f.exists():
        pytest.fail(f"golden vector {f} missing (tools/make_golden.py)")
    g = np.load(f)
    meta = dict(zip(g["meta_keys"].tolist(), g["meta_vals"].tolist()))
    return g, meta


@pytest.fixture(scope="session")
def oracle_runs(orc):
    """Oracle result of every small case, computed once per session (a few seconds in total).
    Frozen-phonon coordinates come from the oracle's own XORWOW restatement."""
    cache = {}

    def get(case):
        if case not in cache:
            p, Z, xyz, dwf, occ = orc.read_cnf(str(DATA / f"{case}.cnf"))
            cache[case] = (orc.build_measurements(p, Z, xyz, dwf, occ), (p, Z, xyz, dwf, occ))
        return cache[case]
    return get
