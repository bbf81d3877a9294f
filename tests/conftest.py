import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

HUBER = ((1, 1), (5.991 ** 0.5, 7.815 ** 0.5))   # reference samples/sample_comparison_with_g2o.cpp:195-200
NONE = ((0, 0), (0.0, 0.0))
TUKEY = ((2, 2), (4.0, 5.0))
KERNELS = {"none": NONE, "huber": HUBER, "tukey": TUKEY}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def pkg():
    ge.build()
    return ge.load_package()


@pytest.fixture(scope="session")
def oracle(pkg):
    return ge.load_oracle()


@pytest.fixture(scope="session")
def golden():
    with open(os.path.join(ROOT, "tests", "golden", "oracle_trajectories.json")) as f:
        return json.load(f)


def fixture_path(name):
    return os.path.join(ROOT, "oracle", "_ref", "fixtures", name + ".cubagraph")


def have_fixture(name):
    return os.path.exists(fixture_path(name))


SUBGRAPHS = ("kitti07_sub", "kitti00_sub")   # stored pieces of the two real graphs (tests/golden/make_subgraphs.py)


def load_subgraph(name):
    with np.load(os.path.join(ROOT, "tests", "golden", name + ".npz")) as z:
        return {k: z[k].astype(np.int32 if z[k].dtype.kind == "i" else np.float64) for k in z.files}


@pytest.fixture(scope="session")
def problems(pkg):
    """cache of flattened problems by name"""
    cache = {}

    def get(name):
        if name not in cache:
            if name.startswith("ba_"):
                g = pkg.graphio.read_graph(fixture_path(name))
            elif name in SUBGRAPHS:
                g = load_subgraph(name)
            else:
                g = pkg.synth.make_config(name)
            cache[name] = pkg.graphio.flatten(g)
        return cache[name]
    return get


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    if a.size == 0 and b.size == 0:
        return 0.0
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def make_engine(pkg, prob, rk, **kw):
    eng = pkg.Engine(device=0, **kw)
    for et in (0, 1):
        eng.set_robust_kernels(rk[0][et], rk[1][et], et)
    eng.initialize(prob)
    return eng
