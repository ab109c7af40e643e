import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def golden_names(prefix_exclude=("metrics_", "c1_metrics")):
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
    return names


def knn_golden_names():
    return [n for n in golden_names() if "metrics" not in n and not n.startswith(("morton", "sinkhorn", "fresh"))]


def metric_golden_names():
    return [n for n in golden_names() if "metrics" in n]


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def assert_pinned(oracle, g, key, got):
    """`got` equals the array a fresh_* fixture pins under `key` (oracle/make_golden_fresh.py): first its sampled
    rows, then, through the digest, every element."""
    rows = g[key + "_rows"]
    assert np.array_equal(got[rows], g[key + "_sample"]), key
    assert oracle.array_digest(got) == str(g[key + "_digest"]), key


def knn_cases(g):
    """Yield (k, leaf, squared, dist, idx) for every combination stored in a knn fixture."""
    for k in g["ks"]:
        for leaf in g["leafs"]:
            for sq in g["squared"]:
                tag = "k%d_leaf%d_sq%d" % (k, leaf, int(sq))
                yield int(k), int(leaf), bool(sq), g["dist_" + tag], g["idx_" + tag].astype(np.int64)


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.build()
    # impl=None everywhere: the reference's own nanoflann path (oracle/_ref) when present -- here and, as a
    # prebuilt file, on the GPU box -- else the restatement that tests/test_oracle.py pins to it.
    O.DEFAULT_FAITHFUL_BUILDS = False   # one tree build instead of the reference's three identical ones
    return O


@pytest.fixture(scope="session")
def pcu():
    import __graft_entry__ as entry
    entry.build()
    import pcu_b200
    return pcu_b200
