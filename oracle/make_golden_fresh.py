"""TEST INFRASTRUCTURE: generate tests/golden/fresh_knn_ref.npz and tests/golden/fresh_morton_ref.npz -- what the
reference's own libraries (oracle/_ref) return on the seeded inputs of
tests/test_oracle.py::test_port_matches_reference_library_on_fresh_inputs and
tests/test_morton.py::test_restatement_matches_reference_library_on_fresh_inputs.

    python oracle/make_golden_fresh.py      (needs the reference tree, see oracle/Makefile)

The outputs are megabytes, so each array is stored as its digest (oracle.array_digest, which pins every element) plus
a fixed sample of its rows, which makes a mismatch readable.  The inputs are regenerated from their seeds by the tests;
their digests are stored too, so that a change of numpy's generators shows up as such.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SAMPLE_ROWS = 256


def pin(rec, key, arr):
    """Digest of the whole array and a seeded sample of its rows."""
    rec[key + "_digest"] = np.array(O.array_digest(arr))
    rows = np.sort(np.random.default_rng(0).choice(len(arr), min(SAMPLE_ROWS, len(arr)), replace=False))
    rec[key + "_rows"] = rows
    rec[key + "_sample"] = arr[rows]


def knn_fixture():
    rec = {}
    rng = np.random.default_rng(11)
    for dt in (np.float32, np.float64):
        sfx = np.dtype(dt).name
        q = rng.random((3000, 3)).astype(dt)
        d = np.concatenate([rng.random((4000, 3)), rng.random((500, 3)).round(1)]).astype(dt)
        rec[sfx + "_query_digest"] = np.array(O.array_digest(q))
        rec[sfx + "_dataset_digest"] = np.array(O.array_digest(d))
        for k, leaf in ((1, 10), (5, 3), (33, 10)):
            dist, idx = O.k_nearest_neighbors(q, d, k, max_points_per_leaf=leaf, impl="reference")
            pin(rec, "%s_k%d_leaf%d_dist" % (sfx, k, leaf), dist)
            pin(rec, "%s_k%d_leaf%d_idx" % (sfx, k, leaf), idx)
    # the serial path of the reference, against which the tests check the restatement's OpenMP path (n >= 100000)
    q = rng.random((100000, 3), dtype=np.float32)
    d = rng.random((20000, 3), dtype=np.float32)
    rec["serial_query_digest"] = np.array(O.array_digest(q))
    rec["serial_dataset_digest"] = np.array(O.array_digest(d))
    dist, idx = O.k_nearest_neighbors(q, d, 2, num_threads=0, impl="reference")
    pin(rec, "serial_k2_dist", dist)
    pin(rec, "serial_k2_idx", idx)
    return rec


def morton_fixture():
    rec = {}
    rng = np.random.default_rng(5)
    pts = rng.integers(-(1 << 20), 1 << 20, (50000, 3)).astype(np.int32)
    a = O.morton_encode(pts, impl="reference")
    b = O.morton_encode(rng.integers(-(1 << 19), 1 << 19, (50000, 3)).astype(np.int32), impl="reference")
    pin(rec, "encode_a", a)
    pin(rec, "encode_b", b)
    pin(rec, "add", O.morton_add(a, b, impl="reference"))
    pin(rec, "subtract", O.morton_subtract(a, b, impl="reference"))
    pin(rec, "decode", O.morton_decode(a, impl="reference"))
    s = np.sort(a)
    for k in (1, 5, 64):
        pin(rec, "knn_k%d" % k, O.morton_knn(s, b[:3000], k, False, impl="reference"))
    return rec


def main():
    O.build(quiet=False)
    assert O.have_reference() and O.have_morton_reference(), "oracle/_ref is required to (re)generate these goldens"
    for name, rec in (("fresh_knn_ref", knn_fixture()), ("fresh_morton_ref", morton_fixture())):
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **rec)
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
