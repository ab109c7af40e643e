"""64-bit Morton codes (SURVEY.md 8f, N3; /root/reference/src/morton.cpp, src/common/morton_code.cpp).
Integer work: everything is compared bit for bit -- the C restatement and the CUDA kernels against golden vectors
produced by the reference's own MortonCode64 class (oracle/make_golden_morton.py) and against what that library
returned on larger seeded inputs (oracle/make_golden_fresh.py).  `morton_knn(sort_dist=True)`: the window is pinned;
the order inside it is the intended one (by distance to the query), which the reference itself leaves undefined
(uninitialised comparator state)."""
import numpy as np
import pytest

from conftest import assert_pinned, load_golden


def _check_against_golden(M, **kw):
    g = load_golden("morton_ref")
    codes = M.morton_encode(g["pts"], **kw)
    assert codes.dtype == np.uint64 and np.array_equal(codes, g["codes"])
    assert np.array_equal(M.morton_encode(g["pts"].astype(np.int64), **kw), g["codes"])
    dec = M.morton_decode(g["codes"], **kw)
    assert dec.dtype == np.int32 and np.array_equal(dec, g["decoded"]) and np.array_equal(dec, g["pts"])
    assert np.array_equal(M.morton_add(g["codes"], g["other"], **kw), g["added"])
    assert np.array_equal(M.morton_subtract(g["codes"], g["other"], **kw), g["subtracted"])
    for k in (1, 2, 7, 16):
        w = M.morton_knn(g["sorted_codes"], g["queries"], k, sort_dist=False, **kw)
        assert w.dtype == np.int64 and np.array_equal(w, g["window_k%d" % k])
        s = M.morton_knn(g["sorted_codes"], g["queries"], k, sort_dist=True, **kw)
        assert np.array_equal(np.sort(s, axis=1), g["window_k%d" % k])          # same window, reordered
        pts = M.morton_decode(g["sorted_codes"], **kw).astype(np.float64)
        q = M.morton_decode(g["queries"], **kw).astype(np.float64)
        d = ((pts[s] - q[:, None, :]) ** 2).sum(-1)
        assert np.all(d[:, 1:] >= d[:, :-1])                                    # ascending distance to the query point
    w = M.morton_knn(g["tiny_codes"], g["queries"], 15, sort_dist=False, **kw)
    assert w.shape == (len(g["queries"]), 10) and np.array_equal(w, g["tiny_window_k15"])   # tests/test_examples.py:506-508


def test_restatement_matches_reference_goldens(oracle):
    _check_against_golden(oracle, impl="port")


def test_restatement_matches_reference_library_on_fresh_inputs(oracle):
    """The reference library's outputs on these seeded inputs are stored in tests/golden/fresh_morton_ref.npz."""
    g = load_golden("fresh_morton_ref")
    rng = np.random.default_rng(5)
    pts = rng.integers(-(1 << 20), 1 << 20, (50000, 3)).astype(np.int32)
    a = oracle.morton_encode(pts, impl="port")
    assert_pinned(oracle, g, "encode_a", a)
    b = oracle.morton_encode(rng.integers(-(1 << 19), 1 << 19, (50000, 3)).astype(np.int32), impl="port")
    assert_pinned(oracle, g, "encode_b", b)
    assert_pinned(oracle, g, "add", oracle.morton_add(a, b, impl="port"))
    assert_pinned(oracle, g, "subtract", oracle.morton_subtract(a, b, impl="port"))
    assert_pinned(oracle, g, "decode", oracle.morton_decode(a, impl="port"))
    s = np.sort(a)
    for k in (1, 5, 64):
        assert_pinned(oracle, g, "knn_k%d" % k, oracle.morton_knn(s, b[:3000], k, False, impl="port"))
    # the arithmetic is the arithmetic of the encoded vectors (no overflow inside 21 bits)
    small = rng.integers(-1000, 1000, (1000, 3)).astype(np.int32)
    other = rng.integers(-1000, 1000, (1000, 3)).astype(np.int32)
    ca, cb = oracle.morton_encode(small), oracle.morton_encode(other)
    assert np.array_equal(oracle.morton_decode(oracle.morton_add(ca, cb)), small + other)
    assert np.array_equal(oracle.morton_decode(oracle.morton_subtract(ca, cb)), small - other)
    # unsigned order of the codes is the order along the curve with signed coordinates
    assert oracle.morton_encode(np.array([[-1, -1, -1]], np.int32))[0] < oracle.morton_encode(np.array([[0, 0, 0]], np.int32))[0]


def test_argument_errors(pcu):
    pts = np.zeros((4, 3), np.int32)
    codes = np.zeros(4, np.uint64)
    with pytest.raises(ValueError, match="scalar type"):
        pcu.morton_encode(pts.astype(np.float32))
    with pytest.raises(ValueError, match="empty"):
        pcu.morton_encode(pts[:0])
    with pytest.raises(ValueError, match="columns"):
        pcu.morton_encode(pts[:, :2])
    with pytest.raises(ValueError, match="scalar type"):
        pcu.morton_decode(codes.astype(np.int64))
    with pytest.raises(ValueError, match="empty"):
        pcu.morton_decode(codes[:0])
    with pytest.raises(ValueError, match="same number"):
        pcu.morton_add(codes, codes[:2])
    with pytest.raises(ValueError, match="greater than 0"):
        pcu.morton_knn(codes, codes, 0)
    with pytest.raises(ValueError, match="match"):
        pcu.morton_knn(codes, codes.astype(np.uint32), 2)


@pytest.mark.gpu
def test_kernels_match_reference_goldens(pcu):
    _check_against_golden(pcu)


@pytest.mark.gpu
def test_kernels_match_the_oracle_at_scale(pcu, oracle):
    """The reference's big-data test shapes (tests/test_examples.py:444-468): 1e6 points, 1e4 queries, k = 7."""
    rng = np.random.default_rng(9)
    pts = (rng.random((1000000, 3)) * 1000).astype(np.int32)
    q = (rng.random((10000, 3)) * 1000).astype(np.int32)
    codes = pcu.morton_encode(pts)
    assert np.array_equal(codes, oracle.morton_encode(pts))
    srt = np.sort(codes)
    qc = pcu.morton_encode(q)
    nn = pcu.morton_knn(srt, qc, 7)
    assert nn.shape == (10000, 7) and nn.dtype == np.int64
    assert np.array_equal(np.sort(nn, axis=1), oracle.morton_knn(srt, qc, 7, sort_dist=False))
    assert np.array_equal(nn, oracle.morton_knn(srt, qc, 7, sort_dist=True))
    assert np.array_equal(pcu.morton_decode(codes), pts)
    other = pcu.morton_encode((rng.random((1000000, 3)) * 1000).astype(np.int32))
    assert np.array_equal(pcu.morton_add(codes, other), oracle.morton_add(codes, other))
    assert np.array_equal(pcu.morton_subtract(codes, other), oracle.morton_subtract(codes, other))
    c32 = (codes & np.uint64(0xffffffff)).astype(np.uint32)                      # uint32 codes are widened like the reference does
    assert np.array_equal(pcu.morton_decode(c32), oracle.morton_decode(c32))
