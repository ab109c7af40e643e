"""CPU: the oracle (our restatement of the reference's kd-tree path) is pinned against the golden
vectors generated from the reference's own nanoflann header (oracle/make_golden.py), and against
what that library returned on larger seeded inputs (oracle/make_golden_fresh.py)."""
import numpy as np
import pytest

from conftest import assert_pinned, knn_cases, knn_golden_names, load_golden, metric_golden_names


@pytest.mark.parametrize("name", knn_golden_names())
def test_port_matches_reference_goldens(oracle, name):
    g = load_golden(name)
    q, d = g["query"], g["dataset"]
    for k, leaf, sq, dist, idx in knn_cases(g):
        got_d, got_i = oracle.k_nearest_neighbors(q, d, k, sq, leaf, impl="port")
        assert got_i.dtype == np.int64 and got_d.dtype == q.dtype
        assert got_i.shape == idx.shape and got_d.shape == dist.shape
        assert np.array_equal(got_i, idx), (name, k, leaf, sq)
        assert np.array_equal(got_d, dist), (name, k, leaf, sq)


@pytest.mark.parametrize("name", metric_golden_names())
def test_port_metrics_match_reference_goldens(oracle, name):
    g = load_golden(name)
    x, y = g["x"], g["y"]
    for sq in (0, 1):
        assert oracle.one_sided_hausdorff_distance(x, y, True, bool(sq)) == tuple(g["one_sided_xy_sq%d" % sq])
        assert oracle.one_sided_hausdorff_distance(y, x, True, bool(sq)) == tuple(g["one_sided_yx_sq%d" % sq])
        assert oracle.hausdorff_distance(x, y, True, bool(sq)) == tuple(g["hausdorff_sq%d" % sq])
        assert oracle.hausdorff_distance(x, y, False, bool(sq)) == g["hausdorff_sq%d" % sq][0]
    c, cxy, cyx = oracle.chamfer_distance(x, y, True)
    assert c.dtype == x.dtype and c == g["chamfer"]
    assert np.array_equal(cxy, g["corrs_xy"]) and np.array_equal(cyx, g["corrs_yx"])
    assert float(oracle.chamfer_distance(x, y, p_norm=1)) == float(g["chamfer_p1"])
    assert float(oracle.chamfer_distance(x, y, p_norm=np.inf)) == float(g["chamfer_pinf"])


def test_conventions(oracle):
    rng = np.random.default_rng(7)
    a, b = rng.random((100, 3)), rng.random((50, 3))
    d, i = oracle.k_nearest_neighbors(a, b, 1)
    assert d.shape == (100,) and i.shape == (100,) and i.dtype == np.int64      # tests/test_examples.py:363-368
    d3, i3 = oracle.k_nearest_neighbors(a, b, 3)
    d3s, i3s = oracle.k_nearest_neighbors(a, b, 3, squared_distances=True)
    assert np.array_equal(i3, i3s) and np.allclose(d3 ** 2, d3s, atol=1e-5)      # :390-396
    assert np.all(np.abs(np.linalg.norm(a[:, None] - b[i3], axis=-1) - d3) < 1e-5)  # :374-383
    with pytest.raises(ValueError):
        oracle.k_nearest_neighbors(a, b, 0)                                     # :385-388
    with pytest.raises(ValueError):
        oracle.k_nearest_neighbors(a, b[:0], 1)
    with pytest.raises(ValueError):
        oracle.k_nearest_neighbors(a.astype(np.float32), b, 1)
    h1 = oracle.one_sided_hausdorff_distance(a, b)
    h2 = oracle.one_sided_hausdorff_distance(b, a)
    h = oracle.hausdorff_distance(a, b, return_index=True)                      # :398-425
    assert h[0] == max(h1[0], h2[0])
    assert abs(h[0] - np.linalg.norm(a[h[1]] - b[h[2]])) < 1e-12
    assert (h[1], h[2]) == ((h1[1], h1[2]) if h1[0] > h2[0] else (h2[2], h2[1]))


def test_port_matches_reference_library_on_fresh_inputs(oracle):
    """The reference library's outputs on these seeded inputs are stored in tests/golden/fresh_knn_ref.npz."""
    g = load_golden("fresh_knn_ref")
    rng = np.random.default_rng(11)
    for dt in (np.float32, np.float64):
        sfx = np.dtype(dt).name
        q = rng.random((3000, 3)).astype(dt)
        d = np.concatenate([rng.random((4000, 3)), rng.random((500, 3)).round(1)]).astype(dt)
        assert oracle.array_digest(q) == str(g[sfx + "_query_digest"]), "numpy generated other inputs than the golden's"
        assert oracle.array_digest(d) == str(g[sfx + "_dataset_digest"]), "numpy generated other inputs than the golden's"
        for k, leaf in ((1, 10), (5, 3), (33, 10)):
            a = oracle.k_nearest_neighbors(q, d, k, max_points_per_leaf=leaf, impl="port")
            assert_pinned(oracle, g, "%s_k%d_leaf%d_idx" % (sfx, k, leaf), a[1])
            assert_pinned(oracle, g, "%s_k%d_leaf%d_dist" % (sfx, k, leaf), a[0])
    # the OpenMP path (n >= 100000) gives the same rows as the reference's serial one
    q = rng.random((100000, 3), dtype=np.float32)
    d = rng.random((20000, 3), dtype=np.float32)
    assert oracle.array_digest(q) == str(g["serial_query_digest"]) and oracle.array_digest(d) == str(g["serial_dataset_digest"])
    a = oracle.k_nearest_neighbors(q, d, 2, num_threads=-1, impl="port")
    assert_pinned(oracle, g, "serial_k2_idx", a[1])
    assert_pinned(oracle, g, "serial_k2_dist", a[0])
