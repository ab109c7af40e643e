"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the nearest-neighbour hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
(``point-cloud-utils_b200``) never does, and has no CPU fallback.

Two back ends with one interface:

``impl=None`` (the default everywhere) means "reference" where ``oracle/_ref`` exists, else "port".

* ``impl="port"``       ``oracle/libpcu_oracle.so`` -- our own restatement of the kd-tree build and
                        search (``oracle/kdtree_oracle.cpp``), available everywhere.
* ``impl="reference"``  ``oracle/_ref/libpcu_ref.so`` -- the reference's *own* vendored
                        ``nanoflann.hpp`` compiled in place by ``oracle/Makefile`` (three tree builds
                        per call like the reference).  Present where it was built (this container)
                        and on the GPU box as a prebuilt file.

The two Python metrics restate ``/root/reference/point_cloud_utils/__init__.py:52-81``
(``hausdorff_distance``) and ``:84-120`` (``chamfer_distance``) on top of the two binding-level
functions (``/root/reference/src/point_cloud_distance.cpp:123-164`` and ``:186-234``), including
their conventions: ``(n,)`` squeeze for k == 1, int64 indices, ``ValueError`` for bad arguments,
``-1`` padding, first maximum for Hausdorff, ``>`` / ``<=`` branch rule, no 1/2 factor in Chamfer.

Parity status: PINNED (see tests/test_oracle.py).
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PORT_PATH = os.path.join(_HERE, "libpcu_oracle.so")
_REF_PATH = os.path.join(_HERE, "_ref", "libpcu_ref.so")
_libs = {}
# Default of `faithful_builds` (reference back end only): True = three tree builds per call like the reference
# (what bench.py times); tests set it to False through the conftest fixture -- the three builds produce the same
# tree, so results are identical and the CPU side of the big parity tests is three builds shorter.
DEFAULT_FAITHFUL_BUILDS = True

_c_i64 = ctypes.c_int64
_c_int = ctypes.c_int
_vp = ctypes.c_void_p


def build(quiet=True):
    """Compile the restatement and, where /root/reference is mounted, oracle/_ref."""
    out = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)
    if not quiet:
        print(out.stdout)


def have_reference():
    return os.path.exists(_REF_PATH)


def array_digest(a):
    """SHA-256 of an array's dtype, shape and bytes: lets a golden file pin a large output exactly in 64 characters."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def resolve_impl(impl=None):
    """None -> the reference's own nanoflann path when oracle/_ref is present (this container, and the GPU
    box as a prebuilt file), else the restatement.  Tests that pin one against the other name them explicitly."""
    if impl is None:
        return "reference" if have_reference() else "port"
    return impl


def _lib(impl):
    impl = resolve_impl(impl)
    if impl in _libs:
        return _libs[impl]
    if impl == "port":
        if not os.path.exists(_PORT_PATH):
            build()
        lib = ctypes.CDLL(_PORT_PATH)
        prefix = "pcu_oracle"
        knn_args = [_vp, _c_i64, _vp, _c_i64, _c_int, _c_int, _c_int, _c_int, _vp, _vp]
    elif impl == "reference":
        if not os.path.exists(_REF_PATH):
            raise FileNotFoundError("oracle/_ref/libpcu_ref.so is not built (needs /root/reference)")
        lib = ctypes.CDLL(_REF_PATH)
        prefix = "pcu_ref"
        knn_args = [_vp, _c_i64, _vp, _c_i64, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _vp]
    else:
        raise ValueError("impl must be 'port' or 'reference'")
    for sfx in ("f32", "f64"):
        f = getattr(lib, "%s_knn_%s" % (prefix, sfx))
        f.argtypes = knn_args
        f.restype = _c_int
        g = getattr(lib, "%s_one_sided_hausdorff_%s" % (prefix, sfx))
        g.argtypes = [_vp, _c_i64, _vp, _c_i64, _c_int, _c_int, _vp, _vp, _vp]
        g.restype = _c_int
    getattr(lib, prefix + "_hardware_threads").restype = _c_int
    _libs[impl] = (lib, prefix)
    return _libs[impl]


def hardware_threads(impl=None):
    lib, prefix = _lib(impl)
    return int(getattr(lib, prefix + "_hardware_threads")())


def _check_pair(a, b, name_a, name_b):
    """dtype / shape rules of the binding (point_cloud_distance.cpp:124-125, :136-149)."""
    a = np.asarray(a)
    b = np.asarray(b)
    if a.dtype not in (np.float32, np.float64):
        raise ValueError("%s must have dtype float32 or float64" % name_a)
    if b.dtype != a.dtype:
        raise ValueError("%s must have the same dtype as %s" % (name_b, name_a))
    if a.ndim != 2 or b.ndim != 2:
        raise ValueError("%s and %s must be 2-D" % (name_a, name_b))
    if a.shape[0] == 0 or b.shape[0] == 0:
        raise ValueError("Invalid input set with zero elements")
    if a.shape[1] != 3 or b.shape[1] != 3:
        raise ValueError("Only 3D inputs are supported")
    return np.ascontiguousarray(a), np.ascontiguousarray(b)


def k_nearest_neighbors(query_points, dataset_points, k, squared_distances=False, max_points_per_leaf=10,
                        num_threads=-1, impl=None, faithful_builds=None):
    """point_cloud_distance.cpp:123-164."""
    if k <= 0:
        raise ValueError("Invalid value for k (%d) must be greater than 0." % k)
    q, d = _check_pair(query_points, dataset_points, "query_points", "dataset_points")
    impl = resolve_impl(impl)
    lib, prefix = _lib(impl)
    n, m = q.shape[0], d.shape[0]
    dists = np.empty((n, k), dtype=q.dtype)
    corrs = np.empty((n, k), dtype=np.int64)
    sfx = "f32" if q.dtype == np.float32 else "f64"
    fn = getattr(lib, "%s_knn_%s" % (prefix, sfx))
    args = [q.ctypes.data, n, d.ctypes.data, m, int(k), int(bool(squared_distances)), int(max_points_per_leaf),
            int(num_threads)]
    if impl == "reference":
        args.append(int(bool(DEFAULT_FAITHFUL_BUILDS if faithful_builds is None else faithful_builds)))
    rc = fn(*args, dists.ctypes.data, corrs.ctypes.data)
    if rc != 0:
        raise RuntimeError("oracle call failed (rc=%d)" % rc)
    # npe::move hands the Eigen matrix to numpy and squeezes every size-1 dimension ((n, 1) -> (n,) is
    # pinned by tests/test_examples.py:363-368; numpyeigen itself is not in the reference tree)
    return dists.squeeze(), corrs.squeeze()


def one_sided_hausdorff_distance(source, target, return_index=True, squared_distances=False, max_points_per_leaf=10,
                                 impl=None):
    """point_cloud_distance.cpp:186-234 (note: return_index defaults to True here)."""
    s, t = _check_pair(source, target, "source", "target")
    lib, prefix = _lib(impl)
    sfx = "f32" if s.dtype == np.float32 else "f64"
    out_max = np.empty(1, dtype=s.dtype)
    out_i = np.empty(1, dtype=np.int64)
    out_j = np.empty(1, dtype=np.int64)
    fn = getattr(lib, "%s_one_sided_hausdorff_%s" % (prefix, sfx))
    rc = fn(s.ctypes.data, s.shape[0], t.ctypes.data, t.shape[0], int(bool(squared_distances)),
            int(max_points_per_leaf), out_max.ctypes.data, out_i.ctypes.data, out_j.ctypes.data)
    if rc != 0:
        raise RuntimeError("oracle call failed (rc=%d)" % rc)
    value = float(out_max[0])  # pybind11::cast of a C++ scalar gives a Python float
    if return_index:
        return value, int(out_i[0]), int(out_j[0])
    return value


def hausdorff_distance(x, y, return_index=False, squared_distances=False, max_points_per_leaf=10, impl=None):
    """point_cloud_utils/__init__.py:52-81."""
    h_xy, ix1, iy1 = one_sided_hausdorff_distance(x, y, True, squared_distances, max_points_per_leaf, impl=impl)
    h_yx, iy2, ix2 = one_sided_hausdorff_distance(y, x, True, squared_distances, max_points_per_leaf, impl=impl)
    h = max(h_xy, h_yx)
    if return_index and h_xy > h_yx:
        return h, ix1, iy1
    elif return_index and h_xy <= h_yx:
        return h, ix2, iy2
    return h


def chamfer_distance(x, y, return_index=False, p_norm=2, max_points_per_leaf=10, impl=None, faithful_builds=None):
    """point_cloud_utils/__init__.py:84-120 (distances are recomputed from the indices with numpy)."""
    x = np.asarray(x)
    y = np.asarray(y)
    _, cxy = k_nearest_neighbors(x, y, 1, False, max_points_per_leaf, impl=impl, faithful_builds=faithful_builds)
    _, cyx = k_nearest_neighbors(y, x, 1, False, max_points_per_leaf, impl=impl, faithful_builds=faithful_builds)
    d_xy = np.linalg.norm(x[cyx] - y, axis=-1, ord=p_norm).mean()
    d_yx = np.linalg.norm(y[cxy] - x, axis=-1, ord=p_norm).mean()
    cham = np.mean(d_xy) + np.mean(d_yx)
    if return_index:
        return cham, cxy, cyx
    return cham


def estimate_point_cloud_normals_knn(points, num_neighbors, view_directions=None, drop_angle_threshold=np.deg2rad(90.0),
                                     max_points_per_leaf=10, impl=None):
    """src/point_cloud_normals.cpp:115-173 + :375-411 restated: the k-NN part is the pinned oracle above (self-query,
    the point itself is neighbour 0); the plane fit follows the reference operation for operation -- offsets
    subtracted in the cloud's precision, widened to fp64, right singular vector of the smallest singular value --
    with numpy's LAPACK SVD standing in for Eigen's JacobiSVD, which is not in the reference tree.
    PARITY UNPINNED for the normal vector itself (no golden vector of the reference exists and its SVD cannot be
    built here): same subspace up to rounding, sign arbitrary unless view directions are given."""
    points = np.asarray(points)
    if num_neighbors <= 0:
        raise ValueError("Invalid number of neighbors (%d) must be greater than 0." % num_neighbors)
    if points.ndim != 2 or points.shape[0] == 0 or points.shape[1] != 3:
        raise ValueError("Invalid point set with zero elements: points must have shape (n, 3)")
    n = points.shape[0]
    has_dirs = view_directions is not None and np.asarray(view_directions).shape[0] != 0
    if has_dirs and np.asarray(view_directions).shape != points.shape:
        raise ValueError("Invalid view directions does not match the number of points.")
    _, idx = k_nearest_neighbors(points, points, num_neighbors, True, max_points_per_leaf, impl=impl, faithful_builds=False)
    idx = idx.reshape(n, num_neighbors)
    found = idx[:, -1] >= 0                                   # :139-142
    safe = np.where(idx >= 0, idx, 0)
    offsets = (points[safe] - points[:, None, :]).astype(np.float64)     # (n, k, 3): subtraction in the cloud's dtype
    _, _, vt = np.linalg.svd(offsets, full_matrices=False)               # V(:, 2) == vt[:, 2, :]  (k >= 3)
    if vt.shape[1] < 3:                                                  # fewer than 3 rows: thin V has no third column
        vt = np.concatenate([vt, np.zeros((n, 3 - vt.shape[1], 3))], axis=1)
    normal = vt[:, 2, :].copy()
    keep = found.copy()
    if has_dirs:
        dirs = np.asarray(view_directions).astype(np.float64)
        sgn = np.sign(np.einsum("ij,ij->i", normal, dirs))
        normal *= sgn[:, None]
        with np.errstate(invalid="ignore"):
            angle = np.arccos(np.einsum("ij,ij->i", normal, dirs))
        keep &= ~(angle > drop_angle_threshold)
    kept = np.nonzero(keep)[0].astype(np.int64)
    return kept, normal[kept].astype(points.dtype)


def ball_neighbourhoods(points, ball_radius, chunk=512):
    """What the reference's tree.index->radiusSearch(query, ball_radius, ...) returns (src/point_cloud_normals.cpp:73-74),
    by brute force: nanoflann's RadiusResultSet keeps a point when `dist < radius` where dist is the L2_Simple value,
    i.e. the SQUARED distance ((dx*dx + dy*dy) + dz*dz, every operation rounded in the cloud's precision,
    nanoflann.hpp:496-507), and radius is ball_radius narrowed to that precision.  Returns a list of index arrays
    (ascending) and the matching squared distances."""
    points = np.ascontiguousarray(points)
    t = points.dtype.type
    r2 = t(ball_radius)
    n = points.shape[0]
    nbrs, d2s = [], []
    for a in range(0, n, chunk):
        q = points[a:a + chunk]
        d = q[:, None, :] - points[None, :, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        inside = d2 < r2
        for i in range(q.shape[0]):
            j = np.nonzero(inside[i])[0]
            nbrs.append(j)
            d2s.append(d2[i, j])
    return nbrs, d2s


def estimate_point_cloud_normals_ball(points, ball_radius, view_directions=None, drop_angle_threshold=np.deg2rad(90.0),
                                      min_pts_per_ball=3, max_pts_per_ball=-1, weight_function="constant"):
    """src/point_cloud_normals.cpp:48-113 + :303-370 restated (max_pts_per_ball <= 0 only: with a cap the reference fits a
    rand()-dependent subset, which no oracle can reproduce).  Neighbourhoods by brute force with the reference's rounded
    metric; weights and offsets as the reference forms them (difference in the cloud's precision, times the double
    weight); numpy's LAPACK SVD stands in for Eigen's JacobiSVD.  PARITY UNPINNED for the normal vector itself (as for
    the k-NN variant); the neighbour sets, hence the kept indices without view directions, are exact by construction."""
    points = np.asarray(points)
    if not ball_radius > 0.0:
        raise ValueError("Invalid radius (%f) must be greater than 0." % ball_radius)
    if min_pts_per_ball < 3:
        raise ValueError("Invalid min_pts_per_ball (%d) must be greater than 3." % min_pts_per_ball)
    if max_pts_per_ball > 0:
        raise ValueError("the oracle does not model the reference's random subset (max_pts_per_ball > 0)")
    if weight_function not in ("constant", "rbf"):
        raise ValueError("Invalid weight_function, must be one of 'constant' or 'rbf'.")
    n = points.shape[0]
    has_dirs = view_directions is not None and np.asarray(view_directions).shape[0] != 0
    nbrs, d2s = ball_neighbourhoods(points, ball_radius)
    kept, normals = [], []
    for i in range(n):
        j = nbrs[i]
        if len(j) < min_pts_per_ball:
            continue
        w = np.ones(len(j))
        if weight_function == "rbf":
            r = np.sqrt(d2s[i].astype(np.float64)) / float(ball_radius)
            w = (1.0 - r) ** 4 * (4 * r + 1.0)
        offsets = (points[j] - points[i]).astype(np.float64) * w[:, None]
        _, _, vt = np.linalg.svd(offsets, full_matrices=False)
        normal = vt[2].copy()
        if has_dirs:
            dirv = np.asarray(view_directions[i], dtype=np.float64)
            normal *= np.sign(normal @ dirv)
            with np.errstate(invalid="ignore"):
                if np.arccos(normal @ dirv) > drop_angle_threshold:
                    continue
        kept.append(i)
        normals.append(normal)
    return np.array(kept, dtype=np.int64), np.array(normals, dtype=np.float64).reshape(-1, 3).astype(points.dtype)


# ---- voxel-grid down-sampling (src/sample_point_cloud.cpp:163-244, point_cloud_utils/__init__.py:123-200) ----
def voxel_indices(points, voxel_size, min_bound):
    """:201-206 -- int(floor((p - min_bound) / voxel_size)) per axis, in the cloud's precision (the binding casts the
    double arguments to the cloud's scalar type first, :346-354)."""
    points = np.asarray(points)
    t = points.dtype.type
    size = np.array([t(v) for v in voxel_size], dtype=points.dtype)
    lo = np.array([t(v) for v in min_bound], dtype=points.dtype)
    return np.floor((points - lo) / size).astype(np.int32)


def downsample_point_cloud_on_voxel_grid(voxel_size, points, *attribs, min_bound=None, max_bound=None, min_points_per_voxel=1,
                                         return_counts=False):
    """The wrapper (:123-200) and the accumulation (:163-244) restated with numpy: voxel membership exactly as the
    reference computes it; sums point after point in the ARRAY's precision like AccumulatedPoint::AddPoint (:119-128) --
    np.add.at accumulates in input order -- and the division of GetAveragePoint (:130-137).  The reference emits voxels
    in std::unordered_map iteration order, which is unspecified: rows are returned here in the order of each voxel's
    first point, and tests compare row SETS.  PARITY: the integer part (membership, counts, number of rows) is pinned by
    construction of the index arithmetic; no golden vector of the reference exists for the means (its build needs
    numpyeigen / Eigen, which are not in the tree)."""
    points = np.asarray(points)
    vs = np.array([voxel_size] * 3, dtype=np.float64) if np.isscalar(voxel_size) else np.array(voxel_size, dtype=np.float64)
    if len(vs) != 3:
        raise ValueError("Invalid voxel size must be a 3-tuple or a single float")
    lo = np.min(points, axis=0) - vs * 0.5 if min_bound is None else np.array(min_bound)
    hi = np.max(points, axis=0) + vs * 0.5 if max_bound is None else np.array(max_bound)
    if np.any(hi - lo <= 0.0):
        raise ValueError("Invalid min_bound and max_bound. max_bound must be greater than min_bound in all dimensions")
    t = points.dtype.type
    for a in range(3):
        if t(vs[a]) <= 0:
            raise ValueError("Voxel size is negative")
        if t(vs[a]) * t(2147483647) < t(hi[a]) - t(lo[a]):
            raise ValueError("Voxel size is too small")
    idx = voxel_indices(points, vs, lo)
    _, first, inverse, counts = np.unique(idx, axis=0, return_index=True, return_inverse=True, return_counts=True)
    inverse = inverse.reshape(-1)
    order = np.argsort(first, kind="stable")                 # voxels by their first point
    rank = np.empty_like(order); rank[order] = np.arange(len(order))
    group = rank[inverse]
    counts = counts[order]
    keep = counts >= min_points_per_voxel
    outs = []
    for arr in (points,) + tuple(np.asarray(a) for a in attribs):
        flat = arr.reshape(arr.shape[0], -1)
        acc = np.zeros((len(counts), flat.shape[1]), dtype=flat.dtype)
        np.add.at(acc, group, flat)                           # sequential, in input order, in the array's precision
        mean = acc / counts[:, None].astype(flat.dtype)
        outs.append(mean[keep].reshape((int(keep.sum()),) + arr.shape[1:]))
    if return_counts:
        outs.append(counts[keep].astype(np.int32))
    return tuple(outs) if len(outs) > 1 else outs[0]


# ---- duplicate removal (src/remove_duplicates.cpp:11-79, :108-176; libigl's round + unique_rows) ----
def deduplicate_point_cloud(points, epsilon, return_index=True):
    """remove_duplicate_vertices (:11-34) restated with numpy.  The reference calls libigl, which is fetched at build
    time and is NOT in the reference tree (PARITY UNPINNED: no golden vector exists and the reference cannot be built
    here; anchored on the published algorithm of igl::round / igl::unique_rows / igl::sortrows and on the properties
    the reference's own test asserts, tests/test_examples.py:509-520):
      epsilon > 0: rV = round(V / epsilon) -- division in V's precision, std::round (halves away from zero) -- and the
      unique rows of rV; else the unique rows of V.  unique_rows = ascending lexicographic row sort, one row per run;
      SVI = an input row of every run (libigl: whichever its non-stable std::sort puts first; here, like np.unique,
      the smallest), SVJ = run of every input row; SV = V[SVI]."""
    points = np.asarray(points)
    t = points.dtype.type
    if epsilon > 0:
        q = points / t(epsilon)
        # std::round: nearest integer, halves away from zero.  (floor(q + 0.5) would be wrong where q + 0.5 rounds up,
        # e.g. q = 0.49999997f; q - trunc(q) is exact.)
        frac = q - np.trunc(q)
        keyed = np.trunc(q) + np.where(np.abs(frac) >= t(0.5), np.sign(q), 0).astype(points.dtype)
    else:
        keyed = points
    keyed = keyed + t(0)                                                          # -0 -> +0 (they compare equal)
    _, svi, svj = np.unique(keyed, axis=0, return_index=True, return_inverse=True)
    svi = svi.astype(np.int32)
    svj = np.asarray(svj).reshape(-1).astype(np.int32)
    sv = points[svi]
    return (sv, svi, svj) if return_index else sv


def deduplicate_mesh_vertices(v, f, epsilon, return_index=True):
    """:36-77 restated: vertices as above; every face is re-indexed through SVJ and dropped when two corners coincide."""
    v = np.asarray(v)
    f = np.asarray(f)
    sv, svi, svj = deduplicate_point_cloud(v, epsilon, True)
    mapped = svj[f].astype(f.dtype)
    degenerate = np.zeros(len(f), dtype=bool)
    for c in range(f.shape[1]):
        for c2 in range(c + 1, f.shape[1]):
            degenerate |= mapped[:, c] == mapped[:, c2]
    sf = mapped[~degenerate]
    return (sv, sf, svi, svj) if return_index else (sv, sf)


# ---- Morton codes (src/morton.cpp, src/common/morton_code.cpp) -----------------------------------------------
_MORTON_PORT = os.path.join(_HERE, "libpcu_oracle_morton.so")
_MORTON_REF = os.path.join(_HERE, "_ref", "libpcu_ref_morton.so")


def have_morton_reference():
    return os.path.exists(_MORTON_REF)


def _morton_lib(impl):
    if impl is None:
        impl = "reference" if have_morton_reference() else "port"
    key = "morton_" + impl
    if key not in _libs:
        if impl == "port" and not os.path.exists(_MORTON_PORT):
            build()
        _libs[key] = (ctypes.CDLL(_MORTON_PORT if impl == "port" else _MORTON_REF), "pcu_oracle" if impl == "port" else "pcu_ref")
    return _libs[key]


def _codes(a, name):
    a = np.asarray(a)
    if a.dtype not in (np.uint32, np.uint64):
        raise ValueError("%s must have dtype uint32 or uint64" % name)
    if a.size == 0:
        raise ValueError("%s must be an array of shape [n] but got an empty array" % name)
    return np.ascontiguousarray(a.reshape(-1), dtype=np.uint64)


def morton_encode(pts, impl=None):
    """morton.cpp:185-239: (n, 3) int32 / int64 -> (n,) uint64."""
    pts = np.asarray(pts)
    if pts.dtype not in (np.int32, np.int64):
        raise ValueError("pts must have dtype int32 or int64")
    if pts.ndim != 2 or pts.shape[0] == 0:
        raise ValueError("pts must be an array of shape [n, 3] but got an empty array")
    if pts.shape[1] != 3:
        raise ValueError("pts must be an array of shape [n, 3] but got an invalid number of columns")
    p32 = np.ascontiguousarray(pts.astype(np.int32))          # int32_t px = pts(i, 0)
    out = np.empty(p32.shape[0], np.uint64)
    lib, prefix = _morton_lib(impl)
    getattr(lib, prefix + "_morton_encode")(_vp(p32.ctypes.data), _c_i64(p32.shape[0]), _vp(out.ctypes.data))
    return out


def morton_decode(codes, impl=None):
    """morton.cpp:253-310: (n,) -> (n, 3) int32."""
    c = _codes(codes, "codes")
    out = np.empty((c.shape[0], 3), np.int32)
    lib, prefix = _morton_lib(impl)
    getattr(lib, prefix + "_morton_decode")(_vp(c.ctypes.data), _c_i64(c.shape[0]), _vp(out.ctypes.data))
    return out


def _morton_binary(name, a, b, impl):
    a, b = _codes(a, "codes_1"), _codes(b, "codes_2")
    if a.shape != b.shape:
        raise ValueError("codes_1 and codes_2 must have the same number of entries.")
    out = np.empty_like(a)
    lib, prefix = _morton_lib(impl)
    getattr(lib, prefix + name)(_vp(a.ctypes.data), _vp(b.ctypes.data), _c_i64(a.shape[0]), _vp(out.ctypes.data))
    return out


def morton_add(codes_1, codes_2, impl=None):
    """morton.cpp:26-103."""
    return _morton_binary("_morton_add", codes_1, codes_2, impl)


def morton_subtract(codes_1, codes_2, impl=None):
    """morton.cpp:106-183."""
    return _morton_binary("_morton_subtract", codes_1, codes_2, impl)


def morton_knn(codes, qcodes, k, sort_dist=True, impl=None):
    """morton.cpp:324-414.  The window of positions is the reference's; with sort_dist the rows are ordered by squared
    distance to the query point, ties by position -- the INTENDED order (the reference's comparator reads three
    uninitialised variables, :381-398, so its own order is undefined and cannot be pinned)."""
    if k <= 0:
        raise ValueError("k must be greater than 0")
    c, q = _codes(codes, "codes"), _codes(qcodes, "qcodes")
    k = min(int(k), c.shape[0])
    out = np.empty((q.shape[0], k), np.int64)
    lib, prefix = _morton_lib(impl)
    getattr(lib, prefix + "_morton_knn_window")(_vp(c.ctypes.data), _c_i64(c.shape[0]), _vp(q.ctypes.data), _c_i64(q.shape[0]),
                                                _c_int(k), _vp(out.ctypes.data))
    if sort_dist:
        pts = morton_decode(c, impl=impl).astype(np.float64)
        qp = morton_decode(q, impl=impl).astype(np.float64)
        d = ((pts[out] - qp[:, None, :]) ** 2).sum(-1)
        order = np.argsort(d, axis=1, kind="stable")   # the window ascends in position, so stable = ties by position
        out = np.take_along_axis(out, order, axis=1)
    return out


def kd_tree(dataset_points, max_points_per_leaf=10):
    """The restatement's built tree (order[] = nanoflann's vAcc, plus the node table), for checking
    GPU-side replicas of the build."""
    d = np.ascontiguousarray(dataset_points)
    lib, _ = _lib("port")
    sfx = "f32" if d.dtype == np.float32 else "f64"
    fn = getattr(lib, "pcu_oracle_tree_" + sfx)
    fn.restype = _c_i64
    fn.argtypes = [_vp, _c_i64, _c_int, _vp, _c_i64] + [_vp] * 7
    m = d.shape[0]
    cap = 2 * m + 16
    order = np.empty(m, np.int64)
    feat = np.empty(cap, np.int32)
    lo = np.empty(cap, d.dtype)
    hi = np.empty(cap, d.dtype)
    first = np.empty(cap, np.int64)
    last = np.empty(cap, np.int64)
    k0 = np.empty(cap, np.int32)
    k1 = np.empty(cap, np.int32)
    nn = fn(d.ctypes.data, m, int(max_points_per_leaf), order.ctypes.data, cap, feat.ctypes.data, lo.ctypes.data,
            hi.ctypes.data, first.ctypes.data, last.ctypes.data, k0.ctypes.data, k1.ctypes.data)
    return dict(order=order, feat=feat[:nn], div_lo=lo[:nn], div_hi=hi[:nn], first=first[:nn], last=last[:nn],
                kid0=k0[:nn], kid1=k1[:nn])
