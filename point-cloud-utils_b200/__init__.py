"""pcu_b200 -- B200-native drop-in for the nearest-neighbour path of point-cloud-utils.

The four callables keep the reference's names, signatures, defaults and conventions
(/root/reference/point_cloud_utils/__init__.py:4-16, :52-120 and
/root/reference/src/point_cloud_distance.cpp:123-131, :186-193):

    k_nearest_neighbors(query_points, dataset_points, k, squared_distances=False,
                        max_points_per_leaf=10, num_threads=-1)        -> (dists, corrs)
    one_sided_hausdorff_distance(source, target, return_index=True, squared_distances=False,
                        max_points_per_leaf=10)                       -> d | (d, i, j)
    hausdorff_distance(x, y, return_index=False, squared_distances=False,
                        max_points_per_leaf=10)                       -> d | (d, i, j)
    chamfer_distance(x, y, return_index=False, p_norm=2, max_points_per_leaf=10)
                                                                      -> c | (c, corrs_x_to_y, corrs_y_to_x)

plus ``batched_chamfer_distance`` (the "[m, n, d] minibatch" the reference's docstring promises at
__init__.py:89-90 but its 2-D-only binding never delivered).

Inputs may be numpy arrays (results come back as numpy / Python scalars, exactly like the
reference) or CUDA ``torch`` tensors (nothing leaves the device: results are CUDA tensors and the
call does not synchronise unless a Python scalar has to be produced).

Everything is computed by hand-written sm_100a kernels behind the C ABI in include/pcu_b200.h.
There is deliberately NO CPU fallback: importing this package without its compiled extension, or
calling it without a Blackwell GPU, raises.
"""
import importlib as _importlib

import numpy as _np

try:
    from . import _pcu_internal
except ImportError as _e:  # pragma: no cover - exercised only on a broken install
    raise ImportError(
        "pcu_b200: the compiled extension (_pcu_internal / libpcu_b200.so) is missing or failed to load: %s.\n"
        "Build it in-tree with `python -c 'import __graft_entry__ as g; g.build()'` from the repository root.\n"
        "There is no pure-Python or CPU fallback for this package." % (_e,)) from _e

__all__ = ["k_nearest_neighbors", "one_sided_hausdorff_distance", "hausdorff_distance", "chamfer_distance",
           "batched_chamfer_distance", "estimate_point_cloud_normals_knn", "estimate_point_cloud_normals_ball",
           "morton_encode", "morton_decode", "morton_add", "morton_subtract", "morton_knn", "pairwise_distances", "sinkhorn",
           "earth_movers_distance", "downsample_point_cloud_on_voxel_grid", "downsample_point_cloud_poisson_disk",
           "deduplicate_point_cloud",
           "deduplicate_mesh_vertices", "prepare_cloud", "pinned_empty", "PreparedCloud", "device_count",
           "current_device", "launch_count"]

_STATS_WORDS = 10  # sizeof(pcu_b200_nn_stats) / 8


def device_count():
    """Number of visible GPUs this build can run on (compute capability 10.x)."""
    return _pcu_internal._device_count()


def current_device():
    """The GPU a numpy-input call runs on when no ``device=`` is given: ``PCU_B200_DEVICE`` if set, else the CUDA
    runtime's current device when it is not 0 (``torch.cuda.set_device`` / ``with torch.cuda.device(i)``), else
    ``LOCAL_RANK`` (torchrun) when that many devices are visible, else 0.  CUDA tensors always run where they live."""
    return _pcu_internal._current_device()


def _dev(device):
    """``device=`` keyword -> ordinal for the native layer (-1: let the library choose, see current_device)."""
    if device is None:
        return -1
    if isinstance(device, int):
        d = device
    elif isinstance(device, str):
        name = device.strip().lower()
        if name == "cuda":
            return -1
        if not name.startswith("cuda:") or not name[5:].isdigit():
            raise ValueError("device must be an int, None, 'cuda' or 'cuda:<i>' (got %r)" % (device,))
        d = int(name[5:])
    elif getattr(device, "type", None) == "cuda":           # torch.device
        d = -1 if device.index is None else int(device.index)
    else:
        raise ValueError("device must be an int, None, 'cuda', 'cuda:<i>' or a CUDA torch.device (got %r)" % (device,))
    if d >= device_count() or d < -1:
        raise ValueError("device %d out of range: %d usable GPU(s) visible" % (d, device_count()))
    return d


def launch_count():
    """Kernels launched by the native library in this process so far."""
    return _pcu_internal._launch_count()


# ---------------------------------------------------------------------------------------------
# torch plumbing (device residency only; no torch op sits on the hot path)
def _torch():
    try:
        return _importlib.import_module("torch")
    except ImportError:  # pragma: no cover
        return None


def _is_tensor(x):
    t = _torch() if type(x).__module__.startswith("torch") else None
    return t is not None and isinstance(x, t.Tensor)


def _check_tensor_pair(a, b, name_a, name_b):
    torch = _torch()
    if not _is_tensor(b):
        raise ValueError("%s and %s must both be torch tensors or both be numpy arrays" % (name_a, name_b))
    if a.dtype not in (torch.float32, torch.float64):
        raise ValueError("Invalid scalar type (%s) for argument '%s'. Expected one of ['float32', 'float64']."
                         % (a.dtype, name_a))
    if b.dtype != a.dtype:
        raise ValueError("Invalid scalar type (%s) for argument '%s'. Expected it to match argument '%s' which is "
                         "of type %s." % (b.dtype, name_b, name_a, a.dtype))
    if a.device != b.device:
        raise ValueError("%s and %s must live on the same device" % (name_a, name_b))
    shapes = "Got %s.shape = %s, %s.shape = %s." % (name_a, tuple(a.shape), name_b, tuple(b.shape))
    if a.dim() != 2 or b.dim() != 2 or a.shape[1] != 3 or b.shape[1] != 3:
        raise ValueError("Only 3D inputs are supported: %s and %s must have shape (n, 3) and (m, 3). %s"
                         % (name_a, name_b, shapes))
    if a.shape[0] == 0 or b.shape[0] == 0:
        raise ValueError("Invalid input set with zero elements: %s and %s must have shape (n, 3) and (m, 3). %s"
                         % (name_a, name_b, shapes))
    return a.detach().contiguous(), b.detach().contiguous()


def _same_device(t, device):
    """CUDA tensors run where they live; a contradicting device= is an argument error."""
    d = _dev(device)
    if d >= 0 and d != (t.device.index or 0):
        raise ValueError("device=%r contradicts the inputs, which live on %s" % (device, t.device))


def _stream_of(t):
    torch = _torch()
    return torch.cuda.current_stream(t.device).cuda_stream


def _stats_from_tensor(buf, which):
    """Decode one pcu_b200_nn_stats from the raw device buffer (synchronises)."""
    host = buf.cpu()
    f = host.view(_torch().float64)
    i = host.view(_torch().int64)
    o = _STATS_WORDS * which
    return {"sum_dist": float(f[o]), "sum_sq_dist": float(f[o + 1]), "max_sq_dist": float(f[o + 2]),
            "argmax_query": int(i[o + 3]), "argmax_data": int(i[o + 4]), "n_queries": int(i[o + 5]),
            "n_tied": int(i[o + 6]), "n_far": int(i[o + 7]), "witness_tied": int(i[o + 8]),
            "pair_value": float(f[o + 9])}


def _resolved_stats(buf, which, q, d, leaf):
    """Stats record `which` of `buf`; when its Hausdorff witness hinges on tie order, have the device replay it."""
    st = _stats_from_tensor(buf, which)
    if st["witness_tied"]:
        torch = _torch()
        _pcu_internal._resolve_witness_device(q.dtype == torch.float64, q.data_ptr(), q.shape[0], d.data_ptr(),
                                              d.shape[0], buf.data_ptr() + 8 * _STATS_WORDS * which, int(leaf),
                                              q.device.index or 0, _stream_of(q))
        st = _stats_from_tensor(buf, which)
    return st


def _stats_device(a, b, both, leaf):
    torch = _torch()
    assert _pcu_internal._stats_nbytes() == 8 * _STATS_WORDS
    buf = torch.empty(2 * _STATS_WORDS, dtype=torch.int64, device=a.device)   # every record is written by the sweep
    val = torch.empty((), dtype=a.dtype, device=a.device)
    _pcu_internal._stats_device(a.dtype == torch.float64, both, a.data_ptr(), a.shape[0], b.data_ptr(), b.shape[0],
                                buf.data_ptr(), val.data_ptr() if both else 0, int(leaf), a.device.index or 0,
                                _stream_of(a))
    return buf, val


def _metric_value(max_sq, squared, dtype):
    d2 = dtype(max_sq)
    return float(d2 if squared else _np.sqrt(d2))


# ---------------------------------------------------------------------------------------------
class PreparedCloud:
    """A point cloud binned once on the GPU (``prepare_cloud``), to be passed as the SECOND argument -- y / target /
    dataset_points -- of ``chamfer_distance``, ``hausdorff_distance``, ``one_sided_hausdorff_distance`` and
    ``k_nearest_neighbors`` as often as wanted: every such call bins only its first argument (and, for numpy inputs,
    copies only that one over PCIe).  Prepared with ``k=...`` the handle also owns the reference's kd-tree replica, so
    k-NN calls neither bin the dataset nor build the tree -- they only replay their tied rows on it.  The reference rebuilds
    its kd-tree three times per direction on every call (/root/reference/src/point_cloud_distance.cpp:41-42).
    Results are those of the plain calls.  Holds a private copy of the points; ``close()`` (or garbage collection)
    frees the device memory."""

    def __init__(self, handle, n, is_f64, device_index, on_device, knn_k=None, max_points_per_leaf=None):
        self._handle, self.shape, self._f64, self.device_index, self._on_device = handle, (int(n), 3), bool(is_f64), int(device_index), on_device
        self.k, self.max_points_per_leaf = knn_k, max_points_per_leaf     # set when prepared for k-NN calls

    @property
    def dtype(self):
        return _np.dtype(_np.float64 if self._f64 else _np.float32)

    def close(self):
        if self._handle:
            _pcu_internal._cloud_destroy(self._handle)
            self._handle = 0

    def __del__(self):
        try:
            self.close()
        except Exception:   # interpreter shutdown
            pass

    def __len__(self):
        return self.shape[0]


def prepare_cloud(points, *, k=None, max_points_per_leaf=10, device=None):
    """Bin ``points`` ((n, 3) float32 / float64 numpy array or CUDA tensor) once; returns a ``PreparedCloud``.
    ``k``: the handle is meant as the dataset of ``k_nearest_neighbors`` calls with (about) this k -- the cell size is
    chosen for it and the reference tree for ``max_points_per_leaf`` is built into the handle (any k works on any
    handle; results never depend on it)."""
    kk = 0 if k is None else int(k)
    if k is not None and kk <= 0:
        raise ValueError("Invalid value for k (%d) must be greater than 0." % kk)
    if int(max_points_per_leaf) <= 0:
        raise ValueError("max_points_per_leaf must be greater than 0.")
    meta = dict(knn_k=(kk or None), max_points_per_leaf=(int(max_points_per_leaf) if kk else None))
    if _is_tensor(points):
        torch = _torch()
        if points.dtype not in (torch.float32, torch.float64) or points.dim() != 2 or points.shape[1] != 3 or points.shape[0] == 0:
            raise ValueError("points must be a float32 / float64 tensor of shape (n, 3) with n > 0")
        if not points.is_cuda:
            return prepare_cloud(points.detach().numpy(), k=k, max_points_per_leaf=max_points_per_leaf, device=device)
        _same_device(points, device)
        p = points.detach().contiguous()
        dev = p.device.index or 0
        h = _pcu_internal._cloud_prepare_device(p.dtype == torch.float64, p.data_ptr(), p.shape[0], dev, _stream_of(p), kk,
                                                int(max_points_per_leaf))
        return PreparedCloud(h, p.shape[0], p.dtype == torch.float64, dev, True, **meta)
    pts = _np.asarray(points)
    d = _dev(device)
    h = _pcu_internal._cloud_prepare(pts, d, kk, int(max_points_per_leaf))
    return PreparedCloud(h, pts.shape[0], pts.dtype == _np.float64, _pcu_internal._current_device() if d < 0 else d, False, **meta)


def pinned_empty(n, dtype=_np.float32, cols=3, *, device=None):
    """An uninitialised (n, cols) numpy array in page-locked host memory placed next to the GPU (the NUMA node of the
    PCI device), for callers that fill their clouds in place and pass them to the numpy-facing functions: such inputs
    are copied by DMA straight from where they are, at the link's rate (24 MB in 0.44 ms).  Ordinary numpy arrays work
    as well -- they go through the library's own page-locked ring (0.8 ms for the same call instead of 0.66); what is
    slow is page-locked memory on the OTHER socket (torch's ``pin_memory()`` lands wherever the calling thread happens
    to run).  Not in the reference."""
    dt = _np.dtype(dtype)
    if dt not in (_np.dtype(_np.float32), _np.dtype(_np.float64)):
        raise ValueError("dtype must be float32 or float64")
    d = _dev(device)
    if d >= 0:
        torch = _torch()
        with torch.cuda.device(d):
            return _pcu_internal._pinned_empty(int(n), int(cols), dt == _np.dtype(_np.float64))
    return _pcu_internal._pinned_empty(int(n), int(cols), dt == _np.dtype(_np.float64))


def _prepared_resolved(buf, which, xs, cloud, leaf):
    """Record `which` of a prepared-cloud call on device tensors, its Hausdorff witness replayed when tie order decided it."""
    st = _stats_from_tensor(buf, which)
    if st["witness_tied"]:
        yp, m = _pcu_internal._cloud_points(cloud._handle), cloud.shape[0]
        q, n, d, k = (xs.data_ptr(), xs.shape[0], yp, m) if which == 0 else (yp, m, xs.data_ptr(), xs.shape[0])
        _pcu_internal._resolve_witness_device(cloud._f64, q, n, d, k, buf.data_ptr() + 8 * _STATS_WORDS * which, int(leaf),
                                              cloud.device_index, _stream_of(xs))
        st = _stats_from_tensor(buf, which)
    return st


def _prepared_stats(x, cloud, both, leaf, device):
    """(where, dtype, value, payload) like _both_stats, for a PreparedCloud second argument."""
    if not cloud._handle:
        raise ValueError("the PreparedCloud has been closed")
    if _is_tensor(x) and x.is_cuda:
        torch = _torch()
        if x.dtype != (torch.float64 if cloud._f64 else torch.float32) or x.dim() != 2 or x.shape[1] != 3 or x.shape[0] == 0:
            raise ValueError("the first argument must be an (n, 3) tensor of the prepared cloud's dtype (%s)" % cloud.dtype)
        if (x.device.index or 0) != cloud.device_index:
            raise ValueError("the points live on %s, the prepared cloud on cuda:%d" % (x.device, cloud.device_index))
        xs = x.detach().contiguous()
        buf = torch.empty(2 * _STATS_WORDS, dtype=torch.int64, device=xs.device)
        val = torch.empty((), dtype=xs.dtype, device=xs.device)
        _pcu_internal._stats_prepared_device(cloud._f64, both, xs.data_ptr(), xs.shape[0], cloud._handle, buf.data_ptr(),
                                             val.data_ptr() if both else 0, int(leaf), cloud.device_index, _stream_of(xs))
        return "cuda", xs.dtype, val, (buf, xs)
    if _is_tensor(x):
        x = x.detach().numpy()
    d = _dev(device)
    if d >= 0 and d != cloud.device_index:
        raise ValueError("device=%r contradicts the prepared cloud, which lives on cuda:%d" % (device, cloud.device_index))
    res = _pcu_internal._stats_prepared(_np.asarray(x), cloud._handle, cloud._f64, both, int(leaf), cloud.device_index)
    return "host", cloud.dtype.type, res[0], res[1:]


# ---------------------------------------------------------------------------------------------
def k_nearest_neighbors(query_points, dataset_points, k, squared_distances=False, max_points_per_leaf=10,
                        num_threads=-1, *, device=None):
    """
    Compute the k nearest neighbors (L2 distance) from each point in the query point cloud to the dataset point cloud.

    Args:
        query_points : n by 3 array of representing a set of n points (each row is a point of dimension 3).
        dataset_points : m by 3 array of representing a set of m points (each row is a point of dimension 3).
        k : the number of nearest neighbors to query per point.
        squared_distances : If set to True, then return squared L2 distances. Default is False.
        max_points_per_leaf : The maximum number of points per leaf node in the KD tree of the reference. Here it
                              only decides how exactly-equal distances are ordered (identically to the reference).
        num_threads : CPU thread count of the reference implementation; accepted and ignored.
        device : (keyword only, not in the reference) GPU for numpy / CPU-tensor inputs: an ordinal, 'cuda:<i>' or a
                 torch.device; None = `current_device()`.  CUDA tensors run on the device they live on.

    Returns:
        dists : An (n, k)-shaped array such that `dists[i,k]` contains the k^th shortest L2 distance from the point
                `query_points[i, :]` to `dataset_points` ((n,) when k == 1; -1.0 where fewer than k points exist)
        corrs : An (n, k)-shaped int64 array such that `corrs[i,k]` contains the index into `dataset_points` of the
                k^th nearest point to `query_points[i, :]` ((n,) when k == 1; -1 where fewer than k points exist)

    Mirrors /root/reference/src/point_cloud_distance.cpp:123-164.
    """
    if isinstance(dataset_points, PreparedCloud):
        return _knn_prepared(query_points, dataset_points, int(k), bool(squared_distances), int(max_points_per_leaf), device)
    if _is_tensor(query_points) or _is_tensor(dataset_points):
        torch = _torch()
        if not _is_tensor(query_points):
            raise ValueError("query_points and dataset_points must both be torch tensors or both be numpy arrays")
        if int(k) <= 0:
            raise ValueError("Invalid value for k (%d) must be greater than 0." % int(k))
        q, d = _check_tensor_pair(query_points, dataset_points, "query_points", "dataset_points")
        if not q.is_cuda:
            dn, cn = _pcu_internal.k_nearest_neighbors(q.numpy(), d.numpy(), int(k), bool(squared_distances),
                                                       int(max_points_per_leaf), int(num_threads), _dev(device))
            return torch.from_numpy(_np.asarray(dn)), torch.from_numpy(_np.asarray(cn))
        _same_device(q, device)
        n = q.shape[0]
        dists = torch.empty((n, int(k)), dtype=q.dtype, device=q.device)
        corrs = torch.empty((n, int(k)), dtype=torch.int64, device=q.device)
        _pcu_internal._knn_device(q.dtype == torch.float64, q.data_ptr(), n, d.data_ptr(), d.shape[0], int(k),
                                  bool(squared_distances), dists.data_ptr(), corrs.data_ptr(), 0,
                                  int(max_points_per_leaf), q.device.index or 0, _stream_of(q))
        return dists.squeeze(), corrs.squeeze()
    return _pcu_internal.k_nearest_neighbors(_np.asarray(query_points), _np.asarray(dataset_points), int(k),
                                             bool(squared_distances), int(max_points_per_leaf), int(num_threads),
                                             _dev(device))


def _knn_prepared(query_points, cloud, k, squared, leaf, device):
    """k_nearest_neighbors against a PreparedCloud: numpy in -> numpy out, CUDA tensor in -> CUDA tensors out."""
    if not cloud._handle:
        raise ValueError("the prepared cloud has been closed")
    if k <= 0:
        raise ValueError("Invalid value for k (%d) must be greater than 0." % k)
    if _is_tensor(query_points) and query_points.is_cuda:
        torch = _torch()
        q = query_points.detach().contiguous()
        if q.dtype != (torch.float64 if cloud._f64 else torch.float32) or q.dim() != 2 or q.shape[1] != 3 or q.shape[0] == 0:
            raise ValueError("query_points must be a non-empty (n, 3) tensor of the prepared cloud's precision (%s)" % cloud.dtype)
        if (q.device.index or 0) != cloud.device_index:
            raise ValueError("query_points live on %s, the prepared cloud on device %d" % (q.device, cloud.device_index))
        _same_device(q, device)
        n = q.shape[0]
        dists = torch.empty((n, k), dtype=q.dtype, device=q.device)
        corrs = torch.empty((n, k), dtype=torch.int64, device=q.device)
        _pcu_internal._knn_prepared_device(cloud._f64, q.data_ptr(), n, cloud._handle, k, squared, dists.data_ptr(),
                                           corrs.data_ptr(), 0, leaf, cloud.device_index, _stream_of(q))
        return dists.squeeze(), corrs.squeeze()
    as_tensor = _is_tensor(query_points)
    qn = query_points.detach().numpy() if as_tensor else _np.asarray(query_points)
    d = _dev(device)
    if d >= 0 and d != cloud.device_index:
        raise ValueError("device=%d was given but the prepared cloud lives on device %d" % (d, cloud.device_index))
    dn, cn = _pcu_internal._knn_prepared(qn, cloud._handle, cloud._f64, k, squared, leaf, cloud.device_index)
    if as_tensor:
        torch = _torch()
        return torch.from_numpy(_np.asarray(dn)), torch.from_numpy(_np.asarray(cn))
    return dn, cn


def one_sided_hausdorff_distance(source, target, return_index=True, squared_distances=False, max_points_per_leaf=10,
                                 *, device=None):
    """
    Compute the one sided Hausdorff distance from source to target

    Args:
        source : n by 3 array of representing a set of n points (each row is a point of dimension 3)
        target : m by 3 array of representing a set of m points (each row is a point of dimension 3)
        return_index : Optionally return the index pair `(i, j)` into source and target such that `source[i, :]` and
                       `target[j, :]` are the two points with maximum shortest distance. Default is True (as in the
                       reference binding).
        squared_distances : If set to True, then return squared L2 distances.
        max_points_per_leaf : see `k_nearest_neighbors`.
        device : see `k_nearest_neighbors` (keyword only).

    Returns:
        d : The largest shortest distance, `d` between each point in `source` and the points in `target` (a float).
        i, j : ints such that `source[i, :]` and `target[j, :]` are the two points with maximum shortest distance.

    Mirrors /root/reference/src/point_cloud_distance.cpp:186-234.  One fused sweep: no per-point distance array
    is written; the maximum, its first row and that row's neighbour are reduced inside the search kernel.
    """
    if isinstance(target, PreparedCloud):
        where, dtype, _, payload = _prepared_stats(source, target, False, max_points_per_leaf, device)
        if where == "cuda":
            st = _prepared_resolved(payload[0], 0, payload[1], target, max_points_per_leaf)
            np_t = _np.float32 if dtype == _torch().float32 else _np.float64
        else:
            st, np_t = payload[0], dtype
        value = _metric_value(st["max_sq_dist"], squared_distances, np_t)
        return (value, st["argmax_query"], st["argmax_data"]) if return_index else value
    if _is_tensor(source) or _is_tensor(target):
        if not _is_tensor(source):
            raise ValueError("source and target must both be torch tensors or both be numpy arrays")
        s, t = _check_tensor_pair(source, target, "source", "target")
        if not s.is_cuda:
            return _pcu_internal.one_sided_hausdorff_distance(s.numpy(), t.numpy(), bool(return_index),
                                                              bool(squared_distances), int(max_points_per_leaf),
                                                              _dev(device))
        _same_device(s, device)
        buf, _ = _stats_device(s, t, False, max_points_per_leaf)
        st = _resolved_stats(buf, 0, s, t, max_points_per_leaf)
        value = _metric_value(st["max_sq_dist"], squared_distances,
                              _np.float32 if s.dtype == _torch().float32 else _np.float64)
        if return_index:
            return value, st["argmax_query"], st["argmax_data"]
        return value
    return _pcu_internal.one_sided_hausdorff_distance(_np.asarray(source), _np.asarray(target), bool(return_index),
                                                      bool(squared_distances), int(max_points_per_leaf), _dev(device))


def _both_stats(x, y, max_points_per_leaf, device=None):
    """(dtype, chamfer value, stats x->y, stats y->x) from ONE fused bidirectional launch sequence."""
    if isinstance(y, PreparedCloud):
        where, dtype, val, payload = _prepared_stats(x, y, True, max_points_per_leaf, device)
        if where == "cuda":
            return ("cuda-prepared", dtype, val, payload + (y,))
        return ("host", dtype, val, payload)
    if _is_tensor(x) or _is_tensor(y):
        if not _is_tensor(x):
            raise ValueError("x and y must both be torch tensors or both be numpy arrays")
        xs, ys = _check_tensor_pair(x, y, "x", "y")
        if xs.is_cuda:
            _same_device(xs, device)
            buf, val = _stats_device(xs, ys, True, max_points_per_leaf)
            return ("cuda", xs.dtype, val, (buf, xs, ys))
        x, y = xs.numpy(), ys.numpy()
    val, sxy, syx = _pcu_internal._chamfer_stats(_np.asarray(x), _np.asarray(y), int(max_points_per_leaf), _dev(device))
    return ("host", _np.asarray(x).dtype.type, val, (sxy, syx))


def hausdorff_distance(x, y, return_index=False, squared_distances=False, max_points_per_leaf=10, *, device=None):
    """
    Compute the Hausdorff distance between x and y

    Args:
        x : n by 3 array of representing a set of n points (each row is a point of dimension 3)
        y : m by 3 array of representing a set of m points (each row is a point of dimension 3)
        return_index : Optionally return the index pair `(i, j)` into x and y such that `x[i, :]` and `y[j, :]` are
                       the two points with maximum shortest distance.
        squared_distances : If set to True, then return squared L2 distances. Default is False.
        max_points_per_leaf : see `k_nearest_neighbors`.

    Returns:
        The largest shortest distance, `d` between each point in `source` and the points in `target`.
        If `return_index` is set, then this function returns a tuple (d, i, j) where `d` is as described above
        and `(i, j)` are such that `source[i, :]` and `target[j, :]` are the two points with maximum shortest
        distance.

    Mirrors /root/reference/point_cloud_utils/__init__.py:52-81 (two one-sided passes, `>` / `<=` branch rule);
    both directions come from one fused launch sequence over the two binned clouds.
    """
    where, dtype, _, st = _both_stats(x, y, max_points_per_leaf, device)
    if where == "cuda-prepared":
        buf, xs, cloud = st
        sxy = _prepared_resolved(buf, 0, xs, cloud, max_points_per_leaf)
        syx = _prepared_resolved(buf, 1, xs, cloud, max_points_per_leaf)
        np_t = _np.float32 if dtype == _torch().float32 else _np.float64
    elif where == "cuda":
        buf, xs, ys = st
        sxy = _resolved_stats(buf, 0, xs, ys, max_points_per_leaf)
        syx = _resolved_stats(buf, 1, ys, xs, max_points_per_leaf)
        np_t = _np.float32 if dtype == _torch().float32 else _np.float64
    else:
        sxy, syx = st
        np_t = dtype
    h_xy = _metric_value(sxy["max_sq_dist"], squared_distances, np_t)
    h_yx = _metric_value(syx["max_sq_dist"], squared_distances, np_t)
    hausdorff = max(h_xy, h_yx)
    if return_index and h_xy > h_yx:
        return hausdorff, sxy["argmax_query"], sxy["argmax_data"]
    elif return_index and h_xy <= h_yx:
        return hausdorff, syx["argmax_data"], syx["argmax_query"]
    return hausdorff


def chamfer_distance(x, y, return_index=False, p_norm=2, max_points_per_leaf=10, *, device=None):
    """
    Compute the chamfer distance between two point clouds x, and y

    Args:
        x : n by 3 array of points
        y : m by 3 array of points
        return_index: If set to True, will return a pair (corrs_x_to_y, corrs_y_to_x) where
                    corrs_x_to_y[i] stores the index into y of the closest point to x[i]
                    (i.e. y[corrs_x_to_y[i]] is the nearest neighbor to x[i] in y).
                    corrs_y_to_x is similar to corrs_x_to_y but with x and y reversed.
        max_points_per_leaf : see `k_nearest_neighbors`.
        p_norm : Which norm to use. p_norm can be any real number, inf (for the max norm) -inf (for the min norm),
                0 (for sum(x != 0)).  The nearest neighbour is always the L2 one, as in the reference.
    Returns:
        The chamfer distance between x an dy: mean_x |x - NN_y(x)|_p + mean_y |y - NN_x(y)|_p (no 1/2, not squared).
        If return_index is set, then this function returns a tuple (chamfer_dist, corrs_x_to_y, corrs_y_to_x).

    Mirrors /root/reference/point_cloud_utils/__init__.py:84-120.  With p_norm == 2 and return_index == False the
    whole computation is one fused bidirectional sweep (no index or distance array is materialised).
    """
    if p_norm == 2 and not return_index:
        where, _, val, _ = _both_stats(x, y, max_points_per_leaf, device)
        return val
    if isinstance(y, PreparedCloud):
        raise ValueError("a PreparedCloud serves the fused metrics (p_norm = 2, return_index = False); pass the array for the others")
    dists_x_to_y, corrs_x_to_y = k_nearest_neighbors(x, y, k=1, squared_distances=False,
                                                     max_points_per_leaf=max_points_per_leaf, device=device)
    dists_y_to_x, corrs_y_to_x = k_nearest_neighbors(y, x, k=1, squared_distances=False,
                                                     max_points_per_leaf=max_points_per_leaf, device=device)
    if _is_tensor(x):
        torch = _torch()
        if p_norm == 2:
            cham = dists_x_to_y.mean() + dists_y_to_x.mean()
        else:
            cham = torch.linalg.vector_norm(x[corrs_y_to_x.reshape(-1)] - y, ord=p_norm, dim=-1).mean() + \
                   torch.linalg.vector_norm(y[corrs_x_to_y.reshape(-1)] - x, ord=p_norm, dim=-1).mean()
    else:
        x = _np.asarray(x)
        y = _np.asarray(y)
        d1 = _np.linalg.norm(x[corrs_y_to_x] - y, axis=-1, ord=p_norm).mean()
        d2 = _np.linalg.norm(y[corrs_x_to_y] - x, axis=-1, ord=p_norm).mean()
        cham = _np.mean(d1) + _np.mean(d2)
    if return_index:
        return cham, corrs_x_to_y, corrs_y_to_x
    return cham


def estimate_point_cloud_normals_knn(points, num_neighbors, view_directions=None, drop_angle_threshold=_np.deg2rad(90.0),
                                     max_points_per_leaf=10, num_threads=-1, *, device=None):
    """
    Estimate normals for a point cloud by locally fitting a plane to the k nearest neighbors of each point.

    This function can optionally consider directions to the sensor for each point to align the final normal
    directions and to drop points whose normal deviates too much from the view direction.

    Args:
        points : (n, 3)-shaped NumPy array (or CUDA tensor) of point positions (each row is a point)
        num_neighbors : Integer number of neighbors to use in each neighborhood (the point itself counts as its own
                        nearest neighbor, as in the reference).
        view_directions : (n, 3)-shaped array or None, the unit direction to the sensor for each point.
        drop_angle_threshold : If view_directions is passed in, drop points whose angle between the normal and view
                               direction exceeds drop_angle_threshold (in radians).
        max_points_per_leaf : see `k_nearest_neighbors` (decides the neighbour set only among exactly equidistant points).
        num_threads : CPU thread count of the reference implementation; accepted and ignored.
        device : see `k_nearest_neighbors` (keyword only).

    Returns:
        idx : an (m,)-shaped int64 array of indices into points (the points that were kept, ascending)
        n : an (m, 3)-shaped array of unit normals for those points

    Mirrors /root/reference/point_cloud_utils/_pointcloud_normals.py:4-54 and
    /root/reference/src/point_cloud_normals.cpp:115-173, :375-411.  Neighbour sets are the reference's; the normal is the
    same plane-fit direction up to rounding (1e-6 in the dot product for well-separated singular values) and, when no
    view directions are given, up to sign -- the reference's sign is whatever Eigen's JacobiSVD returns.
    """
    if _is_tensor(points):
        torch = _torch()
        if points.dtype not in (torch.float32, torch.float64):
            raise ValueError("Invalid scalar type (%s) for argument 'points'. Expected one of ['float32', 'float64']." % points.dtype)
        if points.dim() != 2 or points.shape[-1] != 3:
            raise ValueError("Invalid shape for points, must be (n, 3) but got " + str(tuple(points.shape)))
        if points.shape[0] == 0:
            raise ValueError("Invalid point set with zero elements: points must have shape (n, 3)")
        if int(num_neighbors) <= 0:
            raise ValueError("Invalid number of neighbors (%d) must be greater than 0." % int(num_neighbors))
        dirs = None
        if view_directions is not None:
            if not _is_tensor(view_directions) or view_directions.dtype != points.dtype or \
                    view_directions.device != points.device or tuple(view_directions.shape) != tuple(points.shape):
                raise ValueError("Invalid view directions does not match the number of points. If view directions are passed "
                                 "in, they must be a tensor with the dtype, device and shape of points.")
            dirs = view_directions.detach().contiguous()
        pts = points.detach().contiguous()
        if not pts.is_cuda:
            i, nrm = estimate_point_cloud_normals_knn(pts.numpy(), num_neighbors, None if dirs is None else dirs.numpy(),
                                                      drop_angle_threshold, max_points_per_leaf, num_threads, device=device)
            return torch.from_numpy(i), torch.from_numpy(nrm)
        _same_device(pts, device)
        n = pts.shape[0]
        idx = torch.empty(n, dtype=torch.int64, device=pts.device)
        nrm = torch.empty((n, 3), dtype=pts.dtype, device=pts.device)
        count = torch.empty(1, dtype=torch.int64, device=pts.device)
        _pcu_internal._normals_knn_device(pts.dtype == torch.float64, pts.data_ptr(), n, 0 if dirs is None else dirs.data_ptr(),
                                          int(num_neighbors), float(drop_angle_threshold), idx.data_ptr(), nrm.data_ptr(),
                                          count.data_ptr(), int(max_points_per_leaf), pts.device.index or 0, _stream_of(pts))
        if dirs is None and n >= int(num_neighbors):
            return idx, nrm          # every point is kept: no need to wait for the count
        m = int(count.item())
        return idx[:m], nrm[:m]
    if type(points) != _np.ndarray:
        raise ValueError("Invalid type for points, must be a NumPy array, but got " + str(type(points)) + ".")
    if view_directions is None:
        view_directions = _np.zeros([0, 3], dtype=points.dtype)
    if type(view_directions) != _np.ndarray:
        raise ValueError("Invalid type for view_directions, must be None or a NumPy array, but got " +
                         str(type(view_directions)) + ".")
    if len(points.shape) != 2 or points.shape[-1] != 3:
        raise ValueError("Invalid shape for points, must be (n, 3) but got " + str(points.shape))
    if len(view_directions.shape) != 2:
        raise ValueError("Invalid shape for view_directions, must be (n, 3) but got " + str(view_directions.shape))
    return _pcu_internal.estimate_point_cloud_normals_knn_internal(points, view_directions, int(num_neighbors),
                                                                   int(max_points_per_leaf), float(drop_angle_threshold),
                                                                   int(num_threads), -1, _dev(device))


def estimate_point_cloud_normals_ball(points, ball_radius, view_directions=None, drop_angle_threshold=_np.deg2rad(90.0),
                                      min_pts_per_ball=3, max_pts_per_ball=-1, weight_function="constant",
                                      max_points_per_leaf=10, num_threads=-1, *, device=None):
    """
    Estimate normals for a point cloud by locally fitting a plane to all points within a radius of each point
    (possibly weighted by a radial basis function).

    Args:
        points: (n, 3)-shaped NumPy array (or CUDA tensor) of point positions (each row is a point)
        ball_radius: The radius of each neighborhood used to estimate normals.  As in the reference, this value is
                     handed to the radius search as it is, and that search compares SQUARED distances with it: the
                     neighbourhood of a point is every point whose squared distance is below ball_radius, while the
                     'rbf' weight is evaluated with the true distance d and r = ball_radius.
        view_directions: (n, 3)-shaped array or None, the unit direction to the sensor for each point; used to align
                         the normals and to drop points.
        drop_angle_threshold: If view_directions is passed in, drop points whose angle between the normal and view
                              direction exceeds drop_angle_threshold (in radians).
        min_pts_per_ball: Discard points whose neighborhood contains fewer than min_pts_per_ball points.
        max_pts_per_ball: If set to a positive number, then only use a random subset of max_pts_per_ball points of each
                          neighborhood whose number of points exceeds this value (the subset is drawn from NumPy's
                          global random state: seed it for reproducible results).
        weight_function: 'constant' (weight 1 for every point) or 'rbf' ((1 - d/r)^4 * (4 * d/r + 1)).
        max_points_per_leaf, num_threads: kd-tree leaf size / CPU threads of the reference; accepted and ignored.
        device : see `k_nearest_neighbors` (keyword only).

    Returns:
        idx : an (m,)-shaped int64 array of indices into points (the points that were kept, ascending)
        n : an (m, 3)-shaped array of unit normals for those points

    Mirrors /root/reference/point_cloud_utils/_pointcloud_normals.py:57-123 and
    /root/reference/src/point_cloud_normals.cpp:48-113, :303-370.  Neighbour sets (hence which points are kept by
    min_pts_per_ball) are the reference's; normals agree up to rounding and, without view directions, up to sign.
    """
    seed = int(_np.random.randint(2 ** 31 - 1))
    if _is_tensor(points):
        torch = _torch()
        if points.dtype not in (torch.float32, torch.float64):
            raise ValueError("Invalid scalar type (%s) for argument 'points'. Expected one of ['float32', 'float64']." % points.dtype)
        if points.dim() != 2 or points.shape[-1] != 3:
            raise ValueError("Invalid shape for points, must be (n, 3) but got " + str(tuple(points.shape)))
        if points.shape[0] == 0:
            raise ValueError("Invalid point set with zero elements: points must have shape (n, 3)")
        dirs = None
        if view_directions is not None:
            if not _is_tensor(view_directions) or view_directions.dtype != points.dtype or \
                    view_directions.device != points.device or tuple(view_directions.shape) != tuple(points.shape):
                raise ValueError("Invalid view directions does not match the number of points. If view directions are passed "
                                 "in, they must be a tensor with the dtype, device and shape of points.")
            dirs = view_directions.detach().contiguous()
        pts = points.detach().contiguous()
        if not pts.is_cuda:
            i, nrm = estimate_point_cloud_normals_ball(pts.numpy(), ball_radius, None if dirs is None else dirs.numpy(),
                                                       drop_angle_threshold, min_pts_per_ball, max_pts_per_ball, weight_function,
                                                       max_points_per_leaf, num_threads, device=device)
            return torch.from_numpy(i), torch.from_numpy(nrm)
        _same_device(pts, device)
        n = pts.shape[0]
        idx = torch.empty(n, dtype=torch.int64, device=pts.device)
        nrm = torch.empty((n, 3), dtype=pts.dtype, device=pts.device)
        count = torch.empty(1, dtype=torch.int64, device=pts.device)
        _pcu_internal._normals_ball_device(pts.dtype == torch.float64, pts.data_ptr(), n, 0 if dirs is None else dirs.data_ptr(),
                                           float(ball_radius), int(min_pts_per_ball), int(max_pts_per_ball),
                                           float(drop_angle_threshold), str(weight_function), seed, idx.data_ptr(), nrm.data_ptr(),
                                           count.data_ptr(), pts.device.index or 0, _stream_of(pts))
        m = int(count.item())
        return idx[:m], nrm[:m]
    if type(points) != _np.ndarray:
        raise ValueError("Invalid type for points, must be a NumPy array, but got " + str(type(points)) + ".")
    if view_directions is None:
        view_directions = _np.zeros([0, 3], dtype=points.dtype)
    if type(view_directions) != _np.ndarray:
        raise ValueError("Invalid type for view_directions, must be None or a NumPy array, but got " +
                         str(type(view_directions)) + ".")
    if len(points.shape) != 2 or points.shape[-1] != 3:
        raise ValueError("Invalid shape for points, must be (n, 3) but got " + str(points.shape))
    if len(view_directions.shape) != 2:
        raise ValueError("Invalid shape for view_directions, must be (n, 3) but got " + str(view_directions.shape))
    return _pcu_internal.estimate_point_cloud_normals_ball_internal(points, view_directions, float(ball_radius),
                                                                    int(min_pts_per_ball), int(max_pts_per_ball),
                                                                    float(drop_angle_threshold), int(max_points_per_leaf),
                                                                    int(num_threads), str(weight_function), seed, _dev(device))


# ---------------------------------------------------------------------------------------------
# 64-bit 3-D Morton codes: the reference's five bindings of /root/reference/src/morton.cpp, same names, arguments,
# dtypes and error conditions (numpy in, numpy out; integer work, bit-identical results)
def morton_encode(pts, num_threads=-1, *, device=None):
    """
    Encode n 3D points using Morton coding, possibly sorting them

    Args:
        pts : an (n, 3)-shaped int32 / int64 array of 3D points (coordinates in [-2^20, 2^20))
        num_threads : CPU thread count of the reference; accepted and ignored.

    Returns:
        codes : an (n,)-shaped uint64 array of Morton codes

    Mirrors /root/reference/src/morton.cpp:185-239 (MortonCode64, src/common/morton_code.cpp:43-63).
    """
    return _pcu_internal.morton_encode(_np.asarray(pts), int(num_threads), _dev(device))


def morton_decode(codes, num_threads=-1, *, device=None):
    """
    Decode n points along a Morton curve into 3D points

    Args:
        codes : an (n,)-shaped uint32 / uint64 array of Morton codes

    Returns:
        points : an (n, 3)-shaped int32 array of 3D points

    Mirrors /root/reference/src/morton.cpp:253-310.
    """
    return _pcu_internal.morton_decode(_np.asarray(codes), int(num_threads), _dev(device))


def morton_add(codes_1, codes_2, num_threads=-1, *, device=None):
    """Add morton codes together (corresponding to adding the vectors they encode): (n,), (n,) -> (n,) uint64.
    Mirrors /root/reference/src/morton.cpp:26-103."""
    return _pcu_internal.morton_add(_np.asarray(codes_1), _np.asarray(codes_2), int(num_threads), _dev(device))


def morton_subtract(codes_1, codes_2, num_threads=-1, *, device=None):
    """Subtract morton codes from each other (codes_1 - codes_2): (n,), (n,) -> (n,) uint64.
    Mirrors /root/reference/src/morton.cpp:106-183."""
    return _pcu_internal.morton_subtract(_np.asarray(codes_1), _np.asarray(codes_2), int(num_threads), _dev(device))


def morton_knn(codes, qcodes, k, sort_dist=True, *, device=None):
    """
    Queries a sorted array of morton encoded points to find the (approximate) k nearest neighbors

    Args:
        codes : an (n,)-shaped array of morton codes, sorted ascending
        qcodes : an (m,)-shaped array of query codes (same dtype)
        k : an integer representing the number of nearest neighbors
        sort_dist : (optional, defaults to True) whether to return the nearest neighbors in distance sorted order

    Returns:
        nn_idx : an (m, min(k, n))-shaped int64 array of indices into codes: the k consecutive positions around the
                 lower bound of each query code -- exactly the reference's window.  With sort_dist each row is ordered by
                 squared distance to the query point (ties by position); the reference's own order is undefined there
                 (its comparator reads uninitialised variables, /root/reference/src/morton.cpp:381-398).

    Mirrors /root/reference/src/morton.cpp:324-414.
    """
    return _pcu_internal.morton_knn(_np.asarray(codes), _np.asarray(qcodes), int(k), bool(sort_dist), _dev(device))


from ._sinkhorn import pairwise_distances, sinkhorn, earth_movers_distance  # noqa: E402  (N4: dense metrics)
from ._dedup import deduplicate_point_cloud, deduplicate_mesh_vertices  # noqa: E402  (N2: duplicate removal)


def _voxel_internal(points, attrib, voxel_size, min_bound, max_bound, min_points_per_voxel, device, return_counts=False):
    """downsample_point_cloud_voxel_grid_internal (/root/reference/src/sample_point_cloud.cpp:336-367) on the GPU:
    (mean points, mean attributes[, points per voxel]); numpy in -> numpy out, CUDA tensors in -> CUDA tensors out."""
    torch = _torch()
    is_np = isinstance(points, _np.ndarray)
    if is_np:
        if points.dtype not in (_np.float32, _np.float64):
            raise ValueError("Invalid scalar type (%s) for argument 'v'. Expected one of ['float32', 'float64']." % points.dtype)
        if attrib.dtype not in (_np.float32, _np.float64):
            raise ValueError("Invalid scalar type (%s) for argument 'attrib'. Expected one of ['float32', 'float64']." % attrib.dtype)
        dev = torch.device("cuda", _pcu_internal._current_device() if _dev(device) < 0 else _dev(device))
        pts = torch.from_numpy(_np.ascontiguousarray(points)).to(dev)
        att = torch.from_numpy(_np.ascontiguousarray(attrib)).to(dev) if attrib.size else None
    else:
        if points.dtype not in (torch.float32, torch.float64) or not points.is_cuda:
            raise ValueError("points must be a float32 / float64 numpy array or CUDA tensor")
        pts = points.detach().contiguous()
        att = attrib.detach().contiguous() if attrib is not None and attrib.numel() else None
        if att is not None and (att.dtype not in (torch.float32, torch.float64) or att.device != pts.device):
            raise ValueError("attributes must be float32 / float64 tensors on the device of points")
    if pts.dim() != 2 or pts.shape[1] != 3 or pts.shape[0] == 0:
        raise ValueError("points must have shape (n, 3) with n > 0, got " + str(tuple(pts.shape)))
    n = pts.shape[0]
    cols = 0
    if att is not None:
        if att.shape[0] != n:                                                                   # :184-189
            raise ValueError("Invalid number of attributes (%d). Must match number of input vertices (%d) or be 0." % (att.shape[0], n))
        att = att.reshape(n, -1)
        cols = att.shape[1]
    out_p = torch.empty((n, 3), dtype=pts.dtype, device=pts.device)
    out_a = torch.empty((n, cols), dtype=att.dtype, device=pts.device) if cols else None
    counts = torch.empty(n, dtype=torch.int32, device=pts.device) if return_counts else None
    rows = torch.empty(1, dtype=torch.int64, device=pts.device)
    _pcu_internal._voxel_downsample_device(pts.dtype == torch.float64, pts.data_ptr(), n, att.data_ptr() if cols else 0, cols,
                                           bool(cols and att.dtype == torch.float64), [float(v) for v in voxel_size],
                                           [float(v) for v in min_bound], [float(v) for v in max_bound], int(min_points_per_voxel),
                                           out_p.data_ptr(), out_a.data_ptr() if cols else 0, counts.data_ptr() if return_counts else 0,
                                           rows.data_ptr(), pts.device.index or 0, _stream_of(pts))
    m = int(rows.item())
    out_p = out_p[:m]
    out_a = out_a[:m] if cols else (torch.zeros((0, 0), dtype=pts.dtype, device=pts.device))
    if is_np:
        res = (out_p.cpu().numpy(), out_a.cpu().numpy().reshape((m,) + attrib.shape[1:]) if cols else _np.zeros([0, 0], dtype=attrib.dtype))
        return res + ((counts[:m].cpu().numpy(),) if return_counts else ())
    res = (out_p, out_a.reshape((m,) + tuple(attrib.shape[1:])) if cols else out_a)
    return res + ((counts[:m],) if return_counts else ())


def downsample_point_cloud_on_voxel_grid(voxel_size, points, *args, min_bound=None, max_bound=None, min_points_per_voxel=1,
                                         device=None):
    """
    Downsample a point set to conform with a voxel grid by taking the average of points within each voxel.

    Args:
        voxel_size : a scalar representing the size of each voxel or a 3 tuple representing the size per axis of each voxel.
        points: a [#v, 3]-shaped array of 3d points.
        *args: Any additional arguments of shape [#v, *] are treated as attributes and will averaged into each voxel along
               with the points
        min_bound: a 3 tuple representing the minimum coordinate of the voxel grid or None to use the bounding box of the
                input point cloud.
        max_bound: a 3 tuple representing the maximum coordinate of the voxel grid or None to use the bounding box of the
                input point cloud.
        min_points_per_voxel: If a voxel contains fewer than this many points, then don't include the points in that voxel
                            in the output.

    Returns:
        A tuple (v, attrib0, attrib1, ....) of downsampled points, and point attributes.
        Attributes are returned in the same order they are passed in.
        If no attributes are passed in, then this function simply returns vertices.

    Mirrors /root/reference/point_cloud_utils/__init__.py:123-200 and /root/reference/src/sample_point_cloud.cpp:163-244.
    Voxel membership, the set of output voxels and their sizes are the reference's exactly; rows come in the order of each
    voxel's first input point (the reference's order is that of a std::unordered_map walk, i.e. unspecified); means are
    accumulated in fp64 (the reference sums in the array's precision).
    """
    is_np = isinstance(points, _np.ndarray)
    if not is_np and not _is_tensor(points):
        raise ValueError("points must be a numpy array but got type " + str(type(points)))
    if _np.isscalar(voxel_size):
        voxel_size = _np.array([voxel_size] * 3)
    else:
        voxel_size = _np.array(voxel_size)
        if len(voxel_size) != 3:
            raise ValueError("Invalid voxel size must be a 3-tuple or a single float")
    attribs = []
    for i, arg in enumerate(args):
        if type(arg) != type(points):
            raise ValueError("Additional arguments after points and before keyword arguments must be numpy arrays")
        if arg.shape[0] != points.shape[0]:
            raise ValueError("Attribute " + str(i) + " must have same first dimension as number of points (" +
                             str(tuple(points.shape)) + " but got attrib.shape = " + str(tuple(arg.shape)))
        attribs.append(arg)
    if is_np:
        lo, hi = _np.min(points, axis=0), _np.max(points, axis=0)
    else:
        lo, hi = points.amin(dim=0).cpu().numpy(), points.amax(dim=0).cpu().numpy()
    if min_bound is None:
        min_bound = lo - voxel_size * 0.5
    if max_bound is None:
        max_bound = hi + voxel_size * 0.5
    min_bound, max_bound = _np.array(min_bound), _np.array(max_bound)
    if len(min_bound) != 3:
        raise ValueError("min_bound must be a 3 tuple")
    if len(max_bound) != 3:
        raise ValueError("max_bound must be a 3 tuple")
    if _np.any(max_bound - min_bound <= 0.0):
        raise ValueError("Invalid min_bound and max_bound. max_bound must be greater than min_bound in all dimensions")
    empty = _np.zeros([0, 0]) if is_np else None
    ret_v, ret_a0 = _voxel_internal(points, attribs[0] if attribs else empty, voxel_size, min_bound, max_bound,
                                    min_points_per_voxel, device)
    ret = [ret_v, ret_a0] if (attribs and ret_a0 is not None) else [ret_v]
    for i in range(1, len(attribs)):
        _, ret_ai = _voxel_internal(points, attribs[i], voxel_size, min_bound, max_bound, min_points_per_voxel, device)
        ret.append(ret_ai)
    return tuple(ret) if len(ret) > 1 else ret_v


def downsample_point_cloud_poisson_disk(v, radius, target_num_samples=-1, random_seed=0, sample_num_tolerance=0.04, *, device=None):
    """
    Downsample a point set so that samples are approximately evenly spaced.

    Args:
        v : an (n, 3)-shaped float32 / float64 array (or tensor) of points
        radius : desired separation between points (ignored when target_num_samples > 0)
        target_num_samples : if positive, search for the radius whose sample count lies within sample_num_tolerance of it
        random_seed : 32-bit seed of the sample priorities; 0 draws one from NumPy's global RNG (so np.random.seed makes
                      the call reproducible)
        sample_num_tolerance : relative tolerance of target_num_samples, in (0, 1]
        device : see `k_nearest_neighbors` (keyword only).

    Returns:
        p_idx : an (m,)-shaped int32 array of row indices into v, ASCENDING (numpy for numpy input, an int32 CUDA tensor
                on v's device for a CUDA tensor)

    Mirrors the reference's point_cloud_utils/__init__.py:4-5 and src/sample_point_cloud.cpp:240-333:
    name, arguments, defaults, argument errors and the target_num_samples search (run in v's precision).  The samples
    themselves are the greedy maximal independent set in the order of a seeded hash of the row: rows i and j conflict
    when their squared distance, rounded in v's precision like every distance of this library, is below radius * radius
    (also rounded in v's precision); visiting the rows by priority, a row is kept when it conflicts with no row kept
    before it.  No two samples conflict and every other row conflicts with a sample.  The reference's sampler (libigl's
    blue-noise loop) draws its priorities from rand() and returns the samples in placement order; neither is
    reproducible, so its exact output is not.
    """
    if target_num_samples <= 0 and radius <= 0.0:                               # :265-267
        raise ValueError("Cannot have both num_samples <= 0 and radius <= 0")
    tol = float(_np.float32(sample_num_tolerance))                               # the binding takes a float
    if tol > 1.0 or tol <= 0.0:                                                  # :268-270
        raise ValueError("sample_num_tolerance must be in (0, 1]")
    if not (0 <= int(random_seed) < 2 ** 32):
        raise ValueError("random_seed must fit in 32 unsigned bits (got %d)" % int(random_seed))
    if not (-2 ** 31 <= int(target_num_samples) < 2 ** 31):
        raise ValueError("target_num_samples must fit in a 32-bit int (got %d)" % int(target_num_samples))
    seed = int(random_seed) if int(random_seed) != 0 else int(_np.random.randint(1, 2 ** 32, dtype=_np.uint64))
    if _is_tensor(v):
        torch = _torch()
        if v.dtype not in (torch.float32, torch.float64):
            raise ValueError("Invalid scalar type (%s) for argument 'v'. Expected one of ['float32', 'float64']." % v.dtype)
        if v.dim() != 2 or v.shape[-1] != 3 or v.shape[0] == 0:
            raise ValueError("v must have shape (n, 3) with n > 0, got " + str(tuple(v.shape)))
        pts = v.detach().contiguous()
        if not pts.is_cuda:
            return torch.from_numpy(downsample_point_cloud_poisson_disk(pts.numpy(), radius, target_num_samples, seed,
                                                                        sample_num_tolerance, device=device))
        _same_device(pts, device)
        n = pts.shape[0]
        idx = torch.empty(n, dtype=torch.int32, device=pts.device)
        count = torch.empty(1, dtype=torch.int64, device=pts.device)
        _pcu_internal._poisson_device(pts.dtype == torch.float64, pts.data_ptr(), n, float(radius), int(target_num_samples), seed,
                                      tol, idx.data_ptr(), count.data_ptr(), pts.device.index or 0, _stream_of(pts))
        return idx[:int(count.item())]
    if type(v) != _np.ndarray:
        raise ValueError("Invalid type for v, must be a NumPy array, but got " + str(type(v)) + ".")
    return _pcu_internal.downsample_point_cloud_poisson_disk_internal(v, float(radius), int(target_num_samples), seed, tol,
                                                                      _dev(device))


def batched_chamfer_distance(x, y, max_points_per_leaf=10, *, device=None):
    """
    Chamfer distance of B independent pairs.

    Args:
        x : (B, n, 3) array / CUDA tensor, y : (B, m, 3) array / CUDA tensor (same dtype, float32).
    Returns:
        (B,) chamfer distances (numpy array for numpy inputs, CUDA tensor for CUDA tensors); entry b equals
        chamfer_distance(x[b], y[b]).

    The reference equivalent is a Python loop over `chamfer_distance` (its docstring's minibatch form,
    /root/reference/point_cloud_utils/__init__.py:89-90, was never implemented by the 2-D-only binding).
    """
    from ._batched import batched_chamfer  # noqa: WPS433 (kept separate: multi-GPU plumbing lives there too)
    return batched_chamfer(x, y, max_points_per_leaf, device=_dev(device))
