"""Poisson-disk down-sampling (downsample_point_cloud_poisson_disk): the sequential C oracle against an independent
brute-force check of the rule (CPU), the library against the oracle bit for bit (GPU)."""
import ctypes
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def poisson_oracle():
    from oracle import poisson_oracle as P
    P.build()
    return P


# ---- clouds ---------------------------------------------------------------------------------------------------
def uniform(n, seed=0):
    return np.random.default_rng(seed).random((n, 3))


def sphere(n, seed=1):
    p = np.random.default_rng(seed).normal(size=(n, 3))
    return p / np.linalg.norm(p, axis=1, keepdims=True)


def clustered(n, seed=2):
    rng = np.random.default_rng(seed)
    centres = rng.random((12, 3))
    return centres[rng.integers(0, 12, n)] + rng.normal(scale=0.02, size=(n, 3))


def duplicates(n, seed=3):
    rng = np.random.default_rng(seed)
    base = rng.random((n // 4, 3))
    return base[rng.integers(0, n // 4, n)]             # every point several times over


def planar(n, seed=4):
    rng = np.random.default_rng(seed)
    p = rng.random((n, 3))
    p[:, 2] = 0.25
    return p


CLOUDS = {"uniform": uniform, "sphere": sphere, "clustered": clustered, "duplicates": duplicates, "planar": planar}


# ---- the rule, checked without the oracle ------------------------------------------------------------------------
def d2_rounded(a, b):
    """((dx*dx) + dy*dy) + dz*dz, every operation in the arrays' precision: (len(a), len(b))."""
    dx, dy, dz = (a[:, None, k] - b[None, :, k] for k in range(3))
    return (dx * dx + dy * dy) + dz * dz


def r2_of(v, radius):
    t = v.dtype.type
    return t(radius) * t(radius)


def assert_separated_and_maximal(v, idx, radius, chunk=2048):
    r2 = r2_of(v, radius)
    s = v[idx]
    for i in range(0, len(s), chunk):                    # separation: no two samples conflict
        d = d2_rounded(s[i:i + chunk], s)
        d[np.arange(d.shape[0]), np.arange(i, i + d.shape[0])] = np.inf
        assert not (d < r2).any(), "two samples conflict"
    covered = np.zeros(len(v), dtype=bool)
    covered[idx] = True
    rest = np.flatnonzero(~covered)
    for i in range(0, len(rest), chunk):                 # maximality: every other row conflicts with a sample
        d = d2_rounded(v[rest[i:i + chunk]], s)
        assert (d < r2).any(axis=1).all(), "a row that conflicts with no sample was left out"


# ---- CPU: the oracle -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("name,radius", [("clustered", 0.01), ("duplicates", 0.05), ("planar", 0.04), ("uniform", 1e-5),
                                         ("sphere", 0.2)])
def test_oracle_separated_and_maximal(poisson_oracle, name, radius, dtype):
    v = CLOUDS[name](4000).astype(dtype)
    idx = poisson_oracle.downsample_point_cloud_poisson_disk(v, radius, random_seed=12345)
    assert idx.dtype == np.int32 and np.all(np.diff(idx) > 0)
    assert_separated_and_maximal(v, idx, radius)
    if name == "duplicates":
        assert len(idx) < len(np.unique(v, axis=0)) + 1   # copies of a point conflict (0 < r2)


def test_oracle_is_the_greedy_order(poisson_oracle):
    """The first key is always a sample, and a radius beyond the cloud keeps exactly that one row."""
    def h(i, seed):
        m = 0xffffffff
        def mix(x):
            x ^= x >> 16; x = (x * 0x7feb352d) & m; x ^= x >> 15; x = (x * 0x846ca68b) & m; x ^= x >> 16
            return x
        return mix(seed ^ mix((i * 0x9e3779b9 + 0x85ebca6b) & m))
    v = uniform(500)
    first = min(range(500), key=lambda i: (h(i, 99), i))
    assert list(poisson_oracle.downsample_point_cloud_poisson_disk(v, 1000.0, random_seed=99)) == [first]
    assert first in poisson_oracle.downsample_point_cloud_poisson_disk(v, 0.1, random_seed=99)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_oracle_target_search_follows_the_reference_loop(poisson_oracle, dtype):
    """The radii tried for target_num_samples are those of src/sample_point_cloud.cpp:285-326, recomputed here in the
    cloud's precision from the counts the oracle reports."""
    t = dtype
    v = clustered(3000).astype(dtype)
    target, tol = 200, np.float32(0.04)
    rows, radii, counts = poisson_oracle.downsample_point_cloud_poisson_disk(v, 0.0, target_num_samples=target,
                                                                            random_seed=5, sample_num_tolerance=tol,
                                                                            return_trials=True)
    ext = v.max(0) - v.min(0)
    bbsize = np.sqrt(t(t(ext[0] * ext[0] + ext[1] * ext[1]) + ext[2] * ext[2]))
    rmin = rmax = t(float(bbsize) / 50.0)
    expect, k = [], 0
    while True:                                           # halving
        rmin = t(float(rmin) / 2.0); expect.append(rmin); k += 1
        if counts[k - 1] >= target:
            break
    while True:                                           # doubling
        rmax = t(float(rmax) * 2.0); expect.append(rmax); k += 1
        if counts[k - 1] <= target:
            break
    nmin = int(t(target) * t(np.float32(1.0) - tol))
    nmax = int(t(target) * t(np.float32(1.0) + tol))
    it = 0
    while it < 20 and (counts[k - 1] < nmin or counts[k - 1] > nmax):
        it += 1
        cur = t(float(t(rmin + rmax)) / 2.0); expect.append(cur); k += 1
        if counts[k - 1] > target:
            rmin = cur
        if counts[k - 1] < target:
            rmax = cur
    assert k == len(radii) and np.array_equal(np.array(expect, dtype=np.float64), radii)
    assert len(rows) == counts[-1]
    assert np.array_equal(rows, poisson_oracle.downsample_point_cloud_poisson_disk(v, float(radii[-1]), random_seed=5))


@pytest.mark.parametrize("kwargs", [dict(radius=0.0), dict(radius=-1.0, target_num_samples=0),
                                    dict(radius=0.1, sample_num_tolerance=0.0), dict(radius=0.1, sample_num_tolerance=1.5),
                                    dict(radius=0.1, random_seed=2 ** 32), dict(radius=0.1, random_seed=-1)])
def test_argument_errors_raise_before_any_device_work(pcu, kwargs):
    """The checks of the binding (:265-270) and the seed range raise ValueError in Python, without a GPU."""
    with pytest.raises(ValueError):
        pcu.downsample_point_cloud_poisson_disk(uniform(10).astype(np.float32), **kwargs)


# ---- GPU: the library ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("name,n,radii", [("uniform", 200000, (0.004, 0.02)), ("sphere", 100000, (0.01, 0.05)),
                                          ("clustered", 50000, (0.002, 0.01)), ("duplicates", 40000, (0.01,)),
                                          ("planar", 60000, (0.003, 0.02))])
def test_gpu_matches_oracle(pcu, poisson_oracle, name, n, radii, dtype):
    v = CLOUDS[name](n).astype(dtype)
    for r in radii:
        for seed in (1234567, 7654321):
            got = pcu.downsample_point_cloud_poisson_disk(v, r, random_seed=seed)
            ref = poisson_oracle.downsample_point_cloud_poisson_disk(v, r, random_seed=seed)
            assert got.dtype == np.int32
            assert np.array_equal(got, ref), (name, r, seed, len(got), len(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("name,target", [("sphere", 1000), ("uniform", 5000), ("clustered", 300)])
def test_gpu_target_num_samples_matches_oracle(pcu, poisson_oracle, name, target, dtype):
    v = CLOUDS[name](30000).astype(dtype)
    got = pcu.downsample_point_cloud_poisson_disk(v, 0.0, target_num_samples=target, random_seed=42)
    ref = poisson_oracle.downsample_point_cloud_poisson_disk(v, 0.0, target_num_samples=target, random_seed=42)
    assert np.array_equal(got, ref)
    if name != "clustered":                               # smooth data: the search lands inside the window
        assert int(target * np.float32(0.96)) <= len(got) <= int(target * np.float32(1.04)), len(got)


@pytest.mark.gpu
def test_gpu_reference_examples(pcu):
    """tests/test_examples.py:30-53 of the reference, on a dense sphere."""
    v = sphere(40000).astype(np.float32)
    bbox_diag = float(np.linalg.norm(v.max(0) - v.min(0)))
    a = pcu.downsample_point_cloud_poisson_disk(v, 0.1 * bbox_diag, random_seed=1234567)
    b = pcu.downsample_point_cloud_poisson_disk(v, 0.1 * bbox_diag, random_seed=1234567)
    c = pcu.downsample_point_cloud_poisson_disk(v, 0.1 * bbox_diag, random_seed=7654321)
    assert np.array_equal(a, b)
    assert a.shape != c.shape or not np.array_equal(a, c)
    one = pcu.downsample_point_cloud_poisson_disk(v, 2 * v.shape[0], random_seed=1234567)
    assert one.shape == (1,)
    a = pcu.downsample_point_cloud_poisson_disk(v, 0., target_num_samples=1000, random_seed=1234567)
    b = pcu.downsample_point_cloud_poisson_disk(v, 0., target_num_samples=1000, random_seed=1234567)
    c = pcu.downsample_point_cloud_poisson_disk(v, 0., target_num_samples=1000, random_seed=7654321)
    assert np.array_equal(a, b)
    assert a.shape != c.shape or not np.array_equal(a, c)
    everything = pcu.downsample_point_cloud_poisson_disk(v[:500], 0., target_num_samples=500)
    assert everything.dtype == np.int32 and np.array_equal(everything, np.arange(500, dtype=np.int32))


@pytest.mark.gpu
def test_gpu_seed_zero_follows_numpy(pcu):
    v = uniform(20000).astype(np.float32)
    np.random.seed(3)
    a = pcu.downsample_point_cloud_poisson_disk(v, 0.03)
    np.random.seed(3)
    b = pcu.downsample_point_cloud_poisson_disk(v, 0.03)
    assert np.array_equal(a, b)


@pytest.mark.gpu
def test_gpu_tensor_input(pcu):
    import torch
    v = sphere(30000)
    for dtype in (np.float32, np.float64):
        x = v.astype(dtype)
        ref = pcu.downsample_point_cloud_poisson_disk(x, 0.03, random_seed=11)
        t = torch.from_numpy(x).cuda()
        got = pcu.downsample_point_cloud_poisson_disk(t, 0.03, random_seed=11)
        assert got.is_cuda and got.dtype == torch.int32 and got.device == t.device
        assert np.array_equal(got.cpu().numpy(), ref)
        got = pcu.downsample_point_cloud_poisson_disk(t, 0., target_num_samples=800, random_seed=11, device=t.device)
        assert np.array_equal(got.cpu().numpy(), pcu.downsample_point_cloud_poisson_disk(x, 0., target_num_samples=800, random_seed=11))
        cpu = pcu.downsample_point_cloud_poisson_disk(torch.from_numpy(x), 0.03, random_seed=11)
        assert not cpu.is_cuda and np.array_equal(cpu.numpy(), ref)
    last = pcu.device_count() - 1
    got = pcu.downsample_point_cloud_poisson_disk(v.astype(np.float32), 0.03, random_seed=11, device=last)
    assert np.array_equal(got, pcu.downsample_point_cloud_poisson_disk(v.astype(np.float32), 0.03, random_seed=11))
    with pytest.raises(ValueError):
        pcu.downsample_point_cloud_poisson_disk(torch.from_numpy(v).cuda(), 0.03, device=pcu.device_count())


@pytest.mark.gpu
def test_gpu_full_size_thousand_points_per_ball(pcu, poisson_oracle):
    """10^6 uniform points, a radius holding about 10^3 of them: equal to the oracle, and separated and maximal by an
    independent brute-force pass."""
    v = uniform(10 ** 6, seed=8).astype(np.float32)
    radius = float((1000 / (10 ** 6 * 4 / 3 * np.pi)) ** (1 / 3))
    got = pcu.downsample_point_cloud_poisson_disk(v, radius, random_seed=2024)
    ref = poisson_oracle.downsample_point_cloud_poisson_disk(v, radius, random_seed=2024)
    assert np.array_equal(got, ref)
    import torch
    vt = torch.from_numpy(v).cuda()
    st = torch.from_numpy(v[got]).cuda()
    r2 = np.float32(radius) * np.float32(radius)

    def d2(a, b):
        dx, dy, dz = (a[:, None, k] - b[None, :, k] for k in range(3))
        return (dx * dx + dy * dy) + dz * dz
    for i in range(0, st.shape[0], 4096):                 # torch on the GPU, elementwise in fp32 (no fused reduction)
        d = d2(st[i:i + 4096], st)
        d[torch.arange(d.shape[0]), torch.arange(i, i + d.shape[0])] = float("inf")
        assert not bool((d < float(r2)).any())
    covered = torch.zeros(v.shape[0], dtype=torch.bool, device="cuda")
    for i in range(0, v.shape[0], 8192):
        covered[i:i + 8192] = (d2(vt[i:i + 8192], st) < float(r2)).any(1)
    assert bool(covered.all())                           # samples cover themselves (d2 = 0 < r2)


@pytest.mark.gpu
def test_ctypes_host_entry_points(pcu, poisson_oracle):
    """pcu_b200_poisson_disk_downsample_host_* (numpy memory in and out)."""
    lib = ctypes.CDLL(os.path.join(ROOT, "point-cloud-utils_b200", "libpcu_b200.so"))
    ws = ctypes.c_void_p()
    assert lib.pcu_b200_workspace_create(ctypes.c_int(0), ctypes.byref(ws)) == 0
    try:
        for dtype, fn in ((np.float32, lib.pcu_b200_poisson_disk_downsample_host_f32),
                          (np.float64, lib.pcu_b200_poisson_disk_downsample_host_f64)):
            v = np.ascontiguousarray(clustered(30000).astype(dtype))
            out = np.empty(len(v), dtype=np.int32)
            count = ctypes.c_int64(0)
            fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_int, ctypes.c_uint32,
                           ctypes.c_float, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]
            assert fn(ws, v.ctypes.data, len(v), 0.01, -1, 77, 0.04, out.ctypes.data, ctypes.byref(count)) == 0
            ref = poisson_oracle.downsample_point_cloud_poisson_disk(v, 0.01, random_seed=77)
            assert np.array_equal(out[:count.value], ref)
            assert fn(ws, v.ctypes.data, len(v), 0.0, -1, 77, 0.04, out.ctypes.data, ctypes.byref(count)) == 1   # invalid argument
    finally:
        lib.pcu_b200_workspace_destroy(ws)
