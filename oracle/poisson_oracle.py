"""TEST INFRASTRUCTURE: ctypes wrapper of oracle/poisson_oracle.c, the sequential plain-C statement of the
Poisson-disk down-sampling result of this library (see the header of that file for the rule it computes).

    build()                                               compiles oracle/libpcu_oracle_poisson.so when out of date
    downsample_point_cloud_poisson_disk(v, radius, ...)   -> int32 rows (ascending), like the library's function
    downsample_point_cloud_poisson_disk(..., return_trials=True) -> (rows, radii of the trials, sample counts)
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "poisson_oracle.c")
_LIB_PATH = os.path.join(_HERE, "libpcu_oracle_poisson.so")
_lib = None


def build():
    if os.path.exists(_LIB_PATH) and os.path.getmtime(_LIB_PATH) >= os.path.getmtime(_SRC):
        return _LIB_PATH
    # no FMA contraction: every operation of the distance is rounded on its own, as in the library
    subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-o", _LIB_PATH, _SRC, "-lm"],
                   check=True, capture_output=True)
    return _LIB_PATH


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        for suf, ct in (("f32", ctypes.c_float), ("f64", ctypes.c_double)):
            f = getattr(lib, "pcu_oracle_poisson_" + suf)
            f.restype = ctypes.c_longlong
            f.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_double, ctypes.c_int, ctypes.c_uint32, ctypes.c_float,
                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        _lib = lib
    return _lib


def downsample_point_cloud_poisson_disk(v, radius, target_num_samples=-1, random_seed=0, sample_num_tolerance=0.04,
                                        return_trials=False):
    """The library's result for a given (non-zero or zero) 32-bit seed, computed sequentially: `random_seed` is used
    as it is here (the library draws one from NumPy only when it is 0)."""
    v = np.ascontiguousarray(v)
    if v.dtype not in (np.float32, np.float64) or v.ndim != 2 or v.shape[1] != 3 or v.shape[0] == 0:
        raise ValueError("v must be a non-empty (n, 3) float32 / float64 array")
    lib = _load()
    n = v.shape[0]
    out = np.empty(n, dtype=np.int32)
    cap = 256
    radii = np.empty(cap, dtype=np.float64)
    counts = np.empty(cap, dtype=np.int64)
    trials = ctypes.c_int(0)
    fn = lib.pcu_oracle_poisson_f32 if v.dtype == np.float32 else lib.pcu_oracle_poisson_f64
    m = fn(v.ctypes.data, n, float(radius), int(target_num_samples), int(random_seed) & 0xffffffff, float(sample_num_tolerance),
           out.ctypes.data, radii.ctypes.data, counts.ctypes.data, cap, ctypes.byref(trials))
    if m == -1:
        raise ValueError("invalid arguments")
    if m < 0:
        raise MemoryError("poisson oracle out of memory")
    rows = out[:m].copy()
    if return_trials:
        t = min(trials.value, cap)
        return rows, radii[:t].copy(), counts[:t].copy()
    return rows
