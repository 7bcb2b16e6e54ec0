"""ORACLE -- TEST INFRASTRUCTURE ONLY.  ctypes view of oracle/_build/liboracle_c.so (built by `make -C oracle`)."""
import ctypes
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_DIR, "_build", "liboracle_c.so")
_lib = None


def build():
    subprocess.check_call(["make", "-C", _DIR, "-s"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = ctypes.CDLL(_SO)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def knn(cloud, seeds, k):
    cloud = np.ascontiguousarray(cloud, np.float64)
    seeds = np.ascontiguousarray(seeds, np.float64)
    idx = np.empty((seeds.shape[0], k), np.int32)
    lib().oracle_knn_f64(_p(cloud), ctypes.c_int64(cloud.shape[0]), _p(seeds), ctypes.c_int64(seeds.shape[0]),
                         ctypes.c_int(k), _p(idx))
    return idx


def fps(xyz, npoint, start=None):
    """farthest_point_sample in fp32 (sapcu_oracle.fps restated in C, any start; default N // 2) -> int64 [npoint]"""
    xyz = np.ascontiguousarray(xyz, np.float32)
    n = xyz.shape[0]
    out = np.empty(npoint, np.int64)
    lib().oracle_fps_f32(_p(xyz), ctypes.c_int64(n), ctypes.c_int64(npoint), ctypes.c_int64(n // 2 if start is None else start),
                         _p(out))
    return out


def neuron_chain(x, prm4, T, eif2=None):
    x = np.ascontiguousarray(x, np.float32)
    prm4 = np.ascontiguousarray(prm4, np.float32)
    rows, C = x.shape
    out = np.empty((T, rows, C), np.float32)
    e = None if eif2 is None else np.ascontiguousarray(eif2, np.float32)
    lib().oracle_neuron_chain(_p(x), ctypes.c_int64(rows), ctypes.c_int(C), ctypes.c_int(T), _p(prm4),
                              None if e is None else _p(e), _p(out))
    return out


def rotation_to_x(n):
    n = np.ascontiguousarray(n, np.float32)
    R = np.empty((3, 3), np.float64)
    lib().oracle_rotation_to_x(_p(n), _p(R))
    return R


def gather_center_rotate(cloud, seeds, idx, normals=None):
    cloud = np.ascontiguousarray(cloud, np.float64)
    seeds = np.ascontiguousarray(seeds, np.float64)
    idx = np.ascontiguousarray(idx, np.int32)
    s, k = idx.shape
    out = np.empty((s, k, 3), np.float32)
    nrm = None if normals is None else np.ascontiguousarray(normals, np.float32)
    lib().oracle_gather_center_rotate(_p(cloud), _p(seeds), _p(idx), ctypes.c_int64(s), ctypes.c_int(k),
                                      None if nrm is None else _p(nrm), _p(out))
    return out


def round6_text(v):
    """fprintf("%lf") read back with strtod, elementwise"""
    v = np.ascontiguousarray(v, np.float64)
    out = np.empty_like(v)
    lib().oracle_round6_text(_p(v), ctypes.c_int64(v.size), _p(out))
    return out


def seedgen(cloud, cell, quirk_origin=True, round6=True, cap=None, max_levels=4096):
    """The seed generator as a serial FIFO flood fill -> (seeds [min(count, cap), 3] f64, count, level_stats [levels, 2]).
    An explicit `cap` keeps only the first `cap` seeds (count stays the total); by default all are returned.
    level_stats[L] = (queue entries of BFS level L, 6 * voxels of level L that expand)."""
    cloud = np.ascontiguousarray(cloud, np.float64)
    n = cloud.shape[0]
    grow, cap = cap is None, (1 << 22 if cap is None else cap)
    while True:
        out = np.empty((cap, 3), np.float64)
        stats = np.zeros((max_levels, 2), np.int64)
        count = ctypes.c_int64(0)
        f = lib().oracle_seedgen
        f.restype = ctypes.c_int64
        levels = f(_p(cloud), ctypes.c_int64(n), ctypes.c_double(cell), ctypes.c_int(int(quirk_origin)),
                   ctypes.c_int(int(round6)), _p(out), ctypes.c_int64(cap), ctypes.byref(count), _p(stats),
                   ctypes.c_int64(max_levels))
        if levels < 0:
            raise MemoryError("oracle_seedgen")
        assert levels <= max_levels
        if count.value <= cap or not grow:
            return out[:min(count.value, cap)], count.value, stats[:levels]
        cap = count.value


def displace(seeds, normals, dist):
    seeds = np.ascontiguousarray(seeds, np.float64)
    normals = np.ascontiguousarray(normals, np.float32)
    dist = np.ascontiguousarray(dist, np.float32)
    out = np.empty_like(seeds)
    lib().oracle_displace(_p(seeds), _p(normals), _p(dist), ctypes.c_int64(seeds.shape[0]), _p(out))
    return out
