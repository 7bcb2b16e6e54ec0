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


def displace(seeds, normals, dist):
    seeds = np.ascontiguousarray(seeds, np.float64)
    normals = np.ascontiguousarray(normals, np.float32)
    dist = np.ascontiguousarray(dist, np.float32)
    out = np.empty_like(seeds)
    lib().oracle_displace(_p(seeds), _p(normals), _p(dist), ctypes.c_int64(seeds.shape[0]), _p(out))
    return out
