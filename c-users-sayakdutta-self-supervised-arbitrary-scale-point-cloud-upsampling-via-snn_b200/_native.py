"""ctypes binding of libsapcu_b200.so (the C ABI declared in include/sapcu_b200.h).

The library is built in-tree with nvcc for sm_100a by :func:`build`; :func:`lib` loads it and fails loudly
when it is missing -- there is no Python / CPU fallback for any operator.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_SO = os.path.join(_HERE, "libsapcu_b200.so")
_SOURCES = ["api.cu", "model.cu", "forward.cu", "gemm.cu", "gemm_tc.cu", "gemm_tc2.cu", "knn_seed.cu", "patch_ops.cu",
            "intra_knn.cu", "fn_kernels.cu", "fd_kernels.cu", "seedgen.cu", "post_ops.cu", "lif_table.cu", "orient.cu",
            "mesh_dist.cu", "edge_pairs.cu", "emd.cu"]
# per-file flags: the fp64 geometry of seedgen.cu must round like the g++ build of dense.cpp (no FMA contraction), and that
# of mesh_dist.cu and emd.cu like their numpy restatements
_FILE_FLAGS = {"seedgen.cu": ["-fmad=false"], "mesh_dist.cu": ["-fmad=false"], "emd.cu": ["-fmad=false"]}
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

MODEL_FN, MODEL_FD = 0, 1
MODE_FP32, MODE_TC, MODE_TF32, MODE_FAST = 0, 1, 2, 3

_lock = threading.Lock()
_lib = None


class SapcuError(RuntimeError):
    pass


def _stale():
    if not os.path.exists(_SO):
        return True
    t = os.path.getmtime(_SO)
    for f in os.listdir(_CSRC):
        if os.path.getmtime(os.path.join(_CSRC, f)) > t:
            return True
    return os.path.getmtime(os.path.join(_HERE, "..", "include", "sapcu_b200.h")) > t


def build(force=False, verbose=False, extra_flags=(), out=None):
    """Compile csrc/*.cu into libsapcu_b200.so (sm_100a; cross-compiles without a GPU).
    `extra_flags` / `out` build an experimental variant next to the default library (see SAPCU_LIB)."""
    global _SO
    if out is not None:
        return _build_variant(list(extra_flags), out)
    if not force and not _stale():
        return _SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(_HERE, "build"), exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    for src in _SOURCES:
        obj = os.path.join(_HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + flags + _FILE_FLAGS.get(src, []) + ["-c", os.path.join(_CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise SapcuError("nvcc failed: %s\n%s" % (" ".join(cmd), out.decode(errors="replace")))
        if verbose and out:
            print(out.decode(errors="replace"))
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", _SO] + objs
    subprocess.check_call(cmd)
    return _SO


def _build_variant(extra, out):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    bdir = os.path.join(_HERE, "build", "variant_" + os.path.basename(out))
    os.makedirs(bdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + extra
    procs, objs = [], []
    for src in _SOURCES:
        obj = os.path.join(bdir, src.replace(".cu", ".o"))
        objs.append(obj)
        procs.append(subprocess.Popen([nvcc] + flags + _FILE_FLAGS.get(src, []) + ["-c", os.path.join(_CSRC, src), "-o", obj]))
    for p in procs:
        if p.wait() != 0:
            raise SapcuError("nvcc failed building variant %s" % out)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs)
    return out


class GemmCaseArgs(ctypes.Structure):
    """sapcu_gemm_case_args (include/sapcu_b200.h): one contraction of the forwards for sapcu_gemm_case."""
    _i, _i64, _f, _p = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p
    _fields_ = [("amode", _i), ("act", _i), ("T", _i), ("use_table", _i),
                ("R", _i64), ("K", _i), ("N", _i), ("lda", _i64), ("ldc", _i64), ("ldr", _i64),
                ("h_w", _p), ("h_bias", _p), ("h_scale", _p), ("h_shift", _p), ("h_params4", _p),
                ("d_x", _p), ("x_format", _i), ("x_unit", _i), ("fast", _i),
                ("d_y", _p), ("out_h2", _i), ("d_y2", _p),
                ("d_residual", _p),
                ("d_f", _p), ("ldf", _i64), ("C", _i),
                ("edge_bias", _i), ("d_q", _p), ("d_kf", _p), ("ldq", _i64), ("d_idx", _p), ("ldi", _i), ("kk", _i), ("mpts", _i),
                ("d_pool", _p), ("pool_T", _i), ("pool_M", _i),
                ("d_at_pos", _p), ("d_at_v", _p), ("at_ldv", _i64), ("at_sqrt", _f), ("d_at_pid", _p), ("pos_h2", _i),
                ("d_R_dev", _p), ("tc2_any_rows", _i), ("group", _i)]


_SIGS = {
    "sapcu_last_error": (ctypes.c_char_p, []),
    "sapcu_abi_version": (ctypes.c_int, []),
    "sapcu_launch_count": (ctypes.c_int64, []),
    "sapcu_device_status": (ctypes.c_int, []),
    "sapcu_profile": (ctypes.c_int, [ctypes.c_int]),
    "sapcu_profile_read": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                          ctypes.POINTER(ctypes.c_int64)]),
    "sapcu_profile_report": (ctypes.c_int64, [ctypes.c_char_p, ctypes.c_size_t]),
    "sapcu_knn_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64]),
    "sapcu_knn": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_knn_batched_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int]),
    "sapcu_knn_batched": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_gather_center_rotate": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                                  ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                  ctypes.c_void_p]),
    "sapcu_renormalize": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "sapcu_displace": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                      ctypes.c_void_p, ctypes.c_void_p]),
    "sapcu_seedgen_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_double, ctypes.c_int64]),
    "sapcu_seedgen": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.c_void_p,
                                     ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_outlier_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64]),
    "sapcu_outlier_mask": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int, ctypes.c_double,
                                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_knn_mean_dist": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                           ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "sapcu_outlier_mask_from_means": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                                     ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                                     ctypes.c_void_p]),
    "sapcu_fps": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
                                 ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_orient_normals_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int]),
    "sapcu_orient_normals": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_mesh_distance_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int64]),
    "sapcu_mesh_distance": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                           ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                           ctypes.c_void_p]),
    "sapcu_emd_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64]),
    "sapcu_emd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p,
                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "sapcu_model_create": (ctypes.c_void_p, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int]),
    "sapcu_model_set_tensor": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "sapcu_model_finalize": (ctypes.c_int, [ctypes.c_void_p]),
    "sapcu_model_destroy": (None, [ctypes.c_void_p]),
    "sapcu_model_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]),
    "sapcu_fn_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                        ctypes.c_void_p]),
    "sapcu_fn_indexed_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int64, ctypes.c_int]),
    "sapcu_pair_table_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64]),
    "sapcu_pair_table": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_size_t,
                                        ctypes.c_void_p, ctypes.c_void_p]),
    "sapcu_fn_forward_indexed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                                ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                                ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                                ctypes.c_void_p]),
    "sapcu_fd_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                        ctypes.c_int, ctypes.c_void_p]),
    "sapcu_model_tap": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                                       ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "sapcu_model_tap_format": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p]),
    "sapcu_lif_chain": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "sapcu_lif_table_selftest": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                                                ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint32)]),
    "sapcu_intra_knn": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "sapcu_gemm": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                  ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "sapcu_gemm_case_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(GemmCaseArgs)]),
    "sapcu_gemm_case": (ctypes.c_int, [ctypes.POINTER(GemmCaseArgs), ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                       ctypes.c_void_p]),
}

EXPORTS = tuple(_SIGS)


def lib():
    """The loaded shared library; raises SapcuError when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                so = os.environ.get("SAPCU_LIB", _SO)      # experiments: an alternative build of the same sources
                if not os.path.exists(so):
                    raise SapcuError(
                        "libsapcu_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`. "
                        "There is no CPU fallback for the sapcu_b200 hot path." % so)
                h = ctypes.CDLL(so)
                for name, (res, args) in _SIGS.items():
                    fn = getattr(h, name)   # AttributeError = the .so is missing a declared symbol
                    fn.restype = res
                    fn.argtypes = args
                _lib = h
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().sapcu_last_error()
        raise SapcuError("%s failed (%d): %s" % (what or "sapcu call", rc, msg.decode(errors="replace") if msg else ""))


def check_device(what="device"):
    """Raise if a tensor-core kernel's pipeline watchdog fired on the current device (call after a synchronise)."""
    check(lib().sapcu_device_status(), what + " status")


def ptr(t):
    """Device (or host) address of a torch tensor / None."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
