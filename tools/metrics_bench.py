#!/usr/bin/env python
"""Time the evaluation metrics on the GPU: the exact point-to-mesh distance (sapcu_mesh_distance, LBVH built and queried on
the device) and Chamfer / Hausdorff (sapcu_knn with K = 1, both directions), next to the numpy brute force on the host.

    python tools/metrics_bench.py [--levels 5 7 9] [--queries 8192 388467 2000000] [--reps 5] [--warmup 2] [--out FILE]

Meshes: synthetic.sphere_mesh(level), 20 * 4**level faces (level 5: 20,480; 7: 327,680; 9: 5,242,880).  Queries: points
uniformly within 0.01 of that sphere (radius 0.49 .. 0.51), seeded.  8,192 is one PU-style test shape, 388,467 the output
of configuration 1's pipeline, 2,000,000 a scan-sized cloud.  Per (mesh, queries) case, one JSON object:
  call_ms      the whole sapcu_mesh_distance call (build + query), CUDA events, median after warm-up
  build_ms     the same call with ONE query point: the LBVH build plus a single-thread query
  query_ms     call_ms - build_ms
  morton_*     the same call with the points in generation.morton_order (the permutation's own time reported apart)
  work         nodes whose box bound was computed and point-triangle tests per query point, counted by a build of
               mesh_dist.cu with -DSAPCU_MESH_COUNTERS (a separate library; its times are not used)
  host         the numpy brute force (the restatement of tests/test_metrics.py) on the first `host_points` query points,
               wall time on the host cores, and whether the GPU's distances and faces equal it bitwise on that subsample
CD/HD cases: 8,192 x 8,192 and 388,467 x 8,192 points (pred x gt), both directions, CUDA events.
A 256 MiB buffer is overwritten before every timed run, so no run starts from an L2 (126 MB) left warm by the last one.
The GPU's name, power limit and SM clock are read with nvidia-smi (read-only queries) in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    return {"query": q, "row": out.stdout.strip(), "rc": out.returncode}


def shell(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.normal(size=(n, 3))
    return p * (0.49 + 0.02 * rng.random((n, 1))) / np.linalg.norm(p, axis=1, keepdims=True)


def counters_library(N):
    """libsapcu_b200 with an instrumented mesh_dist.cu, linked in a temporary directory from the package's build objects."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tmp = tempfile.mkdtemp(prefix="sapcu_mesh_counters_")
    obj = os.path.join(tmp, "mesh_dist.o")
    flags = [f for f in N.NVCC_FLAGS if f != "-shared"] + N._FILE_FLAGS["mesh_dist.cu"] + ["-DSAPCU_MESH_COUNTERS"]
    subprocess.check_call([nvcc] + flags + ["-c", os.path.join(N._CSRC, "mesh_dist.cu"), "-o", obj])
    objs = [os.path.join(N._HERE, "build", s.replace(".cu", ".o")) for s in N._SOURCES if s != "mesh_dist.cu"] + [obj]
    so = os.path.join(tmp, "libsapcu_mesh_counters.so")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so] + objs)
    h = ctypes.CDLL(so)
    h.sapcu_mesh_distance.restype = ctypes.c_int
    h.sapcu_mesh_distance.argtypes = N._SIGS["sapcu_mesh_distance"][1]
    h.sapcu_mesh_counters.restype = ctypes.c_int
    h.sapcu_mesh_counters.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--levels", type=int, nargs="+", default=[5, 7, 9])
    ap.add_argument("--queries", type=int, nargs="+", default=[8192, 388467, 2000000])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-points", type=int, default=256, help="host brute force subsample (points) per mesh, fewer on meshes above 2^18 faces")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("metrics_bench needs a CUDA device")
    import sapcu_b200.synthetic as syn
    from sapcu_b200 import _native as N
    from sapcu_b200 import metrics as M
    from sapcu_b200.generation import morton_order
    from test_metrics import mesh_distance_ref

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    L = N.lib()
    st = torch.cuda.current_stream(dev)
    sp = N.stream_ptr(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    C = counters_library(N)
    res = {"gpu": gpu_info(), "cases": [], "chamfer": []}

    def timed(fn):
        for _ in range(a.warmup):
            fn()
        ms = []
        for _ in range(a.reps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            fn()
            e1.record(st)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        N.check_device("metrics_bench")
        return sorted(ms)[len(ms) // 2]

    for level in a.levels:
        v, f = syn.sphere_mesh(level)
        V, F = len(v), len(f)
        d_v, d_f = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
        ws = torch.empty(L.sapcu_mesh_distance_workspace_bytes(V, F), dtype=torch.uint8, device=dev)

        def call(lib, d_p, d2, face):
            N.check(lib.sapcu_mesh_distance(N.ptr(d_v), V, N.ptr(d_f), F, N.ptr(d_p), d_p.shape[0], N.ptr(d2), N.ptr(face),
                                            N.ptr(ws), ws.numel(), sp), "sapcu_mesh_distance")

        one = torch.from_numpy(shell(1, 99)).to(dev)
        o2, of = torch.empty(1, dtype=torch.float64, device=dev), torch.empty(1, dtype=torch.int32, device=dev)
        build_ms = timed(lambda: call(L, one, o2, of))
        for S in a.queries:
            p = shell(S, 1000 + S)
            d_p = torch.from_numpy(p).to(dev)
            d2 = torch.empty(S, dtype=torch.float64, device=dev)
            face = torch.empty(S, dtype=torch.int32, device=dev)
            call_ms = timed(lambda: call(L, d_p, d2, face))
            perm_ms = timed(lambda: morton_order(d_p))
            perm = morton_order(d_p)
            d_pm = d_p[perm].contiguous()
            morton_ms = timed(lambda: call(L, d_pm, d2, face))
            call(L, d_p, d2, face)
            torch.cuda.synchronize()
            g2, gf = d2.cpu().numpy(), face.cpu().numpy()
            C.sapcu_mesh_counters(None, 1)
            cd2, cf = torch.empty_like(d2), torch.empty_like(face)
            call(C, d_p, cd2, cf)
            torch.cuda.synchronize()
            cnt = (ctypes.c_ulonglong * 2)()
            N.check(C.sapcu_mesh_counters(cnt, 0), "sapcu_mesh_counters")
            case = {"level": level, "faces": F, "vertices": V, "queries": S, "workspace_bytes": ws.numel(),
                    "call_ms": call_ms, "build_ms": build_ms, "query_ms": call_ms - build_ms,
                    "morton_call_ms": morton_ms, "morton_order_ms": perm_ms,
                    "work": {"nodes_per_query": cnt[0] / S, "tri_tests_per_query": cnt[1] / S,
                             "tri_tests_share_of_brute_force": cnt[1] / (S * F),
                             "counted_equal_results": bool(torch.equal(cd2, d2) and torch.equal(cf, face))}}
            if S == a.queries[0]:
                h = min(max(16, min(a.host_points, (1 << 26) // F)), S)     # at most ~2^26 point-triangle pairs
                t0 = time.perf_counter()
                r2, rf = mesh_distance_ref(v, f, p[:h])
                host_s = time.perf_counter() - t0
                case["host"] = {"points": h, "seconds": host_s, "cores": os.cpu_count(),
                                "identical": bool(np.array_equal(r2.view(np.uint64), g2[:h].view(np.uint64))
                                                  and np.array_equal(rf, gf[:h]))}
            res["cases"].append(case)
            print(json.dumps(case), flush=True)
            del d_p, d2, face, d_pm, cd2, cf
        del d_v, d_f, ws
        torch.cuda.empty_cache()

    for sp_n, sg_n in ((8192, 8192), (388467, 8192)):
        pred = torch.from_numpy(shell(sp_n, 7)).to(dev)
        gt = torch.from_numpy(shell(sg_n, 8)).to(dev)
        ms = timed(lambda: (M._nn_dist2(pred, gt), M._nn_dist2(gt, pred)))
        r = {"pred": sp_n, "gt": sg_n, "both_directions_ms": ms}
        res["chamfer"].append(r)
        print(json.dumps(r), flush=True)

    res["gpu_end"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
