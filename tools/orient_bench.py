#!/usr/bin/env python
"""Time the orientation of the upsampler's normals on the GPU, next to the host restatement of the same contract.

    python tools/orient_bench.py [--k 10] [--reps 20] [--warmup 3] [--out FILE]

Input: the displaced points and fn normals of configuration 1's cloud (2,048-point sphere) at the default spacing 0.004,
388,467 seeds from sapcu_seedgen through the fast-mode pipeline with bench.py's random-init models.  Prints one JSON line:
  gpu        name and power limit (nvidia-smi --query-gpu, read-only), SM clock at the end
  knn_ms     the self-kNN (sapcu_knn, cloud = queries = points, K = k + 1), CUDA events, after warm-up
  orient_ms  sapcu_orient_normals on that graph, CUDA events, after warm-up, the raw normals copied back before each run
  call_ms    generation.orient_normals end to end (allocations, kNN, orientation), host clock ending in a synchronise
  host_s     scipy cKDTree query (k + 1) and the test suite's restatement (tests/test_oriented_normals.py), one run each
  identical  the GPU normals and roots equal the restatement's on the GPU's graph
A 256 MiB buffer is overwritten before every timed run, so no pass starts from an L2 (126 MB) left warm by the last one.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (configuration 1's models)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    return {"query": q, "row": out.stdout.strip(), "rc": out.returncode}


def stats(ms):
    ms = sorted(ms)
    return {"median": ms[len(ms) // 2], "min": ms[0], "max": ms[-1], "runs": len(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("orient_bench needs a CUDA device")
    import sapcu_b200.synthetic as syn
    from sapcu_b200 import _native as N
    from sapcu_b200.generation import Generator3D6, orient_normals
    from scipy.spatial import cKDTree
    from test_oriented_normals import orient_reference

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    L = N.lib()
    mfn, mfd, _, _ = bench.build_models(dev)
    mfn.set_mode("fast"), mfd.set_mode("fast")
    gen = Generator3D6(mfn, mfd, dev, k_neighbors=100, dense_spacing=0.004, remove_outliers=False)
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = gen.gpu_seeds(cloud)
    pts, _, raw, _ = gen.displace_device(torch.from_numpy(cloud).to(dev), torch.from_numpy(seeds).to(dev), return_parts=True)
    S, K = pts.shape[0], min(a.k + 1, pts.shape[0])

    st = torch.cuda.current_stream(dev)
    sp = N.stream_ptr(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    idx = torch.empty(S, K, dtype=torch.int32, device=dev)
    kws = torch.empty(L.sapcu_knn_workspace_bytes(S), dtype=torch.uint8, device=dev)
    ows = torch.empty(L.sapcu_orient_normals_workspace_bytes(S, K), dtype=torch.uint8, device=dev)
    work = torch.empty_like(raw)
    root = torch.empty(S, dtype=torch.int32, device=dev)

    def knn():
        N.check(L.sapcu_knn(N.ptr(pts), S, N.ptr(pts), S, K, N.ptr(idx), N.ptr(kws), kws.numel(), sp), "sapcu_knn")

    def orient():
        N.check(L.sapcu_orient_normals(N.ptr(pts), S, N.ptr(idx), K, N.ptr(work), N.ptr(root), N.ptr(ows), ows.numel(), sp),
                "sapcu_orient_normals")

    def timed(fn, before=None):
        ms = []
        for r in range(a.warmup + a.reps):
            if before is not None:
                before()
            flush.fill_(r & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            fn()
            e1.record(st)
            e1.synchronize()
            if r >= a.warmup:
                ms.append(e0.elapsed_time(e1))
        return ms

    knn_ms = timed(knn)
    orient_ms = timed(orient, before=lambda: work.copy_(raw))
    call_ms = []
    for r in range(a.warmup + a.reps):
        flush.fill_(r & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = orient_normals(pts, raw, a.k)
        torch.cuda.synchronize()
        if r >= a.warmup:
            call_ms.append((time.perf_counter() - t0) * 1e3)
    N.check_device("orient_bench")

    h_pts, h_raw, h_idx = pts.cpu().numpy(), raw.cpu().numpy(), idx.cpu().numpy()
    t0 = time.perf_counter()
    cKDTree(h_pts).query(h_pts, K)
    t_kd = time.perf_counter() - t0
    t0 = time.perf_counter()
    ref, ref_root = orient_reference(h_pts, h_idx, h_raw)
    t_ref = time.perf_counter() - t0
    got = work.cpu().numpy()
    identical = bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)) and np.array_equal(root.cpu().numpy(), ref_root)
                     and np.array_equal(res.cpu().numpy().view(np.uint32), ref.view(np.uint32)))
    rec = {"tool": "orient_bench", "gpu": gpu_info(), "points": S, "k": a.k, "graph_K": K,
           "components": int(np.unique(ref_root).size), "knn_ms": stats(knn_ms), "orient_ms": stats(orient_ms),
           "call_ms": stats(call_ms), "host_s": {"ckdtree_query": t_kd, "restatement": t_ref, "cpus": os.cpu_count()},
           "identical": identical, "l2": "256 MiB buffer overwritten before every timed run"}
    line = json.dumps(rec)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not identical:
        sys.exit("GPU orientation differs from the restatement")


if __name__ == "__main__":
    main()
