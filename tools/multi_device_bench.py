#!/usr/bin/env python
"""Single-process multi-GPU throughput of Generator3D6 over a device list, next to bench.py's torch.distributed figures.

    python tools/multi_device_bench.py [--devices 1,2,4,8] [--modes tc,fast] [--steps 5] [--warmup 2] [--bench-steps 5]

Prints one JSON line per record:
  gpu          name, power limit and SM clocks of every visible GPU (nvidia-smi --query-gpu, read-only)
  finalize     one-time handle build per device (create + set_tensor + finalize, incl. the LIF tables), fn and fd
  throughput   Generator3D6(mfn, mfd, ["cuda:0", ..., "cuda:N-1"]).displace_host on the configs[1] cloud (2,048-pt sphere,
               K = 100): weak scaling (8,192 seeds per device, bench.py --config 1's workload) and strong scaling (65,536 seeds
               in total); host arrays in and out, host clock around the call (which ends in a stream synchronise on every
               device), a 256 MiB buffer per device overwritten between steps (> 126 MB L2).  `identical`: the N-device points
               equal the 1-device pipeline run shard by shard (strong scaling).
  bench        after each weak-scaling measurement: bench.py --gpus N --config 1 --mode M (torchrun for N > 1), its `value`
               (device-timed) and `e2e` (host arrays in and out) -- the same session, alternating with the line above
  upsample     one multi-device upsample() of the configs[1] cloud at the default spacing (0.004), split into seed generation,
               the sharded displacement and the outlier filter (the first and the last run on the primary device)
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the workload and model definitions bench.py times)


def emit(rec):
    print(json.dumps(rec), flush=True)


def gpu_info():
    q = "index,name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    return {"query": q, "rows": [r.strip() for r in out.stdout.strip().splitlines()], "rc": out.returncode}


def finalize_times(ndev):
    """Handle build per device on fresh modules (nothing cached): host copy of the state_dict, BN folding, LIF tables, upload."""
    res = []
    for d in range(ndev):
        dev = torch.device("cuda", d)
        mfn, mfd, _, _ = bench.build_models(dev)
        row = {"device": d}
        for name, m in (("fn", mfn), ("fd", mfd)):
            with torch.cuda.device(dev):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                m._ensure_handle(dev)
                torch.cuda.synchronize(dev)
                row[name + "_ms"] = (time.perf_counter() - t0) * 1e3
        res.append(row)
        del mfn, mfd
    return res


def timed_displace(gen, cloud, seeds, flush, steps, warmup):
    for _ in range(warmup):
        out = gen.displace_host(cloud, seeds)
    times = []
    for _ in range(steps):
        for f in flush:
            f.zero_()
        for f in flush:
            torch.cuda.synchronize(f.device)
        t0 = time.perf_counter()
        out = gen.displace_host(cloud, seeds)
        times.append(time.perf_counter() - t0)
    return out, times


def release_workspaces(*models):
    for m in models:
        m._ws = None            # drops the module's cached workspaces
    torch.cuda.empty_cache()


def run_bench(n, mode, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--config", "1", "--mode", mode, "--steps", str(steps),
           "--no-cpu-baseline", "--no-gpu-eager"]
    if n > 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(n)] + cmd[1:]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    line = next((ln for ln in reversed(p.stdout.strip().splitlines()) if ln.startswith("{")), None)
    if p.returncode != 0 or line is None:
        return {"rc": p.returncode, "stderr_tail": p.stderr[-2000:]}
    r = json.loads(line)
    return {"rc": 0, "value": r["value"], "e2e": r["e2e"]["value"], "ms_per_step": r["ms_per_step"], "clocks": r.get("clocks")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="1,2,4,8")
    ap.add_argument("--modes", default="tc,fast")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--bench-steps", type=int, default=5, help="bench.py --steps (0: do not run bench.py)")
    ap.add_argument("--no-upsample", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_device_bench.py: no CUDA device (the hot path has no CPU fallback)")
    import sapcu_b200.synthetic as syn
    from sapcu_b200.generation import Generator3D6
    from sapcu_b200.sharding import shard_bounds

    count = torch.cuda.device_count()
    emit({"record": "gpu", "device_count": count, **gpu_info()})
    ns = [n for n in (int(x) for x in args.devices.split(",")) if n <= count]
    emit({"record": "finalize", "per_device": finalize_times(max(ns))})

    primary = torch.device("cuda", 0)
    mfn, mfd, _, _ = bench.build_models(primary)
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    flush = [torch.empty(256 << 20, dtype=torch.uint8, device=torch.device("cuda", d)) for d in range(max(ns))]
    gens = {n: Generator3D6(mfn, mfd, ["cuda:%d" % d for d in range(n)], k_neighbors=bench.K_NEIGH, remove_outliers=False)
            for n in ns}
    single = Generator3D6(mfn, mfd, primary, k_neighbors=bench.K_NEIGH, remove_outliers=False)
    strong_seeds = syn.seeds(cloud, 32, seed=1)                    # 65,536 seeds
    for mode in args.modes.split(","):
        mfn.set_mode(mode), mfd.set_mode(mode)
        for n in ns:
            weak_seeds = syn.seeds(cloud, 4 * n, seed=1)             # bench.py --config 1 at --gpus n
            _, tw = timed_displace(gens[n], cloud, weak_seeds, flush[:n], args.steps, args.warmup)
            out, ts = timed_displace(gens[n], cloud, strong_seeds, flush[:n], args.steps, args.warmup)
            # the 1-device pipeline run shard by shard: what the N-device points must equal in every mode
            ref = np.concatenate([single.displace_host(cloud, strong_seeds[lo:hi]) for lo, hi in shard_bounds(strong_seeds.shape[0], n)])
            rec = {"record": "throughput", "mode": mode, "n_devices": n,
                   "weak": {"seeds": int(weak_seeds.shape[0]), "step_s": tw, "points_per_s": weak_seeds.shape[0] / float(np.mean(tw))},
                   "strong": {"seeds": int(strong_seeds.shape[0]), "step_s": ts, "points_per_s": strong_seeds.shape[0] / float(np.mean(ts))},
                   "identical": bool(np.array_equal(out, ref))}
            emit(rec)
            if args.bench_steps > 0:
                release_workspaces(mfn, mfd)
                b = run_bench(n, mode, args.bench_steps)
                emit({"record": "bench", "mode": mode, "n_devices": n, **b,
                      "single_process_weak_over_bench_e2e": rec["weak"]["points_per_s"] / b["e2e"] if b.get("e2e") else None})
        release_workspaces(mfn, mfd)

    if not args.no_upsample:
        mfn.set_mode("tc"), mfd.set_mode("tc")
        gen = Generator3D6(mfn, mfd, ["cuda:%d" % d for d in range(max(ns))], k_neighbors=bench.K_NEIGH, remove_outliers=True)
        small = syn.seeds(cloud, 1, seed=2)
        gen._outlier_filter(gen.displace_host(cloud, small))          # warm: kernels, handles, workspaces
        gen.gpu_seeds(cloud)
        t0 = time.perf_counter()
        seeds = gen.gpu_seeds(cloud)
        t1 = time.perf_counter()
        pts = gen.displace_host(cloud, seeds)
        t2 = time.perf_counter()
        kept = gen._outlier_filter(pts)
        t3 = time.perf_counter()
        emit({"record": "upsample", "mode": "tc", "n_devices": max(ns), "spacing": gen.dense_spacing, "seeds": int(seeds.shape[0]),
              "kept": int(kept.shape[0]), "seedgen_s": t1 - t0, "displace_s": t2 - t1, "outlier_s": t3 - t2,
              "seedgen_plus_outlier_share": (t1 - t0 + t3 - t2) / (t3 - t0)})


if __name__ == "__main__":
    main()
