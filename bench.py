#!/usr/bin/env python
"""Benchmark of the generation.py hot path (seed->cloud kNN, gather/centre, fn, rotate, fd, x + n*d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|3|4|5] [--mode fp32|tc|tf32|fast]
                    [--dump-outputs DIR]

Workloads (BASELINE.json `configs`, 0-based in the file; the numbers below are the file's positions 1..4 + 1):
  --config 1 (default)  configs[1]: one 2,048-pt sphere cloud x4 -> 8,192 seeds PER GPU (weak scaling), parity mode `tc`
  --config 3            configs[2]: 64 ShapeNet-shaped 2,048-pt clouds x16 = 2,097,152 seeds, FIXED total (strong scaling),
                        one batched kNN over the 64 clouds, fast mode
  --config 4            configs[3]: one 100,000-pt scan x3.7 = 370,000 seeds, fixed total (strong scaling), fast mode
  --config 5            configs[4]: one 2,000,000-pt cloud x16 = 32,000,000 seeds, fixed total (strong scaling), fast mode
A step is one pass of the whole hot path over the rank's seeds; K = 100 neighbours; seeded random-init config/fn.yaml +
config/fd.yaml weights.  N > 1: contiguous ranges of the flat seed list per rank, clouds + weights replicated, ONE NCCL
all-gather of the displaced points ends every step (SURVEY.md section 8e).

Prints ONE JSON line (rank 0).  `value` = seeds/s with inputs resident in HBM (CUDA events, max over ranks); `e2e` = the
same through sharding.upsample_sharded_host (host numpy in, host numpy out: pinned H2D of cloud + seeds, the all-gather
and the D2H of the gathered points inside the timed region).  `--impl reference` times the reference algorithm's CPU path
(the oracle restatement, bit-identical to the reference, SURVEY.md section 8c) on the host cores on a bounded sample.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

K_NEIGH = 100
METRIC = "upsampled points/sec (fn+fd, device-timed)"
UNIT = "points/s"
LIF_CEILING = 1.33e12        # LIF element-steps/s one B200 sustains in registers (tools/mufu_bench.cu, profiles/r01_mufu_microbench.txt)

CONFIGS = {
    1: dict(name="configs[1]", clouds=1, n=2048, ratio=4, shape="sphere", scaling="weak", mode="tc"),
    3: dict(name="configs[2]", clouds=64, n=2048, ratio=16, shape="boxes", scaling="strong", mode="fast"),
    4: dict(name="configs[3]", clouds=1, n=100000, ratio=3.7, shape="boxes", scaling="strong", mode="fast"),
    5: dict(name="configs[4]", clouds=1, n=2000000, ratio=16, shape="sphere", scaling="strong", mode="fast"),
}
MODE_TEXT = {
    "fp32": ("f32", "fp32 parity mode (FFMA contractions)"),
    "tc": ("fp16x3/tf32x3 (fp32 accumulate)", "fp32 parity mode (tcgen05 contractions with 3 split products per MAC: fp16 hi/lo on "
           "spike-tensor inputs, tf32 hi/lo elsewhere; fp32 accumulate)"),
    "tf32": ("tf32", "single-pass TF32 tcgen05 contractions, fp32-grade neuron (deviation in profiles/)"),
    "fast": ("fp16 (fp32 accumulate)", "fast mode: single-product fp16 tcgen05 contractions on fp16 spike tensors, tabulated LIF^T "
             "chains (deviation reported in profiles/r02_parity.json)"),
}


def build_models(device=None, stress=False):
    import sapcu_b200
    import sapcu_b200.synthetic as syn
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=stress)
    syn.init_weights(mfd, seed=200, stress=stress)
    sd_fn = {k: v.clone() for k, v in mfn.state_dict().items()}
    sd_fd = {k: v.clone() for k, v in mfd.state_dict().items()}
    if device is not None:
        mfn, mfd = mfn.to(device), mfd.to(device)
    return mfn, mfd, sd_fn, sd_fd


def workload(cfg_id, world):
    """(cloud [Ntot,3] f64, seeds [S,3] f64, batch=(cloud_off, seed_off) | None, description).  Weak scaling (config 1)
    grows the seed set with the world size; the other configs have a fixed total."""
    import sapcu_b200.synthetic as syn
    c = CONFIGS[cfg_id]
    if c["clouds"] == 1:
        cloud = syn.cloud(c["n"], seed=0, shape=c["shape"])
        ratio = c["ratio"] * (world if c["scaling"] == "weak" else 1)
        seeds = syn.seeds(cloud, ratio, seed=1)
        return cloud, seeds, None
    clouds = [syn.cloud(c["n"], seed=10 + b, shape=c["shape"]) for b in range(c["clouds"])]
    seeds = [syn.seeds(cl, c["ratio"], seed=100 + b) for b, cl in enumerate(clouds)]
    co = np.concatenate([[0], np.cumsum([x.shape[0] for x in clouds])]).astype(np.int64)
    so = np.concatenate([[0], np.cumsum([x.shape[0] for x in seeds])]).astype(np.int64)
    return np.concatenate(clouds, 0), np.concatenate(seeds, 0), (co, so)


def workload_text(cfg_id, mode, world, S_total):
    c = CONFIGS[cfg_id]
    what = {1: "2,048-pt sphere cloud x4 -> 8,192 seeds per GPU",
            3: "batch of 64 ShapeNet-shaped (3 boxes + cylinder) 2,048-pt clouds x16 = 2,097,152 seeds, fixed total, one batched kNN",
            4: "100,000-pt scan x3.7 = 370,000 seeds, fixed total",
            5: "2,000,000-pt cloud x16 = 32,000,000 seeds, fixed total"}[cfg_id]
    return "%s: %s, K=100, fn.yaml+fd.yaml random-init weights, %s" % (c["name"], what, MODE_TEXT[mode][1])


def sample_problem(cfg_id, cloud, seeds, batch, n):
    """A bounded sample of the workload for the CPU / GPU-eager baselines: n seeds of the first cloud (cost is per-seed
    independent; only the kNN depends on the cloud size)."""
    if batch is not None:
        co, so = batch
        return cloud[co[0]:co[1]], seeds[so[0]:so[1]][:n]
    return cloud, seeds[:n]


def cpu_reference_rate(sd_fn, sd_fd, cloud, seeds, n_sample, steps=1, warmup=0, device=None):
    """The reference algorithm's path (oracle, faithful schedule) on `n_sample` seeds per step; device=None: host cores."""
    import sapcu_oracle as orc
    times = []
    for i in range(warmup + steps):
        sl = seeds[(i * n_sample) % max(1, len(seeds) - n_sample):][:n_sample]
        if device is not None:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        orc.pipeline(sd_fn, sd_fd, cloud, sl, K=K_NEIGH, batch=256, schedule="faithful", device=device)
        if device is not None:
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return n_sample * len(times) / sum(times), sum(times) / len(times)


def host_threads():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arms size their thread pool themselves."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled during the timed region: NVML in-process (every 20 ms), else nvidia-smi."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.nvml, self.handle, self.max_mhz = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _nvml_sample(self):
        n = self.nvml
        mhz = int(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = int(get(self.handle))
        bits = [0x8, 0x40, 0x20, 0x4]     # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
        return [str(mhz), str(self.max_mhz)] + ["Active" if r & b else "Not Active" for b in bits]

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self.samples.append(self._nvml_sample())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    if len(f) >= 6:
                        self.samples.append(f)
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nvml is not None else 0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = sorted({n for s in self.samples for n, v in zip(self.NAMES, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port), rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_threads()
    _, _, sd_fn, sd_fd = build_models(None)
    cloud, seeds, batch = workload(args.config, 1)
    n_sample = 48 if args.config != 5 else 16      # ~7 s of host work per step on 16 cores
    # keep the whole --steps K --warmup W run within a few minutes on any host, whatever K and W are (cost is per seed, so the
    # rate does not depend on the sample): one calibration pass of 8 seeds, then the per-step sample that fits ~150 s in total
    c0, s0 = sample_problem(args.config, cloud, seeds, batch, 9)
    r0, _ = cpu_reference_rate(sd_fn, sd_fd, c0, s0, 8)
    n_sample = int(max(4, min(n_sample, r0 * 150.0 / max(1, args.steps + args.warmup))))
    c1, s1 = sample_problem(args.config, cloud, seeds, batch, max(n_sample * (args.steps + args.warmup), n_sample + 1))
    rate, sec = cpu_reference_rate(sd_fn, sd_fd, c1, s1, n_sample, steps=args.steps, warmup=args.warmup)
    c = CONFIGS[args.config]
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.config, "fp32", 1, seeds.shape[0]).rsplit(", ", 1)[0] + ", fp32 (reference algorithm on the host cores)",
                   "bounded_sample": "%d seeds per step (cost is per-seed independent)" % n_sample},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d seeds/step x %d steps through oracle.pipeline (reference algorithm, faithful schedule)" % (n_sample, args.steps)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def dump_points(path, pts, limit=64 << 20):
    """--dump-outputs: the [S,3] f64 points of the last timed step as <path>/points.npy, so that two builds can be compared
    output for output.  Above `limit` bytes, a fixed seeded sample of rows (ascending order) that is the same at every run."""
    if pts.nbytes > limit:
        n = limit // pts.itemsize // pts.shape[1]
        pts = pts[np.sort(np.random.default_rng(0).choice(pts.shape[0], n, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "points.npy"), pts)


def kernel_rooflines(report, steps, peaks, step_ms_total, products=1):
    """Per-kernel roofline entries from the library's live recording: each label is graded on the roofline that binds it
    (tensor: FLOPs vs the measured sustained bf16 peak -- `frac` is ALGORITHMIC, the bound is chosen on the ISSUED products,
    `products` per MAC in this mode; mufu: LIF element-steps vs the measured in-register ceiling of the MUFU recurrence;
    hbm: algorithmic bytes vs the measured copy bandwidth).  A layer that runs above the MUFU ceiling does not execute the
    MUFU recurrence at all (tabulated LIF^T chain): that roofline does not apply to it and it is graded on tensor / HBM."""
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_gb = float(peaks.get("hbm_gbs", 6650.0))
    out = []
    for e in report:
        ms = e["ms"] / steps
        if ms <= 0:
            continue
        tf = e["flops"] / steps / ms / 1e9
        gb = e["bytes"] / steps / ms / 1e6
        ls = e["lif_elsteps"] / steps / ms * 1e3
        fr = {"tensor": tf / peak_tf, "hbm": gb / peak_gb, "mufu": ls / LIF_CEILING}
        contraction = e["flops"] > 0 and "intra_knn" not in e["label"] and "block0" not in e["label"]
        issued = fr["tensor"] * (products if contraction else 1)
        tabulated = fr["mufu"] > 1.0
        cand = {"tensor": issued, "hbm": fr["hbm"]}
        if not tabulated:
            cand["mufu"] = fr["mufu"]
        bound = max(cand, key=cand.get)
        row = {"kernel": e["label"], "launches_per_step": e["launches"] / steps, "ms_per_step": ms,
               "share_of_step": e["ms"] / max(step_ms_total, 1e-9), "bound": bound, "frac": fr[bound],
               "tensor_tflops": tf, "tensor_frac": fr["tensor"], "tensor_issued_frac": issued, "hbm_gbs": gb, "hbm_frac": fr["hbm"],
               "lif_elsteps_per_s": ls, "mufu_frac": fr["mufu"]}
        if tabulated:
            row["lif"] = "tabulated LIF^T chain: no MUFU recurrence executed, the MUFU roofline does not apply"
        if max(cand.values()) < 0.15:
            row["note"] = "below 15 % of every roofline: issue / latency-bound (shared-memory top-k, gathers); pipe utilisation in the ncu summaries under profiles/"
        out.append(row)
    out.sort(key=lambda r: -r["ms_per_step"])
    return out


def run_ours(args):
    import torch.distributed as dist
    import sapcu_b200
    from sapcu_b200 import _native as N
    from sapcu_b200.generation import Generator3D6
    from sapcu_b200.sharding import shard_range, all_gather_rows, shard_batch_offsets, upsample_sharded_host

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sapcu_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = sapcu_b200.lib()
    cfg = CONFIGS[args.config]
    mode = args.mode or cfg["mode"]
    mfn, mfd, sd_fn, sd_fd = build_models(dev, stress=args.init == "stress")
    mfn.set_mode(mode), mfd.set_mode(mode)
    cloud, seeds, batch = workload(args.config, world)
    S_total = seeds.shape[0]
    lo, hi = shard_range(S_total, rank, world)
    lbatch = None if batch is None else (batch[0], shard_batch_offsets(batch[1], lo, hi))
    gen = Generator3D6(mfn, mfd, dev, k_neighbors=K_NEIGH, remove_outliers=False,
                       seeds_per_pass=args.seeds_per_pass if (hi - lo) > args.seeds_per_pass else None)
    d_cloud = torch.from_numpy(cloud).to(dev)
    d_seeds = torch.from_numpy(np.ascontiguousarray(seeds[lo:hi])).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        out = gen.displace_device(d_cloud, d_seeds, batch=lbatch)
        return all_gather_rows(out, S_total) if world > 1 else out

    # warm-up: W steps; for the large fixed-size configs each warm-up step runs on a leading fraction of the rank's seeds
    # (kernels, workspaces, clocks and the NCCL communicator are warm after it; the timed steps are always full size)
    wfrac = args.warmup_frac if args.warmup_frac is not None else {1: 1.0, 3: 0.25, 4: 0.25, 5: 0.0625}[args.config]
    if wfrac >= 1.0:
        for _ in range(args.warmup):
            step()
    else:
        nw = max(1024, int((hi - lo) * wfrac))
        d_seeds_w = d_seeds[:nw].contiguous()
        wb = None if lbatch is None else (lbatch[0], np.minimum(lbatch[1], nw))
        for _ in range(args.warmup):
            o = gen.displace_device(d_cloud, d_seeds_w, batch=wb)
            if world > 1:
                all_gather_rows(o, nw * world)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    L.sapcu_profile(1)
    launches0 = L.sapcu_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in ev:
        flush.zero_()                        # L2 flush between timed iterations (outside the event pair)
        a.record()
        out = step()
        b.record()
    barrier()
    launches = L.sapcu_launch_count() - launches0
    ms = sum(a.elapsed_time(b) for a, b in ev)
    gms, gfl, gn = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
    N.check(L.sapcu_profile_read(ctypes.byref(gms), ctypes.byref(gfl), ctypes.byref(gn)), "profile_read")
    need = L.sapcu_profile_report(None, 0)
    buf = ctypes.create_string_buffer(int(max(need, 2)))
    L.sapcu_profile_report(buf, len(buf))
    report = json.loads(buf.value.decode() or "[]")
    L.sapcu_profile(0)
    sampler.stop_flag.set()
    sampler.join(timeout=5)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = S_total * args.steps / (ms_total / 1e3)
    assert out.shape == (S_total, 3) and bool(torch.isfinite(out).all())
    N.check_device("bench")
    last_out = out.cpu().numpy() if args.dump_outputs and rank == 0 else None      # before the e2e leg reuses the generator

    # ---- end to end through the public host API: every step copies the cloud and the rank's seeds from pinned host memory,
    # runs the pipeline, all-gathers, and copies the gathered [S,3] points back to the host (L2 flushed between steps)
    e2e_steps = args.steps if args.config == 1 else min(args.steps, 1)
    if args.no_e2e:
        e2e_steps = 0
    if args.config == 1:
        upsample_sharded_host(gen, cloud, seeds, batch=batch)          # warm the pinned buffers (small config only)
    e2e_s = 0.0
    pts = None
    for _ in range(e2e_steps):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        pts = upsample_sharded_host(gen, cloud, seeds, batch=batch)
        e2e_s += time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = S_total * e2e_steps / float(t.item()) if e2e_steps else None
    assert pts is None or (pts.shape == (S_total, 3) and np.isfinite(pts).all())

    if rank == 0:
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        kernels = kernel_rooflines(report, args.steps, peaks, ms, products=3 if mode == "tc" else 1)
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        achieved_tf = (gfl.value / max(gms.value, 1e-9)) / 1e9        # FLOP / ms -> TFLOP/s
        traffic = None
        for tr in ("r02_gemm_traffic_%s.json" % mode, "r01_gemm_traffic.json"):
            tr = os.path.join(ROOT, "profiles", tr)
            if args.config == 1 and world == 1 and os.path.exists(tr) and (mode == "tc" or "r02" in tr):
                traffic = json.load(open(tr)).get("traffic_bytes_per_step")   # dram bytes of the same kernels, one ncu pass
                break
        cpu = None
        gpu_eager = None
        if world == 1 and not args.no_cpu_baseline:
            cores = host_threads()
            ns = 96 if args.config != 5 else 16
            c1, s1 = sample_problem(args.config, cloud, seeds, batch, ns)
            rate, _ = cpu_reference_rate(sd_fn, sd_fd, c1, s1, ns)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "%d seeds of the same workload through oracle.pipeline (reference algorithm, faithful schedule)" % ns}
        if world == 1 and not args.no_gpu_eager and args.config != 5:
            # the reference as it would run on this GPU: PyTorch-eager fp32 (TF32 off), 256-patch sub-batches, host kNN/rotations
            # exactly as generation.py does -- the baseline SURVEY.md section 2a names.  Test infrastructure, not the product.
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            ns = 512
            c1, s1 = sample_problem(args.config, cloud, seeds, batch, ns * 3)
            rate, _ = cpu_reference_rate(sd_fn, sd_fd, c1, s1, ns, steps=2, warmup=1, device=dev)
            gpu_eager = {"value": rate, "unit": UNIT, "kind": "port (oracle restatement of the reference, torch eager on cuda:0, TF32 off)",
                         "sample": "512 seeds/step x 2 steps, 256-patch sub-batches, faithful schedule; kNN / gather / rotations on the host as in generation.py"}
        dom = kernels[0] if kernels else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": MODE_TEXT[mode][0], "data": "synthetic",
            "config": {"workload": workload_text(args.config, mode, world, S_total) + (" [stress-init weights: per-channel neuron parameters spread over their clamp ranges]" if args.init == "stress" else ""), "mode": mode,
                       "seeds_total": S_total, "l2": "256 MiB flush buffer written between timed steps",
                       "warmup_steps_seed_fraction": wfrac,
                       "collective": "one all-gather of [S,3] f64 per step" if world > 1 else "none"},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(cloud.nbytes + (hi - lo) * 24), "d2h_bytes_per_step": int(S_total * 24),
                    "path": "sharding.upsample_sharded_host: pinned H2D (cloud + this rank's seeds), pipeline, all-gather, D2H of the gathered [S,3] f64"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "contraction family (gemm_tc2_kernel + gemm_tc_kernel; rows < 1024 on gemm_simt_kernel)" if mode != "fp32" else "gemm_simt_kernel (all contractions)",
                         "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s",
                         "traffic": traffic, "traffic_note": "dram read+write bytes summed over the contraction launches of ONE step (ncu, profiles/); achieved/kernel_ms are likewise per-step sums over the family",
                         "executed_tflops": achieved_tf * (3 if mode == "tc" else 1),
                         "executed_note": {"tc": "3 split products per MAC are issued in the parity mode, so frac <= ~0.3 by construction", "fast": "one fp16 product per MAC", "tf32": "one tf32 product per MAC", "fp32": "FFMA"}[mode],
                         "kernel_ms_per_step": gms.value / args.steps, "kernel_launches_per_step": gn.value / args.steps,
                         "kernel_share_of_step": gms.value / max(ms, 1e-9), "algorithmic_gflop_per_step": gfl.value / args.steps / 1e9,
                         "dominant_kernel": dom,
                         "lif_ceiling_elsteps_per_s": LIF_CEILING, "hbm_peak_gbs": float(peaks.get("hbm_gbs", 6650.0))},
            "roofline_kernels": kernels,
            "cpu_baseline": cpu,
            "gpu_eager_baseline": gpu_eager,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_points(args.dump_outputs, last_out)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS))
    ap.add_argument("--mode", default=None, choices=["fp32", "tc", "tf32", "fast"])
    ap.add_argument("--seeds-per-pass", type=int, default=262144, help="device-side pass size for large seed sets")
    ap.add_argument("--init", default="default", choices=["default", "stress"], help="weight init: the yaml random-init (default) or the parity suite's stress init")
    ap.add_argument("--warmup-frac", type=float, default=None, help="fraction of the rank's seeds a warm-up step runs on (default: 1 for config 1, less for the large configs)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-API end-to-end leg (large configs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the points the last one computed as DIR/points.npy (f64; a fixed sample above 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
