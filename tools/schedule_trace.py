"""Launch-for-launch comparison of two builds of the library (refactors of the host-side schedule must not change it).

    python tools/schedule_trace.py OLD.so NEW.so [--out DIR]

For each build and each set of schedule switches (defaults; the three fusions off; the fast mode's LIF tables off) one
subprocess runs fn and fd in every mode over the cases below and records, per case: the ordered kernel list from
torch.profiler (mangled names carry every template argument) with grid, block and shared memory, sapcu_launch_count, the
tap formats and a hash of the output bytes.  Any difference is printed and makes the exit status 1.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENVS = {"default": {}, "unfused": {"SAPCU_TC_FUSE_ATTNOUT": "0", "SAPCU_TC_FACTOR_ATTNIN": "0", "SAPCU_TC_FUSE_POOL": "0"},
        "no_tables": {"SAPCU_FAST_LIF_TABLES": "0"}}


def _record(lib, m, run, taps, outputs):
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    n0 = lib.sapcu_launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run()
        torch.cuda.synchronize()
    launches = lib.sapcu_launch_count() - n0
    with tempfile.NamedTemporaryFile(suffix=".json") as f:
        prof.export_chrome_trace(f.name)
        ev = json.load(open(f.name))["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    a = lambda e: e.get("args", {})
    return dict(kernels=[[e["name"], a(e).get("grid"), a(e).get("block"), a(e).get("shared memory")] for e in kern],
                launches=launches, taps={t: lib.sapcu_model_tap_format(m._ensure_handle(), t.encode()) for t in taps},
                out=hashlib.sha256(b"".join(t.cpu().numpy().tobytes() for t in outputs(out))).hexdigest())


def child():
    sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
    import copy
    import torch
    import sapcu_b200
    import sapcu_b200.synthetic as syn
    from sapcu_b200 import _native as N
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    import sapcu_oracle as orc
    import oracle_c
    lib, dev = N.lib(), "cuda:0"
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 4, seed=1)

    def patches(B, M):
        return torch.from_numpy(orc.gather_center(cloud, seeds[:B], oracle_c.knn(cloud, seeds[:B], M))).to(dev)

    def models(yaml=True):
        cfn = copy.deepcopy(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
        cfd = copy.deepcopy(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")))
        if not yaml:      # the configs of test_non_yaml_configs_take_the_fallback_paths
            cfn["model"].update(k_values=[16, 10, 6], time_steps_enc=4)
            cfd["model"].update(k=18, k_scales=[4, 8, 12, 20], time_steps_enc=5)
        mfn, mfd = fc.get_model(cfn), dc.get_model(cfd, None)
        syn.init_weights(mfn, seed=100 if yaml else 11, stress=True)
        syn.init_weights(mfd, seed=200 if yaml else 12, stress=True)
        return mfn.to(dev), mfd.to(dev)

    yaml_models, other_models = models(), models(False)
    fn_taps, fd_taps = ["trans1.snn1", "trans1.snn_delta2", "trans1.snn_gamma"], ["spikes"]
    cases = {"48": (48, 100, {}), "16": (16, 100, {}), "8": (8, 100, {}), "M64": (48, 64, {}), "non_yaml": (48, 100, {"yaml": False}),
             "3_chunks": (48, 100, {"cap": 16}), "stop1": (48, 100, {"stop": 1}), "stop2": (48, 100, {"stop": 2}),
             "forced": (48, 100, {"forced": True})}
    res = {}
    for mode in ("fp32", "tc", "tf32", "fast"):
        for name, (B, M, o) in cases.items():
            mfn, mfd = yaml_models if o.get("yaml", True) else other_models
            p = patches(B, M)
            for kind, m in (("fn", mfn), ("fd", mfd)):
                if (kind == "fn" and o.get("forced")) or (kind == "fd" and o.get("stop")):
                    continue
                m.set_mode(mode)
                m.WORKSPACE_CAP = lib.sapcu_model_workspace_bytes(m._ensure_handle(), o["cap"], M) if "cap" in o else type(m).WORKSPACE_CAP
                m._ws = None
                stop, outputs = o.get("stop", 0), lambda out: [out]
                if kind == "fn":
                    run = lambda: m(p, _stop_after_block=stop)
                    if stop:      # the normals are not computed: the stopped block's intermediates are the result
                        outputs = lambda out: [m.tap("trans%d.%s" % (stop, t), B, M) for t in ("snn1", "snn_qkv", "snn_delta2", "snn_gamma", "res")]
                else:
                    g = torch.Generator().manual_seed(B * M)
                    forced = torch.randint(0, M, (3, B, M, min(m.k, M)), generator=g, dtype=torch.int32).to(dev) if o.get("forced") else None
                    run = lambda: m(p, forced_idx=forced)
                res["%s/%s/%s" % (kind, mode, name)] = _record(lib, m, run, fn_taps if kind == "fn" else fd_taps, outputs)
            N.check_device(name)
    json.dump(res, open(sys.argv[sys.argv.index("--child") + 1], "w"))


def main():
    old, new = sys.argv[1], sys.argv[2]
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    bad = 0
    for env_name, env in ENVS.items():
        runs = []
        for so in (old, new):
            with tempfile.NamedTemporaryFile(suffix=".json") as f:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", f.name], env=dict(os.environ, SAPCU_LIB=so, **env),
                                   capture_output=True, text=True)
                if r.returncode:
                    sys.exit("%s (%s) failed:\n%s" % (so, env_name, r.stderr[-4000:]))
                runs.append(json.load(open(f.name)))
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            json.dump(dict(zip(("old", "new"), runs)), open(os.path.join(out_dir, "trace_%s.json" % env_name), "w"))
        for case in sorted(set(runs[0]) | set(runs[1])):
            a, b = runs[0].get(case), runs[1].get(case)
            same = a == b
            bad += not same
            print("%-9s %-22s %s  %3d kernels  taps %s" % (env_name, case, "same" if same else "DIFFERENT",
                                                        len((a or b)["kernels"]), (a or b)["taps"]))
    print("%d difference(s)" % bad)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    child() if "--child" in sys.argv else main()
