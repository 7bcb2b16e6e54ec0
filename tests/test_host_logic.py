"""CPU: host-side logic -- the C ABI surface, configuration / checkpoint boundary, seed sharding."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import sapcu_b200
from sapcu_b200 import _native as N
from conftest import ROOT


def test_library_exports_every_declared_symbol():
    """include/sapcu_b200.h <-> libsapcu_b200.so <-> the ctypes table (no compute calls: no GPU here)."""
    hdr = open(os.path.join(ROOT, "include", "sapcu_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(sapcu_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(N.EXPORTS)
    sapcu_b200.build()
    lib = N.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.sapcu_abi_version() == 1
    # the counter is per process, and GPU tests of the same session may have launched kernels already: load a fresh copy
    fresh = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); import sapcu_b200; "
                            "print(sapcu_b200.lib().sapcu_launch_count())" % ROOT], capture_output=True, text=True, check=True)
    assert fresh.stdout.strip() == "0"
    assert lib.sapcu_knn_workspace_bytes(2048) >= 2048 * 12 + 256


def test_no_cpu_fallback_and_error_reporting():
    lib = N.lib()
    # bad hyper-parameters are rejected with a message, never a crash
    import ctypes
    cfg = (ctypes.c_int32 * 6)(24, 18, 12, 640, 6, 7)
    assert not lib.sapcu_model_create(N.MODEL_FN, cfg, 6)
    assert b"num_heads" in lib.sapcu_last_error()
    from sapcu_b200.fn import config as fc
    m = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    with pytest.raises(N.SapcuError, match="no CPU fallback"):
        m(torch.zeros(2, 100, 3))
    with pytest.raises(N.SapcuError):
        m.train()
    if not torch.cuda.is_available():
        # finalize needs a device: it must fail loudly rather than run anything on the host
        with pytest.raises(N.SapcuError):
            m._ensure_handle()


def test_config_and_checkpoint_boundary(tmp_path):
    from sapcu_b200.fn import config as fc, checkpoints as fck
    from sapcu_b200.fd import config as dc, checkpoints as dck
    import sapcu_b200.synthetic as syn
    # inherit_from + defaults
    base = tmp_path / "base.yaml"
    base.write_text("model:\n  k_values: [24, 18, 12]\n  emb_dims: 640\n  num_heads: 8\n")
    child = tmp_path / "child.yaml"
    child.write_text("inherit_from: base.yaml\nmodel:\n  time_steps_enc: 6\n  time_steps_dec: 9\n")
    cfg = fc.load_config(str(child))
    assert cfg["model"]["k_values"] == [24, 18, 12] and cfg["model"]["time_steps_enc"] == 6
    assert cfg["model"]["decoder_dropout"] == 0.1
    with pytest.raises(FileNotFoundError):
        fc.load_config(str(tmp_path / "nope.yaml"))
    with pytest.raises(ValueError):
        fc.get_model({"model": {"emb_dims": 640}})
    m = fc.get_model(cfg)
    assert m._cfg_ints() == [24, 18, 12, 640, 6, 8]
    d = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    assert d._cfg_ints() == [32, 768, 7, 8, 4, 8, 16, 32, 48]
    # checkpoint round trip, incl. the DataParallel 'module.' prefix the reference strips
    syn.init_weights(m, 5, True)
    sd = {("module." + k): v.clone() for k, v in m.state_dict().items()}
    torch.save({"model": sd, "epoch_it": 3}, tmp_path / "model_best.pt")
    m2 = fc.get_model(cfg)
    scalars = fck.CheckpointIO(str(tmp_path), model=m2).load("model_best.pt")
    assert scalars == {"epoch_it": 3}
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    with pytest.raises(FileExistsError):
        fck.CheckpointIO(str(tmp_path), model=m2).load("missing.pt")
    with pytest.raises(FileNotFoundError):
        dck.CheckpointIO(str(tmp_path), model=d).load("missing.pt")


def test_reference_yaml_loads_unchanged():
    """The reference's own full config files (SAPCU_REFERENCE names its checkout) load through our loaders."""
    ref = os.path.join(os.environ.get("SAPCU_REFERENCE", ""), "config")
    if not os.environ.get("SAPCU_REFERENCE") or not os.path.isdir(ref):
        pytest.skip("SAPCU_REFERENCE does not name a checkout of the reference")
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    assert fc.get_model(fc.load_config(ref + "/fn.yaml"))._cfg_ints() == [24, 18, 12, 640, 6, 8]
    assert dc.get_model(dc.load_config(ref + "/fd.yaml"), None)._cfg_ints() == [32, 768, 7, 8, 4, 8, 16, 32, 48]


def test_shard_bounds():
    from sapcu_b200.sharding import shard_bounds
    for S in (0, 1, 7, 8192, 370000):
        for G in (1, 2, 4, 8):
            b = shard_bounds(S, G)
            assert b[0][0] == 0 and b[-1][1] == S
            assert all(b[i][1] == b[i + 1][0] for i in range(G - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
import sapcu_b200
from sapcu_b200.sharding import shard_range, all_gather_rows
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%%s' %% sys.argv[2], rank=int(sys.argv[1]), world_size=2)
S = 11
full = torch.arange(S * 3, dtype=torch.float64).view(S, 3) * 0.5
lo, hi = shard_range(S, dist.get_rank(), 2)
out = all_gather_rows(full[lo:hi].clone(), S)
assert torch.equal(out, full), out
dist.destroy_process_group()
print('ok')
"""


def test_all_gather_rows_world2_gloo(tmp_path):
    """N>1 path on CPU: two gloo ranks shard 11 rows (ragged: 6 + 5), pad, all-gather, trim."""
    script = tmp_path / "w.py"
    script.write_text(_WORKER % ROOT)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=300)
        assert p.returncode == 0 and b"ok" in out, out.decode()


def test_shard_batch_offsets():
    """Strong-scaling shards of a batch of clouds: the flat (cloud, seed) list is cut into contiguous ranges; each rank's
    per-cloud seed offsets are the global prefix table clipped to its range."""
    from sapcu_b200.sharding import shard_bounds, shard_batch_offsets
    so = np.array([0, 5, 5, 12, 20], dtype=np.int64)           # 4 clouds, the second without seeds
    for world in (1, 2, 3, 8):
        total = np.zeros(4, dtype=np.int64)
        for lo, hi in shard_bounds(20, world):
            loc = shard_batch_offsets(so, lo, hi)
            assert loc[0] == 0 and loc[-1] == hi - lo and (np.diff(loc) >= 0).all()
            total += np.diff(loc)
        assert np.array_equal(total, np.diff(so))


def test_bench_kernel_roofline_grading():
    """bench.kernel_rooflines: the tensor bound is chosen on the issued products (3 per MAC in the parity-grade mode) while `frac`
    stays algorithmic; a layer running above the MUFU ceiling is tabulated and is not graded on the MUFU roofline."""
    import importlib
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    bench = importlib.import_module("bench")
    peaks = {"bf16_tflops_sustained": 1000.0, "hbm_gbs": 5000.0}
    ms = 10.0
    rep = [
        # 200 TFLOP/s algorithmic (0.2), 2 TB/s (0.4), LIF 2x the ceiling -> tabulated, tensor issued 0.6 wins over hbm 0.4
        {"label": "fn.fc_delta2+lif", "launches": 3, "ms": ms, "flops": 200e12 * ms / 1e3, "bytes": 2000e9 * ms / 1e3, "lif_elsteps": 2 * bench.LIF_CEILING * ms / 1e3},
        # a MUFU-bound layer below the ceiling keeps the MUFU roofline
        {"label": "fn.conv1+lif", "launches": 1, "ms": ms, "flops": 0.0, "bytes": 100e9 * ms / 1e3, "lif_elsteps": 0.5 * bench.LIF_CEILING * ms / 1e3},
        # top-k kernel: flops recorded but not a contraction, far below every roofline
        {"label": "fd.intra_knn(features)", "launches": 3, "ms": ms, "flops": 1e12 * ms / 1e3, "bytes": 50e9 * ms / 1e3, "lif_elsteps": 0.0},
    ]
    rows = {r["kernel"]: r for r in bench.kernel_rooflines(rep, 1, peaks, 3 * ms, products=3)}
    d2 = rows["fn.fc_delta2+lif"]
    assert d2["bound"] == "tensor" and abs(d2["frac"] - 0.2) < 1e-9 and abs(d2["tensor_issued_frac"] - 0.6) < 1e-9 and "lif" in d2
    c1 = rows["fn.conv1+lif"]
    assert c1["bound"] == "mufu" and abs(c1["frac"] - 0.5) < 1e-9 and "lif" not in c1
    kn = rows["fd.intra_knn(features)"]
    assert kn["tensor_issued_frac"] == kn["tensor_frac"] and "note" in kn


def test_lif_table_host_selftest():
    """The tabulated LIF^T chains without a GPU: the library builds the table as sapcu_model_finalize does and evaluates the host
    restatement of the kernels' lookup (same fp32 operations) against the exact fp64 recurrence -- default-initialised neurons
    (all channels share one fit) and parameters spread over the reference's clamp ranges, incl. zero, the cell boundaries and
    their fp32 neighbours.  Bound: 5e-5 absolute on soft spikes in (0, 0.7) (the fit accepts 4e-5 at its check points)."""
    import ctypes
    import numpy as np
    import sapcu_b200
    L = sapcu_b200.lib()
    rng = np.random.default_rng(5)
    C = 256
    default = np.stack([np.full(C, 0.9), np.full(C, 0.01), np.full(C, 0.5), np.full(C, 1.0)]).astype(np.float32)
    spread = np.stack([rng.uniform(0.5, 0.99, C), rng.uniform(0.0, 0.1, C), rng.uniform(0.1, 0.9, C), rng.uniform(0.5, 2.0, C)]).astype(np.float32)
    for name, prm, T in (("default", default, 4), ("spread", spread, 4), ("spread_T6", spread[:, :128].copy(), 6)):
        prm = np.ascontiguousarray(prm)
        err, fit, blk = ctypes.c_double(), ctypes.c_double(), ctypes.c_uint32()
        rc = L.sapcu_lif_table_selftest(prm.ctypes.data_as(ctypes.c_void_p), prm.shape[1], T, 400, ctypes.byref(err), ctypes.byref(fit), ctypes.byref(blk))
        assert rc == 0, sapcu_b200.lib().sapcu_last_error()
        print("lif table [%s]: max |table - exact| %.2e, fit %.2e, largest block %d bytes" % (name, err.value, fit.value, blk.value))
        assert err.value < 5e-5 and fit.value <= 4.0001e-5
        assert blk.value <= 120 * 1024
    assert L.sapcu_lif_table_selftest(None, 4, 4, 10, ctypes.byref(err), ctypes.byref(fit), ctypes.byref(blk)) != 0
