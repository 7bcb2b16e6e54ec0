"""GPU: one process driving several devices -- Generator3D6 over a device list, nn.DataParallel over the model shims, the
device guard of the C ABI and one module on two streams.  Seeds are independent units, so a sharded run must equal the
single-device pipeline run shard by shard; in MODE_FP32 (split-invariant) it also equals the unsharded run.  Repeated
entries of one device emulate several workers on a one-GPU box."""
import os
import threading

import numpy as np
import pytest
import torch

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
from sapcu_b200.generation import Generator3D6
from sapcu_b200.sharding import shard_batch_offsets, shard_bounds

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SAPCU_ESTATE = -4


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


@pytest.fixture(scope="module")
def sphere():
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    return cloud, syn.seeds(cloud, 4, seed=1)[:600]


def _models(device=DEV):
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    return mfn.to(device), mfd.to(device)


def _real_devices(lib):
    n = min(8, torch.cuda.device_count())
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    return ["cuda:%d" % i for i in range(n)]


def _check_sharded_displace(mfn, mfd, devices, cloud, seeds, mode):
    """displace_device / displace_host over `devices` against the single-device pipeline run shard by shard."""
    mfn.set_mode(mode), mfd.set_mode(mode)
    single = Generator3D6(mfn, mfd, DEV, k_neighbors=100, remove_outliers=False)
    multi = Generator3D6(mfn, mfd, devices, k_neighbors=100, remove_outliers=False)
    assert multi.device == torch.device(DEV) and len(multi.devices) == len(devices)
    d_c, d_s = torch.from_numpy(cloud).to(DEV), torch.from_numpy(seeds).to(DEV)
    bounds = shard_bounds(seeds.shape[0], len(devices))
    ref = [single.displace_device(d_c, d_s[lo:hi].contiguous(), return_parts=True) for lo, hi in bounds]
    ref = [torch.cat([r[j] for r in ref]).cpu().numpy() for j in range(4)]
    got = multi.displace_device(d_c, d_s, return_parts=True)
    assert all(t.device == torch.device(DEV) for t in got)
    got = [t.cpu().numpy() for t in got]
    for j, name in enumerate(("points", "idx", "normals", "dist")):
        assert np.array_equal(got[j], ref[j]), (mode, name)
    assert np.array_equal(multi.displace_device(d_c, d_s).cpu().numpy(), ref[0])
    assert np.array_equal(multi.displace_host(cloud, seeds), ref[0])
    if mode == "fp32":                       # MODE_FP32 is split-invariant: the unsharded run too
        assert np.array_equal(single.displace_device(d_c, d_s).cpu().numpy(), ref[0])
    return single, multi


@pytest.mark.parametrize("mode", ["fp32", "tc", "fast"])
def test_emulated_workers_equal_per_shard_runs(lib, sphere, mode):
    cloud, seeds = sphere
    assert seeds.shape[0] == 600
    mfn, mfd = _models()
    _check_sharded_displace(mfn, mfd, [DEV] * 3, cloud, seeds, mode)
    N.check_device("emulated workers")


def test_worker_exception_is_raised_after_all_workers_finish(lib, sphere):
    cloud, seeds = sphere
    mfn, mfd = _models()
    gen = Generator3D6(mfn, mfd, [DEV] * 3, k_neighbors=100, remove_outliers=False)
    d_c, d_s = torch.from_numpy(cloud).to(DEV), torch.from_numpy(seeds).to(DEV)
    finished = []

    def work(dev, lo, hi):
        if lo == 0:
            raise ValueError("shard 0 failed")
        finished.append(lo)
        return gen._displace_local(d_c, d_s[lo:hi].contiguous())
    with pytest.raises(ValueError, match="shard 0 failed"):
        gen._run_shards(600, work)
    assert sorted(finished) == [200, 400]
    torch.cuda.synchronize()
    N.check_device("after a failed worker")


@pytest.mark.parametrize("mode", ["fp32", "tc", "fast"])
def test_real_devices_equal_per_shard_runs(lib, sphere, mode):
    devices = _real_devices(lib)
    cloud, seeds = sphere
    mfn, mfd = _models()
    _check_sharded_displace(mfn, mfd, devices, cloud, seeds, mode)


def test_real_devices_upsample_and_batch(lib, sphere):
    devices = _real_devices(lib)
    cloud, seeds = sphere
    mfn, mfd = _models()
    mfn.set_mode("tc"), mfd.set_mode("tc")
    single = Generator3D6(mfn, mfd, DEV, k_neighbors=100, remove_outliers=True)
    multi = Generator3D6(mfn, mfd, devices, k_neighbors=100, remove_outliers=True)
    bounds = shard_bounds(seeds.shape[0], len(devices))
    recon = np.concatenate([single.displace_host(cloud, seeds[lo:hi]) for lo, hi in bounds])
    assert np.array_equal(multi.upsample(np.expand_dims(cloud, 0), seeds=seeds), single._outlier_filter(recon))
    # a batch of three clouds of different sizes: the flat (cloud, seed) list is what gets sharded
    clouds = [syn.cloud(n, seed=40 + b, shape="boxes") for b, n in enumerate((2048, 1500, 3000))]
    sds = [syn.seeds(c, r, seed=50 + b) for b, (c, r) in enumerate(zip(clouds, (0.05, 0.02, 0.031)))]
    co = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    so = np.concatenate([[0], np.cumsum([s.shape[0] for s in sds])]).astype(np.int64)
    flat_c, flat_s = np.concatenate(clouds, 0), np.concatenate(sds, 0)
    bounds = shard_bounds(flat_s.shape[0], len(devices))
    recon = np.concatenate([single.displace_host(flat_c, flat_s[lo:hi], batch=(co, shard_batch_offsets(so, lo, hi)))
                            for lo, hi in bounds])
    multi.remove_outliers = False
    res = multi.upsample_batch(clouds, sds)
    for b in range(3):
        assert np.array_equal(res[b], recon[so[b]:so[b + 1]]), b


def test_data_parallel_over_the_shims(lib, sphere):
    import sapcu_oracle as orc
    import oracle_c
    from torch.nn.parallel.scatter_gather import scatter
    devices = _real_devices(lib)
    ids = list(range(len(devices)))
    cloud, seeds = sphere
    idx = oracle_c.knn(cloud, seeds[:64], 100)
    p = torch.from_numpy(orc.gather_center(cloud, seeds[:64], idx)).to(DEV)
    mfn, mfd = _models()
    mfn.set_mode("tc"), mfd.set_mode("tc")
    chunks = [c.to(DEV) for c in scatter(p, ids)]
    for m in (mfn, mfd):
        ref = torch.cat([m(c) for c in chunks]).clone()
        dp = torch.nn.DataParallel(m, device_ids=ids)
        assert torch.equal(dp(p), ref)
        handles = dict(m._handles)
        assert sorted(handles) == ids                      # one handle per device, all in the owner's cache
        assert torch.equal(dp(p), ref)
        assert m._handles == handles                       # reused by the next replicas, not rebuilt
        del dp
        assert torch.equal(torch.cat([m(c) for c in chunks]), ref)       # the owner's own handle survived its replicas
    torch.cuda.synchronize()
    for d in ids:
        with torch.cuda.device(d):
            N.check_device("DataParallel")


def test_device_guard_refuses_another_device(lib, sphere):
    devices = _real_devices(lib)
    mfn, mfd = _models()
    B = 8
    with torch.cuda.device(0):
        hfn, hfd = mfn._ensure_handle(torch.device(DEV)), mfd._ensure_handle(torch.device(DEV))
    d1 = torch.device(devices[1])
    p = torch.zeros(B, 100, 3, device=d1)
    n = torch.empty(B, 3, device=d1)
    d = torch.empty(B, device=d1)
    ws = torch.empty(lib.sapcu_model_workspace_bytes(hfd, B, 100), dtype=torch.uint8, device=d1)
    torch.cuda.synchronize(d1)
    with torch.cuda.device(d1):
        before = lib.sapcu_launch_count()
        st = N.stream_ptr(d1)
        assert lib.sapcu_fn_forward(hfn, N.ptr(p), B, 100, N.ptr(n), N.ptr(ws), ws.numel(), N.MODE_TC, st) == SAPCU_ESTATE
        msg = lib.sapcu_last_error().decode()
        assert "device 0" in msg and "device %d" % d1.index in msg, msg
        assert lib.sapcu_fd_forward(hfd, N.ptr(p), B, 100, N.ptr(d), None, N.ptr(ws), ws.numel(), N.MODE_TC, st) == SAPCU_ESTATE
        assert lib.sapcu_launch_count() == before
        # a handle finalized on device 1 is freed there while device 0 is current, and device 0 stays current
        mfn._ensure_handle(d1)
    with torch.cuda.device(0):
        del mfn
        import gc
        gc.collect()
        assert torch.cuda.current_device() == 0


def test_two_threads_one_module_two_streams(lib, sphere):
    import sapcu_oracle as orc
    import oracle_c
    cloud, seeds = sphere
    B = 48
    idx = oracle_c.knn(cloud, seeds[:B], 100)
    p = torch.from_numpy(orc.gather_center(cloud, seeds[:B], idx)).to(DEV)
    mfn, mfd = _models()
    mfn.set_mode("tc"), mfd.set_mode("tc")
    ref = (mfn(p).cpu().numpy(), mfd(p).cpu().numpy())
    outs, errs = [[], []], []

    def worker(i):
        try:
            torch.cuda.set_device(0)
            s = torch.cuda.Stream(device=DEV)
            with torch.cuda.stream(s):
                for _ in range(4):
                    n, d = mfn(p), mfd(p)
                    s.synchronize()
                    outs[i].append((n.cpu().numpy(), d.cpu().numpy()))
        except Exception as e:      # noqa: BLE001
            errs.append(e)
    ts = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    N.check_device("two threads, one module")
    for res in outs:
        assert len(res) == 4
        for n, d in res:
            assert np.array_equal(n, ref[0]) and np.array_equal(d, ref[1])
    # every stream got its own workspace on the device
    assert len({k for k in mfn._workspaces if k[0] == 0}) >= 3
