"""fn's pair schedule (sapcu_fn_forward_indexed): pos evaluated once per distinct pair of cloud points.

On a dyadic cloud (points and seeds on multiples of 2^-12 inside [-1, 1]) the patch offsets fl32(x_i - s) - fl32(x_j - s) and
the pair offsets (float)(x_i - x_j) are the same exact numbers, so the indexed forward must equal the patch forward bit for
bit: everything past the offset (pair table, pair-row contractions, per-edge gamma epilogue, pid-indexed attention tail) is
then pinned.  The fp32 / tf32 / fast modes do not take the pair schedule and must match as well.  On a general cloud the offsets
differ by a few ulp of the patch coordinates; the normals through Generator3D6 must stay inside the parity threshold.
"""
import os

import numpy as np
import pytest
import torch

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
K = 100


def _knn_patches(cloud64, seeds64):
    L = N.lib()
    S = seeds64.shape[0]
    st = N.stream_ptr(torch.device(DEV))
    idx = torch.empty(S, K, dtype=torch.int32, device=DEV)
    kws = torch.empty(L.sapcu_knn_workspace_bytes(cloud64.shape[0]), dtype=torch.uint8, device=DEV)
    N.check(L.sapcu_knn(N.ptr(cloud64), cloud64.shape[0], N.ptr(seeds64), S, K, N.ptr(idx), N.ptr(kws), kws.numel(), st), "knn")
    p = torch.empty(S, K, 3, dtype=torch.float32, device=DEV)
    N.check(L.sapcu_gather_center_rotate(N.ptr(cloud64), cloud64.shape[0], N.ptr(seeds64), N.ptr(idx), S, K, None, N.ptr(p), st),
            "gather_center")
    return idx, p


@pytest.fixture(scope="module")
def fn_model():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    from sapcu_b200.fn import config as fc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    syn.init_weights(mfn, seed=100, stress=True)
    return mfn.to(DEV)


@pytest.fixture(scope="module")
def dyadic_problem():
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    q = lambda a: np.clip(np.round(a * 4096.0) / 4096.0, -1.0, 1.0)
    cloud = q(cloud)
    seeds = q(syn.seeds(cloud, 4, seed=1)[:1024])
    c64 = torch.from_numpy(np.ascontiguousarray(cloud, dtype=np.float64)).to(DEV)
    s64 = torch.from_numpy(np.ascontiguousarray(seeds, dtype=np.float64)).to(DEV)
    idx, p = _knn_patches(c64, s64)
    return c64, idx, p


@pytest.mark.parametrize("mode", ["tc", "fast", "fp32", "tf32"])
def test_indexed_equals_patch_forward_on_dyadic_cloud(fn_model, dyadic_problem, mode):
    c64, idx, p = dyadic_problem
    fn_model.set_mode(mode)
    a = fn_model(p)
    b = fn_model.forward_indexed(p, c64, idx)
    torch.cuda.synchronize()
    N.check_device("indexed forward")
    assert torch.equal(a, b), "max |diff| %g" % (a - b).abs().max().item()


def test_indexed_on_second_stream_and_strided_gidx(fn_model, dyadic_problem):
    c64, idx, p = dyadic_problem
    fn_model.set_mode("tc")
    ref = fn_model(p[:256])
    wide = torch.full((256, K + 7), -5, dtype=torch.int32, device=DEV)
    wide[:, :K] = idx[:256]
    s2 = torch.cuda.Stream()
    s2.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s2):
        out = fn_model.forward_indexed(p[:256], c64, wide[:, :K])
    s2.synchronize()
    N.check_device("indexed forward, second stream")
    assert torch.equal(ref, out)


def test_indexed_rejects_out_of_range_gidx(fn_model, dyadic_problem):
    c64, idx, p = dyadic_problem
    fn_model.set_mode("tc")
    bad = idx[:64].clone()
    bad[3, 7] = c64.shape[0] + 1000
    with pytest.raises(N.SapcuError):
        fn_model.forward_indexed(p[:64], c64, bad)
        torch.cuda.synchronize()
        N.check_device("indexed forward, bad gidx")
    torch.cuda.synchronize()
    N.check_device("after the rejected call")       # the flag was consumed: the device is usable again
    assert torch.equal(fn_model(p[:64]), fn_model.forward_indexed(p[:64], c64, idx[:64]))


class _PatchPath(torch.nn.Module):
    """The fn model behind a plain module: Generator3D6 then runs the per-edge (patch) schedule."""

    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, p):
        return self.m(p)


def _angles_deg(a, b):
    a = a.double() / a.double().norm(dim=1, keepdim=True).clamp_min(1e-30)
    b = b.double() / b.double().norm(dim=1, keepdim=True).clamp_min(1e-30)
    return torch.rad2deg(torch.acos((a * b).sum(1).clamp(-1, 1)))


def test_generator_close_to_patch_path_on_bench_cloud():
    """configs[1]'s cloud and 8,192 seeds in `tc`: normals and distances of the pair schedule against the patch schedule.
    The only difference is the offset (a few ulp of the patch coordinates), so the deviation is bounded by what the same
    model does when every patch coordinate moves by one ulp: that control is measured here too."""
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    from sapcu_b200.generation import Generator3D6
    torch.cuda.set_device(0)
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100), syn.init_weights(mfd, seed=200)
    mfn, mfd = mfn.to(DEV).set_mode("tc"), mfd.to(DEV).set_mode("tc")
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 4, seed=1)
    c64 = torch.from_numpy(np.ascontiguousarray(cloud, dtype=np.float64)).to(DEV)
    s64 = torch.from_numpy(np.ascontiguousarray(seeds, dtype=np.float64)).to(DEV)
    _, _, n_new, d_new = Generator3D6(mfn, mfd, DEV, k_neighbors=K, remove_outliers=False)._displace_local(c64, s64, return_parts=True)
    _, _, n_old, d_old = Generator3D6(_PatchPath(mfn), mfd, DEV, k_neighbors=K, remove_outliers=False)._displace_local(
        c64, s64, return_parts=True)
    _, p = _knn_patches(c64, s64)
    p_ulp = torch.nextafter(p, torch.zeros_like(p))              # every patch coordinate one ulp towards the seed
    ang_pair = _angles_deg(n_new, n_old)
    ang_ulp = _angles_deg(mfn(p_ulp), mfn(p))
    rel_d = ((d_new - d_old).abs().max() / d_old.abs().max()).item()
    worst = int(ang_pair.argmax())
    print("pair vs patch: max normal angle %.3g deg (seed %d), median %.3g deg, max rel distance %.3g; one-ulp control: max %.3g deg"
          % (ang_pair.max().item(), worst, ang_pair.median().item(), rel_d, ang_ulp.max().item()))
    assert ang_pair.max().item() <= 2.0 * ang_ulp.max().item() + 1e-4
    assert ang_pair.max().item() < 0.1 and rel_d < 1e-3          # the parity thresholds


# ---------------------------------------------------------------------------------------------------- the pair table itself
def _pair_table(graph, S, M, kmax, kk, gidx, cloud):
    import ctypes
    L = N.lib()
    kk_c = (ctypes.c_int * 3)(*kk)
    nb = L.sapcu_pair_table_workspace_bytes(S, M, kmax, kk_c, cloud.shape[0])
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    off = (ctypes.c_int64 * 7)()
    N.check(L.sapcu_pair_table(N.ptr(graph), S, M, kmax, kk_c, N.ptr(gidx), gidx.stride(0), N.ptr(cloud), cloud.shape[0],
                               N.ptr(ws), nb, off, N.stream_ptr(torch.device(DEV))), "pair_table")
    torch.cuda.synchronize()
    raw = ws.cpu().numpy()
    U = raw[off[6]: off[6] + 12].view(np.int32)
    out = []
    for b in range(3):
        pid = raw[off[b]: off[b] + S * M * kk[b] * 4].view(np.int32)
        delta = raw[off[3 + b]: off[3 + b] + int(U[b]) * 16].view(np.float32).reshape(-1, 4)
        out.append((int(U[b]), pid, delta))
    return out


@pytest.mark.parametrize("S,M,kmax,kk,disjoint", [
    (1, 50, 24, (24, 18, 12), False),
    (2, 128, 24, (24, 18, 12), False),
    (8192, 100, 24, (24, 18, 12), False),
    (4, 16, 16, (16, 16, 12), False),          # M < k: kk_b = M, kmax < 24
    (3, 50, 24, (24, 18, 12), True),           # patches that share no points
])
def test_pair_table_matches_numpy_unique(S, M, kmax, kk, disjoint):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    rng = np.random.default_rng(S * 1000 + M)
    Ncl = S * M if disjoint else 2048
    cloud = rng.standard_normal((Ncl, 3))
    gidx = np.arange(S * M, dtype=np.int32).reshape(S, M) if disjoint else \
        np.stack([rng.choice(Ncl, M, replace=False) for _ in range(S)]).astype(np.int32)
    # patch-local graph: self first, then kmax - 1 distinct other points (as intra_knn's top-k lists)
    graph = np.empty((S * M, kmax), np.int32)
    for pt in range(S * M):
        i = pt % M
        others = rng.permutation(M - 1)[: kmax - 1]
        graph[pt, 0] = i
        graph[pt, 1:] = np.where(others >= i, others + 1, others)
    g_dev = torch.from_numpy(graph).to(DEV)
    gi_dev = torch.from_numpy(gidx).to(DEV)
    c_dev = torch.from_numpy(np.ascontiguousarray(cloud)).to(DEV)
    tables = _pair_table(g_dev, S, M, kmax, kk, gi_dev, c_dev)
    s_of = np.repeat(np.arange(S), M)
    gi_pt = gidx.reshape(-1)                                                    # cloud row of each patch point
    for b, (U, pid, delta) in enumerate(tables):
        k = kk[b]
        nbr = graph[:, :k]
        gi = np.repeat(gi_pt, k)
        gj = gidx[np.repeat(s_of, k), nbr.reshape(-1)]
        key = gi.astype(np.int64) * Ncl + gj
        uniq, inv = np.unique(key, return_inverse=True)
        assert U == uniq.size
        np.testing.assert_array_equal(pid, inv.reshape(-1))                  # pair rows numbered in key order: one row per pair
        ui, uj = uniq // Ncl, uniq % Ncl
        want = (cloud[ui] - cloud[uj]).astype(np.float32)
        np.testing.assert_array_equal(delta[:, :3], want)
