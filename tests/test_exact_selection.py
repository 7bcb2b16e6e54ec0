"""GPU: the two selection kernels whose output is exact integers -- the seed kNN (csrc/knn_seed.cu) and farthest-point
sampling (csrc/post_ops.cu) -- on every launch path, against plain-C brute force (oracle/oracle_c.c), whole index arrays.

kNN: fp64 squared distance, ascending, ties to the lowest cloud index (oracle_c.knn).  The two flavours switch at
N = 2^20 (one warp per seed below, one thread per seed with TMA-staged tiles of 2,048 rows above); the cases sit at the
partial last tiles, the padding rows, exact ties, fp32-collapsed points, K = 1 / 30 / 128 (the metrics, the outlier
filter, the cap) and, in batched launches, clouds that start at rows not a multiple of 4.
FPS: fp32, `dist < distance`, first maximum (oracle_c.fps), compared over the full pick sequence from several starts,
across the one-CTA / spread-grid switch and the boundary where the cooperative grid needs two CTAs per SM.
Mean neighbour distance: numpy's own summation order, bit for bit.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
import oracle_c

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BIG = 1 << 20                 # smallest cloud on the thread-per-seed kNN flavour
EINVAL = -1


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


def _offset_ptr(t, off):
    return ctypes.c_void_p(t.data_ptr() + off)


def _knn(lib, cloud, seeds, K):
    dc, ds = torch.from_numpy(cloud).to(DEV), torch.from_numpy(np.ascontiguousarray(seeds)).to(DEV)
    idx = torch.full((seeds.shape[0], K), -1, dtype=torch.int32, device=DEV)
    ws = torch.empty(lib.sapcu_knn_workspace_bytes(cloud.shape[0]), dtype=torch.uint8, device=DEV)
    N.check(lib.sapcu_knn(N.ptr(dc), cloud.shape[0], N.ptr(ds), seeds.shape[0], K, N.ptr(idx), N.ptr(ws), ws.numel(), None))
    torch.cuda.synchronize()
    return idx.cpu().numpy()


def _knn_batched(lib, clouds, seeds, K):
    co = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    so = np.concatenate([[0], np.cumsum([s.shape[0] for s in seeds])]).astype(np.int64)
    dc = torch.from_numpy(np.concatenate(clouds, 0)).to(DEV)
    ds = torch.from_numpy(np.concatenate(seeds, 0)).to(DEV)
    idx = torch.full((int(so[-1]), K), -1, dtype=torch.int32, device=DEV)
    ws = torch.empty(lib.sapcu_knn_batched_workspace_bytes(int(co[-1]), len(clouds)), dtype=torch.uint8, device=DEV)
    N.check(lib.sapcu_knn_batched(N.ptr(dc), co.ctypes.data, N.ptr(ds), so.ctypes.data, len(clouds), K, N.ptr(idx), N.ptr(ws),
                                  ws.numel(), None), "knn_batched")
    torch.cuda.synchronize()
    return idx.cpu().numpy(), co, so


def _check_knn(lib, cloud, seeds, Ks, what):
    for K in Ks:
        got = _knn(lib, cloud, seeds, K)
        ref = oracle_c.knn(cloud, seeds, K)
        assert np.array_equal(got, ref), "%s K=%d: %d of %d seeds differ" % (what, K, int((got != ref).any(1).sum()), len(seeds))


def _collapsed_cluster(rng, nbase, spread):
    """nbase points near (1e3, -2e3, 5e2), each stored 16 times with offsets of m * 2^-40 |x| (m = 0..15) per coordinate:
    distinct in fp64, one value in fp32 -- the fp32 filter cannot separate them, only the exact fp64 pass can."""
    base = np.array([1000.0, -2000.0, 500.0]) + rng.normal(size=(nbase, 3)) * spread
    m = np.arange(16, dtype=np.float64)[None, :, None] * rng.choice([-1.0, 1.0], size=(1, 16, 3))
    cloud = (base[:, None, :] + m * np.abs(base[:, None, :]) * 2.0 ** -40).reshape(-1, 3)
    return cloud, base


# ----------------------------------------------------------------------------------------- kNN, one warp per seed
def test_knn_warp_flavour_partial_last_tile(lib):
    """N = 2^20 - 1: the largest cloud of the warp flavour, its last 1,024-row tile one row short."""
    rng = np.random.default_rng(101)
    cloud = rng.normal(size=(BIG - 1, 3))
    seeds = np.concatenate([rng.normal(size=(60, 3)), cloud[-7:] + 1e-9])       # seeds next to the last tile's rows too
    _check_knn(lib, cloud, seeds, (1, 128), "N=2^20-1")


def test_knn_warp_flavour_fp32_collapsed_cluster(lib):
    rng = np.random.default_rng(102)
    cloud, base = _collapsed_cluster(rng, 256, 1e-3)
    seeds = base[rng.integers(0, 256, size=40)] + rng.normal(size=(40, 3)) * 1e-4
    assert len(np.unique(cloud, axis=0)) == 4096 and len(np.unique(cloud.astype(np.float32), axis=0)) <= 256 + 16
    _check_knn(lib, cloud, seeds, (16, 100), "collapsed cluster")


# ----------------------------------------------------------------------------------------- kNN, one thread per seed
@pytest.fixture(scope="module")
def big_normal():
    """N = 2^20 + 3: the last 2,048-row tile holds 3 rows and one padding row."""
    rng = np.random.default_rng(103)
    return rng.normal(size=(BIG + 3, 3)), rng.normal(size=(300, 3))


def test_knn_thread_flavour_partial_tile_padding(lib, big_normal):
    cloud, seeds = big_normal
    seeds = seeds.copy()
    seeds[:4] = cloud[-4:] + 1e-7                         # the last rows (in the partial tile) are these seeds' nearest
    _check_knn(lib, cloud, seeds, (1, 30, 100, 128), "N=2^20+3")


def test_knn_thread_flavour_empty_and_single_seed(lib, big_normal):
    cloud, seeds = big_normal
    assert _knn(lib, cloud, seeds[:0], 8).shape == (0, 8)
    assert np.array_equal(_knn(lib, cloud, seeds[5:6], 8), oracle_c.knn(cloud, seeds[5:6], 8))


def test_knn_thread_flavour_tie_shells(lib):
    """Integer lattice 102 x 102 x 101 (1,050,804 points, last tile 180 rows) under a fixed row permutation, so index order
    is not spatial order.  Around a half-integer centre the shells hold 8, 24, 24, 32, 40 ... equidistant points and
    K = 100, 127 cut inside one; lattice-point seeds are cloud points themselves."""
    rng = np.random.default_rng(104)
    g = np.stack(np.meshgrid(np.arange(102), np.arange(102), np.arange(101), indexing="ij"), -1).reshape(-1, 3)
    cloud = np.ascontiguousarray(g[rng.permutation(len(g))].astype(np.float64))
    assert cloud.shape[0] == 1050804 and cloud.shape[0] % 2048 == 180
    centres = rng.integers(4, 96, size=(64, 3)) + 0.5
    points = rng.integers(0, 101, size=(64, 3)).astype(np.float64)
    points[:4] = [[0, 0, 0], [101, 101, 100], [0, 101, 50], [50, 50, 100]]      # corners and faces: truncated shells
    _check_knn(lib, cloud, np.concatenate([centres, points]), (100, 127, 128), "lattice")


def test_knn_thread_flavour_duplicates_self_query(lib):
    """262,145 distinct points stored 4 times, rows permuted (1,048,580 points), queried at cloud points themselves as the
    outlier filter and the normal orientation do: K = 1 answers the LOWEST-index copy, not the seed's own row."""
    rng = np.random.default_rng(105)
    base = rng.normal(size=(262145, 3))
    cloud = np.ascontiguousarray(np.tile(base, (4, 1))[rng.permutation(4 * 262145)])
    rows = rng.choice(cloud.shape[0], size=200, replace=False)
    seeds = cloud[rows]
    ref1 = oracle_c.knn(cloud, seeds, 1)
    assert (ref1[:, 0] != rows).sum() > 100                    # most seeds' own row is not their lowest-index copy
    assert np.array_equal(_knn(lib, cloud, seeds, 1), ref1)
    _check_knn(lib, cloud, seeds, (4, 30), "duplicates")


def test_knn_thread_flavour_far_from_origin_and_large_scale(lib):
    rng = np.random.default_rng(106)
    cloud, base = _collapsed_cluster(rng, BIG // 16, 1e-2)
    cloud = np.ascontiguousarray(cloud[rng.permutation(len(cloud))])
    assert cloud.shape[0] == BIG
    seeds = base[rng.integers(0, len(base), size=64)] + rng.normal(size=(64, 3)) * 1e-4
    _check_knn(lib, cloud, seeds, (100,), "collapsed cluster N=2^20")
    cloud = rng.normal(size=(BIG + 5, 3)) * 1e6
    _check_knn(lib, cloud, rng.normal(size=(64, 3)) * 1e6, (100,), "scale 1e6")


def test_knn_thread_flavour_seeds_far_outside(lib):
    rng = np.random.default_rng(107)
    v = rng.normal(size=(BIG + 1, 3))
    cloud = v / np.linalg.norm(v, axis=1, keepdims=True)
    u = rng.normal(size=(32, 3))
    _check_knn(lib, cloud, 1e4 * u / np.linalg.norm(u, axis=1, keepdims=True), (128,), "seeds at 1e4")


def test_knn_refusals(lib):
    """A workspace that is not 16-byte aligned (the cloud's fp32 copy is read with bulk copies) and K = 129 are refused
    with a code and a message, before any launch."""
    rng = np.random.default_rng(108)
    cloud = rng.normal(size=(5000, 3))
    dc = torch.from_numpy(cloud).to(DEV)
    idx = torch.empty(4, 129, dtype=torch.int32, device=DEV)
    nb = lib.sapcu_knn_workspace_bytes(5000)
    ws = torch.empty(nb + 64, dtype=torch.uint8, device=DEV)
    for off in (4, 8):
        assert lib.sapcu_knn(N.ptr(dc), 5000, N.ptr(dc), 4, 8, N.ptr(idx), _offset_ptr(ws, off), nb, None) == EINVAL
        assert b"16-byte aligned" in lib.sapcu_last_error()
    assert lib.sapcu_knn(N.ptr(dc), 5000, N.ptr(dc), 4, 129, N.ptr(idx), N.ptr(ws), nb, None) == EINVAL
    assert b"K=129" in lib.sapcu_last_error()
    co = np.array([0, 1000, 5000], dtype=np.int64); so = np.array([0, 2, 4], dtype=np.int64)
    nbb = lib.sapcu_knn_batched_workspace_bytes(5000, 2)
    wsb = torch.empty(nbb + 64, dtype=torch.uint8, device=DEV)
    assert lib.sapcu_knn_batched(N.ptr(dc), co.ctypes.data, N.ptr(dc), so.ctypes.data, 2, 8, N.ptr(idx), _offset_ptr(wsb, 4),
                                 nbb, None) == EINVAL
    assert b"16-byte aligned" in lib.sapcu_last_error()
    torch.cuda.synchronize()
    # the aligned workspace still works after the refusals
    assert np.array_equal(_knn(lib, cloud, cloud[:4], 8), oracle_c.knn(cloud, cloud[:4], 8))


# ----------------------------------------------------------------------------------------- batched kNN
def _batch_problem(rng, sizes, nseeds):
    """Overlapping clouds around the origin; each seed set starts with exact copies of the 3 rows before its cloud and the 4
    rows after it in the concatenated array, so a row read from a neighbouring cloud would be a distance-0 neighbour."""
    clouds = [rng.normal(size=(n, 3)) for n in sizes]
    seeds = []
    for b, s in enumerate(nseeds):
        sd = rng.normal(size=(s, 3))
        edge = ([clouds[b - 1][-3:]] if b > 0 else []) + ([clouds[b + 1][:4]] if b + 1 < len(clouds) else [])
        edge = np.concatenate(edge, 0)[:s] if edge else np.zeros((0, 3))
        sd[:len(edge)] = edge
        seeds.append(sd)
    return clouds, seeds


def _check_batched(lib, clouds, seeds, Ks):
    for K in Ks:
        idx, co, so = _knn_batched(lib, clouds, seeds, K)
        for b in range(len(clouds)):
            if seeds[b].shape[0] == 0:
                continue
            got = idx[so[b]:so[b + 1]]
            assert np.array_equal(got, _knn(lib, clouds[b], seeds[b], K) + int(co[b])), "cloud %d K=%d vs sapcu_knn" % (b, K)
            assert np.array_equal(got, oracle_c.knn(clouds[b], seeds[b], K) + int(co[b])), "cloud %d K=%d vs oracle" % (b, K)


def test_knn_batched_thread_flavour_unaligned_offsets(lib):
    """Clouds of >= 2^20 points put the whole batch on the thread-per-seed flavour; the clouds start at rows 1,001,
    1,049,578, 1,049,581 and 1,049,711 (= 1, 2, 1, 3 mod 4) of the concatenated array."""
    rng = np.random.default_rng(109)
    sizes = [1001, BIG + 1, 3, 130, BIG + 2]
    clouds, seeds = _batch_problem(rng, sizes, [37, 300, 0, 9, 50])
    co = np.cumsum([0] + sizes)
    assert [int(c) % 4 for c in co[1:5]] == [1, 2, 1, 3]
    _check_batched(lib, clouds, seeds, (1, 100, 128))


def test_knn_batched_warp_flavour_unaligned_offsets(lib):
    rng = np.random.default_rng(110)
    sizes = [1001, 5003, 3, 130, 70001]
    clouds, seeds = _batch_problem(rng, sizes, [37, 100, 0, 9, 50])
    assert [int(c) % 4 for c in np.cumsum([0] + sizes)[1:5]] == [1, 0, 3, 1]
    _check_batched(lib, clouds, seeds, (1, 100, 128))


def test_upsample_batch_with_large_cloud_equals_per_cloud(lib):
    """Generator3D6.upsample_batch on a 1,001-point cloud followed by a 1,048,581-point one (the second cloud starts at
    row 1,001: its kNN runs on the thread flavour from an unaligned row) returns per cloud exactly the points of
    upsample."""
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    from sapcu_b200.generation import Generator3D6
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    mfn, mfd = mfn.to(DEV), mfd.to(DEV)
    mfn.set_mode("tc"), mfd.set_mode("tc")
    gen = Generator3D6(mfn, mfd, DEV, k_neighbors=100, remove_outliers=False)
    clouds = [syn.cloud(1001, seed=60, shape="boxes"), syn.cloud(BIG + 5, seed=61, shape="sphere")]
    seeds = [syn.seeds(clouds[0], 0.2, seed=62), syn.seeds(clouds[1], 300.0 / (BIG + 5), seed=63)]
    res = gen.upsample_batch(clouds, seeds)
    for b, (c, s) in enumerate(zip(clouds, seeds)):
        single = gen.upsample(np.expand_dims(c, 0), seeds=s)
        assert res[b].shape == single.shape and np.array_equal(res[b], single), "cloud %d" % b


# ----------------------------------------------------------------------------------------- FPS
def _fps(lib, xyz32, npoint, start, ws_off=0):
    d = torch.from_numpy(xyz32).to(DEV)
    out = torch.full((max(npoint, 1),), -1, dtype=torch.int32, device=DEV)
    ws = torch.zeros(64, dtype=torch.uint8, device=DEV)
    rc = lib.sapcu_fps(N.ptr(d), xyz32.shape[0], npoint, start, N.ptr(out), _offset_ptr(ws, ws_off), 32, None)
    if rc != 0:
        return rc
    torch.cuda.synchronize()
    return out[:npoint].cpu().numpy().astype(np.int64)


def _check_fps(lib, xyz, npoint, starts=None, what=""):
    xyz32 = np.ascontiguousarray(xyz, np.float32)
    n = xyz32.shape[0]
    for start in (starts if starts is not None else sorted({0, n // 2, n - 1})):
        got = _fps(lib, xyz32, npoint, start)
        ref = oracle_c.fps(xyz32, npoint, start)
        assert not isinstance(got, int), "%s N=%d start=%d refused: %s" % (what, n, start, lib.sapcu_last_error())
        bad = np.flatnonzero(got != ref)
        assert bad.size == 0, "%s N=%d start=%d: first wrong pick at %d of %d" % (what, n, start, bad[0], npoint)
    return got


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def test_fps_small_and_around_the_spread_switch(lib):
    """N = 1; and N around 512, where the kernel switches from one CTA to one CTA per 512 points over the SMs."""
    assert np.array_equal(_check_fps(lib, np.zeros((1, 3)), 3, starts=(0,)), [0, 0, 0])
    _check_fps(lib, np.ones((1, 3)), 1, starts=(0,))
    rng = np.random.default_rng(111)
    for n in (2, 511, 512, 513, 4097):
        _check_fps(lib, rng.normal(size=(n, 3)), min(n, 300), what="normal")


def test_fps_exhaustion(lib):
    """npoint = N picks every point once; after that every running distance is 0 and the picks are index 0."""
    pts = np.random.default_rng(112).normal(size=(2000, 3))
    got = _check_fps(lib, pts, 2000, what="npoint=N")
    assert np.array_equal(np.sort(got), np.arange(2000))
    got = _check_fps(lib, pts, 2005, what="npoint=N+5")
    assert (got[2000:] == 0).all()


def test_fps_identical_points(lib):
    got = _check_fps(lib, np.full((1000, 3), 0.3), 50, what="identical")
    assert (got[1:] == 0).all()


def test_fps_grid_stored_twice(lib):
    """Every running distance is shared by at least two rows: each pick is a tie broken to the lowest index."""
    grid = np.stack(np.meshgrid(np.arange(12), np.arange(12), np.arange(12), indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    got = _check_fps(lib, np.concatenate([grid, grid], 0), 400, what="grid twice")
    assert (got[1:] < len(grid)).all()                      # after the start, always the first copy


def test_fps_far_from_origin(lib):
    _check_fps(lib, 1e4 + _unit(np.random.default_rng(117), 20000), 500, what="1e4 + sphere")


def _fps_capacity(lib):
    """Points the co-resident cooperative grid can hold, from the refusal of a size far beyond it."""
    tiny = torch.zeros(4, 3, dtype=torch.float32, device=DEV)
    out = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws = torch.zeros(32, dtype=torch.uint8, device=DEV)
    assert lib.sapcu_fps(N.ptr(tiny), 1 << 30, 4, 0, N.ptr(out), N.ptr(ws), 32, None) == EINVAL
    m = re.search(rb"co-resident capacity (\d+)", lib.sapcu_last_error())
    assert m, lib.sapcu_last_error()
    return int(m.group(1))


def test_fps_one_and_two_ctas_per_sm(lib):
    """N = SMs x 4,096 (606,208 on a 148-SM B200) fills one CTA per SM; one point more needs a 149th CTA, co-resident only
    with two CTAs per SM -- else it is refused."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cap = _fps_capacity(lib)
    assert cap >= sms * 4096 and cap % (sms * 4096) == 0
    rng = np.random.default_rng(113)
    pts = _unit(rng, sms * 4096 + 1)
    _check_fps(lib, pts[:-1], 1024, what="one CTA per SM")
    if cap > sms * 4096:
        _check_fps(lib, pts, 1024, what="%d CTAs" % (sms + 1))
    else:
        assert _fps(lib, np.ascontiguousarray(pts, np.float32), 1024, 0) == EINVAL
        assert b"co-resident capacity" in lib.sapcu_last_error()


def test_fps_real_use_full_sequence(lib):
    """generate.py's use: ~390,000 upsampled points down to 8,192, started at N // 2; every pick."""
    rng = np.random.default_rng(114)
    pts = 0.5 * _unit(rng, 390000)
    _check_fps(lib, pts, 8192, starts=(195000,), what="390k")


def test_fps_refusals(lib):
    pts = np.ascontiguousarray(np.random.default_rng(115).normal(size=(1000, 3)), np.float32)
    for off in (4, 12):
        assert _fps(lib, pts, 10, 0, ws_off=off) == EINVAL
        assert b"8-byte aligned" in lib.sapcu_last_error()
    assert np.array_equal(_fps(lib, pts, 10, 0, ws_off=8), oracle_c.fps(pts, 10, 0))        # 8-byte aligned is enough


# ----------------------------------------------------------------------------------------- mean neighbour distance
def test_knn_mean_dist_is_numpy_mean_bit_for_bit(lib):
    rng = np.random.default_rng(116)
    pts = rng.normal(size=(3000, 3)) * rng.uniform(0.1, 10, size=(3000, 1))
    q = np.concatenate([pts[:2000], rng.normal(size=(1000, 3))])
    d_p, d_q = torch.from_numpy(pts).to(DEV), torch.from_numpy(q).to(DEV)
    for K in (1, 5, 7, 8, 9, 16, 17, 30, 100, 127, 128):
        idx = oracle_c.knn(pts, q, K)
        d = pts[idx] - q[:, None, :]
        dist = np.ascontiguousarray(np.sqrt(((d[..., 0] * d[..., 0]) + (d[..., 1] * d[..., 1])) + (d[..., 2] * d[..., 2])))
        ref = np.mean(dist, axis=1)
        d_i = torch.from_numpy(idx).to(DEV)
        mean = torch.full((len(q),), np.nan, dtype=torch.float64, device=DEV)
        N.check(lib.sapcu_knn_mean_dist(N.ptr(d_p), 3000, N.ptr(d_q), len(q), N.ptr(d_i), K, N.ptr(mean), None))
        torch.cuda.synchronize()
        got = mean.cpu().numpy()
        assert np.array_equal(got, ref), "K=%d: %d rows differ" % (K, int((got != ref).sum()))


def test_mean_dist_entries_refuse_k_above_128(lib):
    pts = torch.zeros(200, 3, dtype=torch.float64, device=DEV)
    idx = torch.zeros(200, 129, dtype=torch.int32, device=DEV)
    mean = torch.empty(200, dtype=torch.float64, device=DEV)
    keep = torch.empty(200, dtype=torch.uint8, device=DEV)
    ws = torch.empty(lib.sapcu_outlier_workspace_bytes(200), dtype=torch.uint8, device=DEV)
    assert lib.sapcu_knn_mean_dist(N.ptr(pts), 200, N.ptr(pts), 200, N.ptr(idx), 129, N.ptr(mean), None) == EINVAL
    assert b"K=129" in lib.sapcu_last_error()
    assert lib.sapcu_outlier_mask(N.ptr(pts), 200, N.ptr(idx), 129, 1.5, N.ptr(keep), N.ptr(ws), ws.numel(), None) == EINVAL
    assert b"K=129" in lib.sapcu_last_error()
