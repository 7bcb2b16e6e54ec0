"""The seed generator (csrc/seedgen.cu) against a serial restatement of the reference's flood fill (oracle_c.seedgen).

The oracle is the plain FIFO of dense.cpp: one pop at a time, a hash set of evaluated voxel ids (any int), an exact
grid-accelerated 10-NN ordered by (distance, index), point_tri in geom.cuh's operation order, and the "%lf" text round
trip for the 6-decimal coordinates.  It shares none of the device's level / keep-first claim / scan structure.

CPU part (any host): the oracle reproduces the reference binary's goldens bit for bit, and the 6-decimal rounding (the
text round trip, and the residual-corrected formula the device uses) agrees with float("%f") on every reachable voxel
centre, including the cells 1/320 and 1/960 where rounding c * 1e6 with nearbyint does not.
GPU part: full ordered float64 seed arrays and counts, np.array_equal, over cells, border aliasing, exact ties,
degenerate and tiny clouds, the largest frontier (chunked scan), the finest grid, capacity, streams and refusals.
"""
import ctypes
import functools
import hashlib
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
import oracle_c

DEV = "cuda:0"
SAPCU_EINVAL, SAPCU_EWORKSPACE = -1, -3
SCAN_TILE = 2048              # seedgen.cu: elements per scan tile; scan_sums_kernel runs one 1,024-tile chunk per pass
CELLS = [0.01, 0.008, 0.005, 0.0033, 0.0045, 0.003125, 1.0 / 960]
MODES = [(True, True), (True, False), (False, True), (False, False)]          # (quirk_origin, round6)


def _key(a):
    return hashlib.sha256(np.ascontiguousarray(a, np.float64).tobytes()).hexdigest()


_CLOUDS = {}


def _reg(cloud):
    cloud = np.ascontiguousarray(cloud, np.float64)
    k = _key(cloud)
    _CLOUDS[k] = cloud
    return k


@functools.lru_cache(maxsize=None)
def _oracle_k(k, cell, quirk, r6):
    return oracle_c.seedgen(_CLOUDS[k], cell, quirk_origin=quirk, round6=r6)


def oracle(cloud, cell, quirk=True, r6=True):
    return _oracle_k(_reg(cloud), cell, quirk, r6)


def _centres(cell):
    """every voxel-centre coordinate the fill can emit: index -k .. B + k (seedgen.cu seed_plan)"""
    B = int(round(1.0 / cell))
    k = int(math.ceil(0.015 / cell)) + 2
    x = np.arange(-k, B + k + 1, dtype=np.float64)
    return (x * cell + 0.5 * cell) - 0.5


def _round6_device(c):
    """seedgen.cu round6_text restated: nearbyint(c * 1e6) unless the product rounded onto a half-integer, where the
    sign of the exact residual (here a Fraction) decides."""
    p = c * 1e6
    m = np.rint(p)
    for i in np.nonzero(p - np.floor(p) == 0.5)[0]:
        r = Fraction(float(c[i])) * 10 ** 6 - Fraction(float(p[i]))
        if r != 0:
            m[i] = np.floor(p[i]) + (1.0 if r > 0 else 0.0)
    return m / 1e6


# ------------------------------------------------------------------------------------------------------ clouds
@functools.lru_cache(maxsize=None)
def shape_cloud(shape, cell):
    """syn.cloud shapes.  At cells below 0.008 the points of a dense sample within 800 cell^1.5 of a spot on the +x face
    (the sphere's pole, the cloud point nearest a corner of the boxes' long box): a band of ~60k voxels at any cell, so that the serial oracle
    stays well under a second"""
    if cell >= 0.008:
        return syn.cloud(512, seed=11, shape=shape)
    c = syn.cloud(100000, seed=11, shape=shape)
    spot = c[np.argmin(np.linalg.norm(c - ([0.5, 0.0, 0.0] if shape == "sphere" else [0.5, 0.2, 0.1]), axis=1))]
    return np.ascontiguousarray(c[np.linalg.norm(c - spot, axis=1) < 800 * cell ** 1.5])


def box_faces_cloud(cell, n=3000, seed=2):
    """points on all six faces of [-0.5, 0.5]^3, the 8 corners, and points on voxel boundaries k * cell - 0.5"""
    rng = np.random.default_rng(seed)
    p = rng.uniform(-0.5, 0.5, size=(n, 3))
    face = rng.integers(0, 6, size=n)
    p[np.arange(n), face % 3] = np.where(face < 3, -0.5, 0.5)
    corners = np.array([[sx, sy, sz] for sx in (-0.5, 0.5) for sy in (-0.5, 0.5) for sz in (-0.5, 0.5)])
    B = int(round(1.0 / cell))
    k = rng.integers(0, B + 1, size=(200, 2))
    on = np.stack([np.full(200, -0.5), k[:, 0] * cell - 0.5, k[:, 1] * cell - 0.5], 1)      # -x face, voxel-boundary y, z
    on2 = np.stack([k[:, 1] * cell - 0.5, np.full(200, 0.5), k[:, 0] * cell - 0.5], 1)      # +y face
    return np.clip(np.concatenate([p, corners, on, on2]), -0.5, 0.5)


def corner_cloud(cell, n=1500, seed=3, w=0.04):
    """three face patches meeting at the (-0.5, -0.5, -0.5) corner"""
    rng = np.random.default_rng(seed)
    p = rng.uniform(-0.5, -0.5 + w, size=(n, 3))
    p[np.arange(n), np.arange(n) % 3] = -0.5
    return p


def plus_x_patch(n=1500, seed=4, w=0.03):
    """a curved patch whose apex touches the +x face"""
    rng = np.random.default_rng(seed)
    yz = rng.uniform(-w, w, size=(n, 2))
    x = 0.5 - 2.0 * (yz ** 2).sum(1)
    return np.concatenate([[[0.5, 0.0, 0.0]], np.stack([x, yz[:, 0], yz[:, 1]], 1)])


def lattice_planar():
    """17 x 17 dyadic lattice in the plane z = 1/64: 10-NN distances tie exactly at the dyadic voxel centres"""
    g = np.arange(-8, 9) / 32.0
    x, y = np.meshgrid(g, g, indexing="ij")
    return np.stack([x.ravel(), y.ravel(), np.full(x.size, 1.0 / 64)], 1)


def lattice_cubic():
    """9^3 dyadic lattice that contains the origin, which ties with the reference's extra origin point (index N)"""
    g = np.arange(-4, 5) / 16.0
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)


# ------------------------------------------------------------------------------------------------------ CPU part
def test_oracle_reproduces_reference_binary(golden):
    """the serial restatement emits exactly what the compiled dense.cpp emitted (tests/golden/seeds.npz)"""
    g = golden.seeds
    cases = {"sphere256_c010": (syn.cloud(256, seed=5, shape="sphere"), 0.01),
             "boxes2048_c008": (syn.cloud(2048, seed=3, shape="boxes"), 0.008),
             "sphere2048_c004": (syn.cloud(2048, seed=0, shape="sphere"), 0.004)}
    for name, (cloud, cell) in cases.items():
        seeds, count, _ = oracle(cloud, cell)
        m = np.rint(seeds * 1e6).astype(np.int32)
        assert np.array_equal(m / 1e6, seeds), name                        # exactly the 6-decimal values
        assert count == seeds.shape[0] == int(g[name + "_count"]), name
        if name in g.files:
            assert np.array_equal(m, g[name]), name
        else:
            assert np.array_equal(m[:512], g[name + "_head"]) and np.array_equal(m[-512:], g[name + "_tail"]), name
        digest = np.frombuffer(hashlib.sha256(np.ascontiguousarray(m).tobytes()).digest(), dtype=np.uint8)
        assert np.array_equal(digest, g[name + "_sha256"]), name


@pytest.mark.parametrize("cell", [0.003125, 1.0 / 960, 0.01, 0.005, 0.004, 0.0025, 0.002, 0.001, 0.008, 0.0045, 0.0033])
def test_round6_matches_text_round_trip(cell):
    """the oracle's "%lf" + strtod and the device's residual-corrected formula both equal float("%f") on every
    reachable voxel centre; at 1/320 and 1/960 plain nearbyint(c * 1e6) / 1e6 does not"""
    c = _centres(cell)
    ref = np.array([float("%f" % v) for v in c])
    assert np.array_equal(oracle_c.round6_text(c), ref)
    assert np.array_equal(_round6_device(c), ref)
    naive = np.rint(c * 1e6) / 1e6
    if cell in (0.003125, 1.0 / 960):
        assert (naive != ref).sum() > 30
    else:
        assert np.array_equal(naive, ref)                  # centres with at most 6 decimals: no half to break


@pytest.mark.parametrize("shape", ["sphere", "boxes"])
@pytest.mark.parametrize("cell", [0.003125, 1.0 / 960])
def test_rounding_cells_emit_affected_coordinates(shape, cell):
    """the GPU cases at 1/320 and 1/960 emit seeds whose coordinates nearbyint(c * 1e6) would round wrongly"""
    raw, n_raw, _ = oracle(shape_cloud(shape, cell), cell, True, False)
    r6, n_r6, _ = oracle(shape_cloud(shape, cell), cell, True, True)
    assert n_raw == n_r6 > 0
    assert np.array_equal(oracle_c.round6_text(raw), r6)
    assert (np.rint(raw * 1e6) / 1e6 != r6).any(1).sum() > 0.01 * n_r6


def test_oracle_largest_frontier_reaches_chunked_scan():
    """the large case's statistics: some BFS level holds more than 1,024 scan tiles, and the level lengths chain
    (6 x expanding voxels of level L = queue entries of level L + 1)"""
    _, count, stats = oracle(*LARGEST)
    assert stats[:, 0].max() > 1024 * SCAN_TILE
    assert np.array_equal(stats[1:, 0], stats[:-1, 1]) and stats[-1, 1] == 0
    assert stats[0, 0] == LARGEST[0].shape[0] and count > 0


# ------------------------------------------------------------------------------------------------------ GPU part
LARGEST = (syn.cloud(8192, seed=0, shape="sphere"), 0.003)


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


def _run(lib, cloud, cell, quirk=True, r6=True, cap=None, stream=None, ws_bytes=None):
    """sapcu_seedgen through the C ABI -> (return code, seeds [min(count, cap)], count, untouched rows past them)"""
    cloud = np.ascontiguousarray(cloud, np.float64)
    n = cloud.shape[0]
    d_cloud = torch.from_numpy(cloud).to(DEV)
    cap = cap or 1 << 20
    out = torch.full((cap + 8, 3), float("nan"), dtype=torch.float64, device=DEV)       # 8 guard rows past the capacity
    need = lib.sapcu_seedgen_workspace_bytes(n, cell, cap)
    assert need > 0
    ws = torch.empty(need if ws_bytes is None else ws_bytes, dtype=torch.uint8, device=DEV)
    cnt = ctypes.c_int64(-1)
    rc = lib.sapcu_seedgen(N.ptr(d_cloud), n, cell, int(quirk), int(r6), N.ptr(out), cap, ctypes.byref(cnt), N.ptr(ws),
                           ws.numel(), None if stream is None else ctypes.c_void_p(stream.cuda_stream))
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    if rc:
        return rc, None, cnt.value, o
    k = min(cnt.value, cap)
    assert np.isnan(o[k:]).all(), "rows past the emitted seeds were written"
    return rc, o[:k], cnt.value, o


def _check(lib, cloud, cell, quirk=True, r6=True, what=""):
    ref, count, stats = oracle(cloud, cell, quirk, r6)
    rc, got, gcount, _ = _run(lib, cloud, cell, quirk, r6, cap=max(count, 1) + 16)
    assert rc == 0, N.lib().sapcu_last_error()
    assert gcount == count, "%s: %d seeds, oracle %d" % (what, gcount, count)
    if not np.array_equal(got, ref):
        bad = np.nonzero((got != ref).any(1))[0]
        raise AssertionError("%s: %d of %d seeds differ, first at %d: %r vs %r"
                             % (what, len(bad), count, bad[0], got[bad[0]], ref[bad[0]]))
    return ref, stats


@pytest.mark.gpu
@pytest.mark.parametrize("quirk,r6", MODES)
@pytest.mark.parametrize("cell", CELLS)
@pytest.mark.parametrize("shape", ["sphere", "boxes"])
def test_shapes_and_cells(lib, shape, cell, quirk, r6):
    _check(lib, shape_cloud(shape, cell), cell, quirk, r6, "%s cell=%r" % (shape, cell))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", [0.01, 0.005, 0.0045])
def test_border_aliasing(lib, cell):
    """a cloud on all six faces of the box: the band runs past x = B (ids above B^3), below x = 0 at the (-,-,-) corner
    (negative ids) and past y, z = B (ids that alias into the next x)"""
    ref, _ = _check(lib, box_faces_cloud(cell), cell, what="box faces cell=%r" % cell)
    assert ref[:, 0].max() > 0.5 + cell                                     # seeds beyond x = B
    if cell <= 0.005:
        assert (ref.min(0) < -0.5 - cell).all()                             # and beyond the corner, ids below -B^2
    else:
        _check(lib, box_faces_cloud(cell), cell, False, False, "box faces, no quirks, cell=%r" % cell)


@pytest.mark.gpu
@pytest.mark.parametrize("quirk,r6", MODES)
@pytest.mark.parametrize("cell", [1.0 / 128, 0.01])
@pytest.mark.parametrize("which", ["planar", "cubic"])
def test_exact_ties(lib, which, cell, quirk, r6):
    cloud = lattice_planar() if which == "planar" else lattice_cubic()
    assert which == "planar" or (cloud == 0).all(1).any()
    _check(lib, cloud, cell, quirk, r6, "%s lattice cell=%r" % (which, cell))


@pytest.mark.gpu
@pytest.mark.parametrize("quirk", [True, False])
def test_degenerate_clouds(lib, quirk):
    t = np.linspace(-0.4, 0.45, 300)
    collinear = np.stack([t, 0.5 * t + 0.01, -0.25 * t], 1)                # every triangle degenerate: NaN distances
    dup = np.tile([[0.1, -0.2, 0.3]], (40, 1))
    for name, cloud in (("collinear", collinear), ("duplicates", dup)):
        _check(lib, cloud, 0.01, quirk, True, name)
        _check(lib, cloud, 0.005, quirk, False, name)


@pytest.mark.gpu
@pytest.mark.parametrize("quirk", [True, False])
@pytest.mark.parametrize("n", [1, 2, 9, 10, 11])
def test_tiny_clouds(lib, n, quirk):
    """fewer than 10 search points leave neighbour slots empty (the origin stands in)"""
    rng = np.random.default_rng(n)
    v = rng.normal(size=(n, 3))
    cloud = 0.3 * v / np.linalg.norm(v, axis=1, keepdims=True)
    _check(lib, cloud, 0.01, quirk, True, "N=%d" % n)
    _check(lib, cloud, 0.005, quirk, False, "N=%d" % n)


@pytest.mark.gpu
def test_largest_frontier(lib):
    """a level above 1,024 scan tiles: scan_sums_kernel carries over more than one chunk"""
    _, stats = _check(lib, *LARGEST, what="sphere 8192 cell 0.003")
    assert stats[:, 0].max() > 1024 * SCAN_TILE


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["plus_x", "corner"])
def test_finest_grid(lib, where):
    """cell = 0.001 (the finest accepted grid): ids near 1.02e9 at the +x face, negative ids below x = 0 at the corner"""
    cloud = plus_x_patch() if where == "plus_x" else corner_cloud(0.001)
    ref, _ = _check(lib, cloud, 0.001, what=where)
    if where == "plus_x":
        assert ref[:, 0].max() > 0.51
    else:
        assert (ref.min(0) < -0.51).all()
    _check(lib, cloud, 0.001, False, False, where + " no quirks")


@pytest.mark.gpu
@pytest.mark.parametrize("cell", [0.005, 0.0025])
def test_corner_below_zero(lib, cell):
    """voxels two and more cells below x = 0 at the (-,-,-) corner: negative ids below -(B^2 + B + 1)"""
    ref, _ = _check(lib, corner_cloud(cell), cell, what="corner cell=%r" % cell)
    assert (ref.min(0) < -0.5 - 1.5 * cell).all()


@pytest.mark.gpu
def test_capacity_prefix(lib):
    cloud, cell = syn.cloud(256, seed=5, shape="sphere"), 0.01
    ref, count, _ = oracle(cloud, cell)
    for cap in (1, 7, count // 3, count - 1, count):
        rc, got, gcount, _ = _run(lib, cloud, cell, cap=cap)
        assert rc == 0 and gcount == count, cap
        assert np.array_equal(got, ref[:cap]), cap
        o_seeds, o_count, _ = oracle_c.seedgen(cloud, cell, cap=cap)
        assert o_count == count and np.array_equal(o_seeds, ref[:cap])


@pytest.mark.gpu
def test_second_stream_bitwise(lib):
    cloud, cell = syn.cloud(1024, seed=9, shape="boxes"), 0.005
    _, a, ca, _ = _run(lib, cloud, cell)
    s = torch.cuda.Stream()
    _, b, cb, _ = _run(lib, cloud, cell, stream=s)
    assert ca == cb and np.array_equal(a, b)
    ref, count, _ = oracle(cloud, cell)
    assert count == ca and np.array_equal(a, ref)


@pytest.mark.gpu
def test_refusals(lib):
    cloud = syn.cloud(64, seed=1, shape="sphere")
    d = torch.from_numpy(cloud).to(DEV)
    out = torch.zeros(1024, 3, dtype=torch.float64, device=DEV)
    cnt = ctypes.c_int64(-1)
    need = lib.sapcu_seedgen_workspace_bytes(64, 0.01, 1024)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    call = lambda n=64, cell=0.01, cap=1024, c=N.ptr(d), o=N.ptr(out), h=ctypes.byref(cnt), w=N.ptr(ws), wb=need: \
        lib.sapcu_seedgen(c, n, cell, 1, 1, o, cap, h, w, wb, None)
    before = lib.sapcu_launch_count()
    assert call(wb=need - 1) == SAPCU_EWORKSPACE
    assert lib.sapcu_launch_count() == before                             # refused before any launch
    assert call(cell=1.0 / 1000.5) == SAPCU_EINVAL
    assert call(n=0) == SAPCU_EINVAL
    assert call(cap=0) == SAPCU_EINVAL
    assert call(cell=0.0) == SAPCU_EINVAL and call(cell=-0.01) == SAPCU_EINVAL
    for kw in ({"c": None}, {"o": None}, {"h": None}, {"w": None}):
        assert call(**kw) == SAPCU_EINVAL, kw
    assert lib.sapcu_launch_count() == before
    # the workspace size is 0 exactly where the call refuses its sizes
    for n, cell, cap in ((0, 0.01, 1024), (1 << 30, 0.01, 1024), (64, 1.0 / 1000.5, 1024), (64, 0.0, 1024),
                         (64, -0.01, 1024), (64, 0.01, 0)):
        assert lib.sapcu_seedgen_workspace_bytes(n, cell, cap) == 0, (n, cell, cap)
    for n, cell, cap in ((1, 0.001, 1), (64, 0.01, 1), ((1 << 30) - 1, 0.5, 1)):
        assert lib.sapcu_seedgen_workspace_bytes(n, cell, cap) > 0, (n, cell, cap)
    assert call() == 0 and cnt.value > 0


@pytest.mark.gpu
def test_clouds_past_the_unit_box(lib):
    """coordinates beyond [-0.5 - cell, 0.5 + cell] are refused, naming the bound; within one cell they are served"""
    cell = 0.01
    base = syn.cloud(512, seed=6, shape="sphere")
    for name, cloud in (("scaled x1.1", base * 1.1), ("shifted 3 cells", base + [3 * cell, 0.0, 0.0]),
                        ("shifted -3 cells in z", base - [0.0, 0.0, 3 * cell]), ("NaN", np.where(np.arange(512)[:, None] == 77, np.nan, base))):
        rc, _, _, _ = _run(lib, cloud, cell)
        assert rc == SAPCU_EINVAL, name
        assert "0.51" in lib.sapcu_last_error().decode(), name
    for shift in ([0.5 * cell, 0.0, 0.0], [-0.9 * cell, -0.9 * cell, 0.9 * cell]):
        _check(lib, base + shift, cell, what="shift %r" % (shift,))
