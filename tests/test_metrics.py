"""Evaluation metrics: sapcu_mesh_distance against a numpy restatement of its contract, and the sapcu_b200.metrics API.

The restatement (face_dist2_ref) is a vectorised copy of the device's per-face distance (csrc/geom.cuh point_tri, the
segment fallback and the box clamp of csrc/mesh_dist.cu): every branch is computed, the first true one is selected with
np.where, in the device's operation order (numpy rounds every operation and never contracts, like the -fmad=false build).
A brute-force argmin over (D, face index) over all faces is then the reference of the LBVH query, bit for bit.
"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
from sapcu_b200 import metrics as M

DEV = "cuda:0"
SAPCU_EINVAL, SAPCU_EWORKSPACE = -1, -3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------------------- the restatement
def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)


def _d2(p, q):
    d = p - q
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def point_tri_ref(a, b, c, p):
    """geom.cuh point_tri, broadcast over leading axes ([..., 3] each)."""
    with np.errstate(all="ignore"):
        ab, ac, bc = b - a, c - a, c - b
        snom, sdenom = _dot(p - a, ab), _dot(p - b, a - b)
        tnom, tdenom = _dot(p - a, ac), _dot(p - c, a - c)
        unom, udenom = _dot(p - b, bc), _dot(p - c, b - c)
        n = _cross(b - a, c - a)
        vc = _dot(n, _cross(a - p, b - p))
        va = _dot(n, _cross(b - p, c - p))
        vb = _dot(n, _cross(c - p, a - p))
        e_ab = a + (ab * snom[..., None]) / (snom + sdenom)[..., None]
        e_bc = b + (bc * unom[..., None]) / (unom + udenom)[..., None]
        e_ac = a + (ac * tnom[..., None]) / (tnom + tdenom)[..., None]
        u = va / ((va + vb) + vc)
        v = vb / ((va + vb) + vc)
        w = (1.0 - u) - v
        bary = (a * u[..., None] + b * v[..., None]) + c * w[..., None]
    conds = [(snom <= 0) & (tnom <= 0), (sdenom <= 0) & (unom <= 0), (tdenom <= 0) & (udenom <= 0),
             (vc <= 0) & (snom >= 0) & (sdenom >= 0), (va <= 0) & (unom >= 0) & (udenom >= 0),
             (vb <= 0) & (tnom >= 0) & (tdenom >= 0)]
    vals = [a, b, c, e_ab, e_bc, e_ac]
    out = bary
    for cnd, val in zip(conds[::-1], vals[::-1]):
        out = np.where(cnd[..., None], np.broadcast_to(val, out.shape), out)
    return out


def _seg_ref(a, b, p):
    with np.errstate(all="ignore"):
        e = b - a
        ee = _dot(e, e)
        t = np.where(ee > 0, _dot(p - a, e) / np.where(ee > 0, ee, 1.0), 0.0)
    t = np.where(t < 0, 0.0, np.where(t > 1, 1.0, t))
    return a + e * t[..., None]


def face_dist2_ref(a, b, c, p):
    """D(p, f) of include/sapcu_b200.h, broadcast over leading axes."""
    q = point_tri_ref(a, b, c, p)
    bad = ~np.isfinite(q).all(-1)
    if bad.any():
        q1, q2, q3 = _seg_ref(a, b, p), _seg_ref(b, c, p), _seg_ref(c, a, p)
        d1, d2 = _d2(p, q1), _d2(p, q2)
        qs = np.where((d2 < d1)[..., None], q2, q1)
        ds = np.where(d2 < d1, d2, d1)
        qs = np.where((_d2(p, q3) < ds)[..., None], q3, qs)
        q = np.where(bad[..., None], qs, q)
    lo = np.fmin(np.fmin(a, b), c)
    hi = np.fmax(np.fmax(a, b), c)
    q = np.fmin(np.fmax(q, lo), hi)
    return _d2(p, q)


def mesh_distance_ref(vertices, faces, points, chunk_pairs=1 << 19):
    """Brute force: (min D [S] f64, lowest face index attaining it [S] int32) over the faces with indices in [0, V)."""
    v = np.asarray(vertices, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    ok = ((f >= 0) & (f < len(v))).all(1)
    fi = np.flatnonzero(ok)
    S = len(p)
    best, face = np.full(S, np.inf), np.full(S, -1, np.int32)
    if len(fi) == 0 or S == 0:
        return best, face
    a, b, c = (v[f[fi, k]][None] for k in range(3))
    step = max(1, chunk_pairs // len(fi))
    for s0 in range(0, S, step):
        D = face_dist2_ref(a, b, c, p[s0:s0 + step, None, :])
        j = np.argmin(D, axis=1)                              # first occurrence: the lowest face index among equal D
        best[s0:s0 + step] = D[np.arange(len(j)), j]
        face[s0:s0 + step] = fi[j]
    return best, face


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


# ----------------------------------------------------------------------------------------- CPU: restatement, reader, formulas
def test_restatement_analytic_distances():
    a, b, c = np.array([0.0, 0, 0]), np.array([1.0, 0, 0]), np.array([0.0, 1, 0])
    cases = [((0.25, 0.25, 2.0), 4.0),            # above the interior
             ((0.5, -1.0, 0.0), 1.0),             # beyond edge ab
             ((1.0, 1.0, 0.0), 0.5),              # beyond edge bc (closest point (0.5, 0.5, 0))
             ((-3.0, -4.0, 0.0), 25.0),           # beyond vertex a
             ((2.0, 0.0, 1.0), 2.0),              # beyond vertex b
             ((0.25, 0.5, 0.0), 0.0)]             # on the face
    for p, d2 in cases:
        assert face_dist2_ref(a, b, c, np.array(p)) == d2, p


@pytest.mark.parametrize("tri", ["collinear", "ab_coincident", "bc_coincident", "ca_coincident", "all_coincident"])
def test_restatement_degenerate_faces_no_nan(tri):
    rng = np.random.default_rng(1)
    x, y = np.array([0.1, 0.2, 0.3]), np.array([0.7, -0.4, 0.9])
    a, b, c = {"collinear": (x, (x + y) / 2, y), "ab_coincident": (x, x, y), "bc_coincident": (y, x, x),
               "ca_coincident": (x, y, x), "all_coincident": (x, x, x)}[tri]
    p = rng.normal(size=(4000, 3)) * 2.0
    p[:8] = [x, y, (x + y) / 2, 2 * y - x, 2 * x - y, x + [0, 0, 1], y + [1, 0, 0], (x + y) / 2 + [0, 1, 0]]
    D = face_dist2_ref(a, b, c, p)
    assert np.isfinite(D).all()
    # the exact distance to the segment [x, y] (or to the point x) -- the degenerate face's point set
    e = y - x if tri != "all_coincident" else np.zeros(3)
    t = np.clip(((p - x) @ e) / max(e @ e, 1e-300), 0, 1)
    exact = ((p - (x + t[:, None] * e)) ** 2).sum(1)
    np.testing.assert_allclose(D, exact, rtol=1e-12, atol=1e-15)
    if tri == "ab_coincident":             # the routine's own 0/0 is reached here, and replaced by the fallback
        assert not np.isfinite(point_tri_ref(a, b, c, p)).all()


def test_restatement_matches_dense_distance_on_a_sphere():
    v, f = syn.sphere_mesh(2)
    rng = np.random.default_rng(2)
    p = rng.normal(size=(300, 3))
    p *= (0.3 + 0.4 * rng.random((300, 1))) / np.linalg.norm(p, axis=1, keepdims=True)
    d2, face = mesh_distance_ref(v, f, p)
    a, b, c = v[f[face, 0]], v[f[face, 1]], v[f[face, 2]]
    n = np.cross(b - a, c - a)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    plane = ((p - a) * n).sum(1) ** 2
    assert (d2 >= plane - 1e-15).all() and np.allclose(np.sqrt(d2), np.abs(np.linalg.norm(p, axis=1) - 0.5), atol=2e-2)


def _write_off(path, v, f, header="OFF\n"):
    with open(path, "w") as fh:
        fh.write(header)
        fh.write("%d %d 0\n" % (len(v), len(f)))
        for r in v:
            fh.write("%.17g %.17g %.17g\n" % tuple(r))
        for r in f:
            fh.write("3 %d %d %d\n" % tuple(r))


def test_read_off_round_trip_and_rejections(tmp_path):
    v, f = syn.sphere_mesh(1)
    _write_off(tmp_path / "s.off", v, f, header="# comment\nOFF\n")
    rv, rf = M.read_off(str(tmp_path / "s.off"))
    assert rf.dtype == np.int32 and np.array_equal(rv, v) and np.array_equal(rf, f)
    (tmp_path / "inline.off").write_text("OFF 3 1 0\n0 0 0\n1 0 0\n0 1 0 # c\n3 0 1 2 255 0 0\n")
    rv, rf = M.read_off(str(tmp_path / "inline.off"))
    assert rv.shape == (3, 3) and rf.tolist() == [[0, 1, 2]]
    bad = {"quad.off": "OFF\n4 1 0\n0 0 0\n1 0 0\n1 1 0\n0 1 0\n4 0 1 2 3\n",
           "range.off": "OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 3\n",
           "negative.off": "OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 -1 1 2\n",
           "short.off": "OFF\n3 2 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n",
           "long.off": "OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n3 0 1 2\n",
           "header.off": "PLY\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n",
           "counts.off": "OFF\nthree 1 0\n",
           "coords.off": "OFF\n3 1 0\n0 0\n1 0 0\n0 1 0\n3 0 1 2\n"}
    for name, text in bad.items():
        (tmp_path / name).write_text(text)
        with pytest.raises(ValueError):
            M.read_off(str(tmp_path / name))


def test_metric_formulas_hand_computed():
    # pred {0, 3} x {0}, gt {1, 2, 10} on the x axis: d_pg = (1, 1), d_gp = (1, 1, 7)
    pg2 = torch.tensor([1.0, 1.0], dtype=torch.float64)
    gp2 = torch.tensor([1.0, 1.0, 49.0], dtype=torch.float64)
    r = M.cd_hd_from_dist2(pg2, gp2)
    assert r["cd"] == pytest.approx(1.0 + 3.0, rel=1e-15)
    assert r["cd_sq"] == pytest.approx(1.0 + 17.0, rel=1e-15)
    assert r["hd"] == 7.0
    s = M.normal_stats(np.array([[0, 0, 2.0], [0, 0, -1.0], [1.0, 0, 1.0], [0, 0, 0]]), np.array([[0, 0, 3.0]] * 4))
    assert s["flipped"] == 0.25 and s["angle_max"] == 90.0
    assert s["angle_median"] == pytest.approx(22.5) and s["angle_mean"] == pytest.approx(135.0 / 4)
    c, r = M.unit_ball(np.array([[0.0, 0, 0], [2.0, 0, 0], [1.0, 3.0, 0]]))
    assert np.allclose(c, [1.0, 1.0, 0.0]) and r == pytest.approx(2.0)


def test_workspace_bytes_limits():
    L = N.lib()
    for V, F in ((0, 10), (10, 0), (10, -1), (10, 1 << 31), (-5, 5)):
        assert L.sapcu_mesh_distance_workspace_bytes(V, F) == 0
    small, big = L.sapcu_mesh_distance_workspace_bytes(3, 1), L.sapcu_mesh_distance_workspace_bytes(3, (1 << 31) - 1)
    assert 0 < small < big and big < 300 * (1 << 31)
    assert L.sapcu_mesh_distance_workspace_bytes(1, 1000) == L.sapcu_mesh_distance_workspace_bytes(10 ** 6, 1000)


def test_sphere_mesh_closed_and_outward():
    for level in (0, 1, 3):
        v, f = syn.sphere_mesh(level)
        assert f.dtype == np.int32 and len(f) == 20 * 4 ** level
        np.testing.assert_allclose(np.linalg.norm(v, axis=1), 0.5, rtol=1e-15)
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).astype(np.int64)
        # closed and consistently wound: every directed edge appears once and its reverse once
        fwd = e[:, 0] * len(v) + e[:, 1]
        assert len(np.unique(fwd)) == len(fwd) and np.array_equal(np.sort(fwd), np.sort(e[:, 1] * len(v) + e[:, 0]))
        a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
        assert ((np.cross(b - a, c - a) * (a + b + c)).sum(1) > 0).all()
        assert len(v) - len(fwd) // 2 + len(f) == 2


# ----------------------------------------------------------------------------------------- GPU: the operator
@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


def _gpu(v, f, p, stream=None, ws_bytes=None):
    L = N.lib()
    d_v = torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64).reshape(-1, 3)).to(DEV)
    d_f = torch.from_numpy(np.ascontiguousarray(f, dtype=np.int32).reshape(-1, 3)).to(DEV)
    d_p = torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 3)).to(DEV)
    S = d_p.shape[0]
    d2 = torch.full((S,), -1.0, dtype=torch.float64, device=DEV)
    face = torch.full((S,), -7, dtype=torch.int32, device=DEV)
    ws = torch.empty(L.sapcu_mesh_distance_workspace_bytes(d_v.shape[0], d_f.shape[0]), dtype=torch.uint8, device=DEV)
    st = stream or torch.cuda.current_stream(DEV)
    st.wait_stream(torch.cuda.current_stream(DEV))
    N.check(L.sapcu_mesh_distance(N.ptr(d_v), d_v.shape[0], N.ptr(d_f), d_f.shape[0], N.ptr(d_p), S, N.ptr(d2), N.ptr(face),
                                  N.ptr(ws), ws.numel() if ws_bytes is None else ws_bytes, ctypes.c_void_p(st.cuda_stream)),
            "sapcu_mesh_distance")
    st.synchronize()
    return d2.cpu().numpy(), face.cpu().numpy()


def _check(v, f, p):
    got, gface = _gpu(v, f, p)
    ref, rface = mesh_distance_ref(v, f, p)
    assert np.array_equal(_bits(got), _bits(ref)), np.flatnonzero(_bits(got) != _bits(ref))[:10]
    assert np.array_equal(gface, rface)
    return got, gface


def _shell(n, rng, r_lo, r_hi, centre=(0.0, 0.0, 0.0)):
    p = rng.normal(size=(n, 3))
    p *= (r_lo + (r_hi - r_lo) * rng.random((n, 1))) / np.linalg.norm(p, axis=1, keepdims=True)
    return p + np.asarray(centre)


@pytest.mark.gpu
def test_random_triangle_soup(lib):
    rng = np.random.default_rng(10)
    F = 3000
    v = rng.random((3 * F, 3))
    f = rng.permutation(3 * F).reshape(F, 3)
    p = rng.random((2000, 3)) * 1.6 - 0.3
    _check(v, f, p)
    small = v[f[:, :1]] + 0.02 * rng.normal(size=(F, 3, 3))             # small scattered triangles
    _check(small.reshape(-1, 3), np.arange(3 * F).reshape(F, 3), p)


@pytest.mark.gpu
def test_icosphere_near_on_far(lib):
    rng = np.random.default_rng(11)
    v, f = syn.sphere_mesh(3)
    near = _shell(3000, rng, 0.49, 0.51)
    far = np.concatenate([_shell(500, rng, 2.0, 50.0), _shell(300, rng, 0.0, 0.1)])
    on = v[f[:, 0]] * 0.2 + v[f[:, 1]] * 0.3 + v[f[:, 2]] * 0.5        # on the faces (up to rounding)
    d2, _ = _check(v, f, np.concatenate([near, far, on]))
    assert (d2[-len(on):] < 1e-28).all()


@pytest.mark.gpu
def test_points_at_vertices_and_on_shared_edges(lib):
    v, f = syn.sphere_mesh(2)
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    mids = (v[e[:, 0]] + v[e[:, 1]]) / 2
    quarter = v[e[:, 0]] * 0.75 + v[e[:, 1]] * 0.25
    d2, face = _check(v, f, np.concatenate([v, mids, quarter]))
    assert (d2[:len(v)] == 0).all()


@pytest.mark.gpu
def test_duplicated_and_coplanar_overlapping_faces(lib):
    rng = np.random.default_rng(12)
    v, f = syn.sphere_mesh(2)
    rot = f[:, [1, 2, 0]]                                              # the same faces, rotated vertex order
    dup = np.concatenate([f, rot[::-1], f])
    p = np.concatenate([_shell(2000, rng, 0.45, 0.55), v])
    _, face = _check(v, dup, p)
    assert (face < 2 * len(f)).all()                                   # an exact copy with a higher index never wins
    # coplanar overlapping triangles in the plane z = 0: one big, shifted copies, and sub-triangles
    pv = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0.5, 0, 0], [0, 0.5, 0], [0.5, 0.5, 0], [0.25, 0.25, 0],
                   [1.25, 0.25, 0], [0.25, 1.25, 0]], dtype=np.float64)
    pf = np.array([[6, 7, 8], [0, 1, 2], [3, 5, 4], [0, 3, 4], [2, 0, 1], [4, 5, 2]])
    q = np.concatenate([rng.random((2000, 3)) * [1.5, 1.5, 0.0] - 0.2, rng.random((1000, 3)) * [1.5, 1.5, 0.2] - 0.2])
    _check(pv, pf, q)


@pytest.mark.gpu
def test_degenerate_faces(lib):
    rng = np.random.default_rng(13)
    v, f = syn.sphere_mesh(2)
    x, y, z = v[f[:50, 0]], v[f[:50, 1]], v[f[:50, 2]]
    extra_v = np.concatenate([x, y, (x + y) / 2, z])
    n = 50
    ix, iy, im, iz = (len(v) + k * n + np.arange(n) for k in range(4))
    extra_f = np.concatenate([np.stack(t, 1) for t in ((ix, im, iy), (ix, ix, iz), (iz, ix, ix), (ix, iz, ix), (iz, iz, iz),
                                                       (iy, ix, im))])
    vv = np.concatenate([v, extra_v])
    ff = np.concatenate([extra_f, f])
    p = np.concatenate([_shell(2000, rng, 0.4, 0.6), extra_v, (extra_v[:n] + extra_v[3 * n:]) / 2])
    d2, _ = _check(vv, ff, p)
    assert np.isfinite(d2).all()
    _check(vv, extra_f, p)                                             # a mesh of degenerate faces only


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["F1", "S1", "S0"])
def test_extreme_sizes(lib, case):
    rng = np.random.default_rng(14)
    v, f = syn.sphere_mesh(1)
    if case == "F1":
        _check(v, f[:1], _shell(1000, rng, 0.0, 2.0))
        _check(v, f[:1], v[f[:1]].reshape(-1, 3))
    elif case == "S1":
        _check(v, f, np.array([[0.1, 0.2, 0.7]]))
    else:
        got, face = _gpu(v, f, np.zeros((0, 3)))
        assert got.shape == (0,) and face.shape == (0,)


@pytest.mark.gpu
def test_far_from_origin_millimetre_triangles(lib):
    rng = np.random.default_rng(15)
    v, f = syn.sphere_mesh(5)                                          # edges ~0.02 at radius 0.5
    centre = np.array([1234.5678, -987.654, 1000.125])
    v = v * 0.05 + centre                                             # ~1 mm triangles around 10^3
    p = np.concatenate([_shell(1500, rng, 0.0249, 0.0251, centre), _shell(200, rng, 0.0, 0.1, centre),
                        v[f[:300]].mean(axis=1)])
    _check(v, f, p)


@pytest.mark.gpu
def test_deep_tree(lib):
    rng = np.random.default_rng(16)
    v, f = syn.sphere_mesh(7)                                          # 327,680 faces
    assert len(f) >= 1 << 18
    p = np.concatenate([_shell(250, rng, 0.499, 0.501), _shell(50, rng, 0.0, 2.0)])
    _check(v, f, p)


@pytest.mark.gpu
def test_query_order_repeat_and_second_stream(lib):
    rng = np.random.default_rng(17)
    v, f = syn.sphere_mesh(4)
    p = _shell(20000, rng, 0.45, 0.55)
    d2, face = _gpu(v, f, p)
    perm = rng.permutation(len(p))
    d2p, facep = _gpu(v, f, p[perm])
    assert np.array_equal(_bits(d2p), _bits(d2[perm])) and np.array_equal(facep, face[perm])
    again = _gpu(v, f, p)
    assert np.array_equal(_bits(again[0]), _bits(d2)) and np.array_equal(again[1], face)
    side = torch.cuda.Stream(device=DEV)
    other = _gpu(v, f, p, stream=side)
    assert np.array_equal(_bits(other[0]), _bits(d2)) and np.array_equal(other[1], face)
    # the call does not synchronise: it returns while a long kernel queued before it still runs on its stream
    L = N.lib()
    d_v = torch.from_numpy(v).to(DEV)
    d_f = torch.from_numpy(f).to(DEV)
    d_p = torch.from_numpy(p).to(DEV)
    out = torch.empty(len(p), dtype=torch.float64, device=DEV)
    ws = torch.empty(L.sapcu_mesh_distance_workspace_bytes(len(v), len(f)), dtype=torch.uint8, device=DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        N.check(L.sapcu_mesh_distance(N.ptr(d_v), len(v), N.ptr(d_f), len(f), N.ptr(d_p), len(p), N.ptr(out), None, N.ptr(ws),
                                      ws.numel(), ctypes.c_void_p(side.cuda_stream)))
        busy = not side.query()
    side.synchronize()
    assert busy
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(d2))


@pytest.mark.gpu
def test_out_of_range_faces_are_skipped(lib):
    rng = np.random.default_rng(18)
    v, f = syn.sphere_mesh(2)
    bad = f.astype(np.int64).copy()
    sel = rng.random(len(f)) < 0.3
    bad[sel, rng.integers(0, 3, sel.sum())] = rng.choice(np.array([-1, len(v), 2 ** 31 - 1, -2 ** 31]), sel.sum())
    p = _shell(2000, rng, 0.3, 0.7)
    d2, face = _check(v, bad, p)
    assert not sel[face].any()
    d2, face = _gpu(v, np.full((5, 3), -1), p[:10])                    # no valid face at all
    assert np.isinf(d2).all() and (face == -1).all()


@pytest.mark.gpu
def test_error_codes(lib):
    L = N.lib()
    v = torch.zeros(3, 3, dtype=torch.float64, device=DEV)
    f = torch.tensor([[0, 1, 2]], dtype=torch.int32, device=DEV)
    p = torch.zeros(4, 3, dtype=torch.float64, device=DEV)
    d2 = torch.full((4,), 5.0, dtype=torch.float64, device=DEV)
    need = L.sapcu_mesh_distance_workspace_bytes(3, 1)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    st = N.stream_ptr(DEV)
    before = L.sapcu_launch_count()
    for V, F, S in ((0, 1, 4), (3, 0, 4), (3, 1, -1), (3, 1 << 31, 4)):
        assert L.sapcu_mesh_distance(N.ptr(v), V, N.ptr(f), F, N.ptr(p), S, N.ptr(d2), None, N.ptr(ws), need, st) == SAPCU_EINVAL
    assert L.sapcu_mesh_distance(N.ptr(v), 3, N.ptr(f), 1, N.ptr(p), 4, N.ptr(d2), None, N.ptr(ws), need - 1, st) == SAPCU_EWORKSPACE
    assert L.sapcu_mesh_distance(N.ptr(v), 3, N.ptr(f), 1, None, 0, None, None, None, 0, st) == 0
    assert L.sapcu_launch_count() == before
    assert (d2 == 5.0).all()


# ----------------------------------------------------------------------------------------- GPU: the Python API
def _nn_ref(a, b):
    out = np.empty(len(a))
    for s0 in range(0, len(a), 256):
        d = a[s0:s0 + 256, None, :] - b[None]
        out[s0:s0 + 256] = ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).min(1)
    return out


@pytest.mark.gpu
def test_nn_distances_and_chamfer_hausdorff(lib):
    rng = np.random.default_rng(20)
    a = rng.random((3000, 3))
    b = np.concatenate([rng.random((2500, 3)), a[:100]])              # exact duplicates give zero distances
    got = M.nn_distances(a, b)
    assert np.array_equal(_bits(got), _bits(np.sqrt(_nn_ref(a, b))))
    assert np.array_equal(_bits(M.nn_distances(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV))), _bits(got))
    r = M.chamfer_hausdorff(a, b)
    pg2, gp2 = _nn_ref(a, b), _nn_ref(b, a)
    np.testing.assert_allclose(r["cd"], np.sqrt(pg2).mean() + np.sqrt(gp2).mean(), rtol=1e-12)
    np.testing.assert_allclose(r["cd_sq"], pg2.mean() + gp2.mean(), rtol=1e-12)
    assert r["hd"] == max(np.sqrt(pg2).max(), np.sqrt(gp2).max())
    with pytest.raises(ValueError):
        M.nn_distances(np.array([[0.0, np.nan, 0.0]]), b)
    with pytest.raises(N.SapcuError):
        M.nn_distances(torch.zeros(3, 3, dtype=torch.float64), b)


@pytest.mark.gpu
def test_point_to_mesh_and_normal_errors(lib):
    from sapcu_b200.generation import orient_normals
    rng = np.random.default_rng(21)
    v, f = syn.sphere_mesh(4)
    p = _shell(4000, rng, 0.495, 0.505)
    dist, face = M.point_to_mesh(p, v, f, return_face=True)
    ref, rface = mesh_distance_ref(v, f, p)
    assert np.array_equal(_bits(dist), _bits(np.sqrt(ref))) and np.array_equal(face, rface)
    assert np.array_equal(_bits(M.point_to_mesh(torch.from_numpy(p).to(DEV), torch.from_numpy(v).to(DEV), f)), _bits(dist))
    radial = (p / np.linalg.norm(p, axis=1, keepdims=True)).astype(np.float32)
    assert M.normal_errors(p, radial, v, f)["flipped"] == 0.0
    flip = rng.random(len(p)) < 0.3
    signed = np.where(flip[:, None], -radial, radial)
    e = M.normal_errors(p, signed, v, f)
    assert e["flipped"] == flip.mean() and e["angle_max"] < 10.0
    oriented = orient_normals(torch.from_numpy(p).to(DEV), torch.from_numpy(signed).to(DEV)).cpu().numpy()
    assert M.normal_errors(p, oriented, v, f)["flipped"] == 0.0
    for bad in (np.array([[np.inf, 0, 0]]), p[:, :2]):
        with pytest.raises(ValueError):
            M.point_to_mesh(bad, v, f)
    with pytest.raises(ValueError):
        M.point_to_mesh(p, v, np.array([[0, 1, len(v)]]))


def _models():
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    mfn, mfd = mfn.to(DEV), mfd.to(DEV)
    mfn.set_mode("tc"), mfd.set_mode("tc")
    return mfn, mfd


def _evaluate_ref(pred, gt, v, f, normals):
    c, r = M.unit_ball(gt)
    pred, gt, v = (pred - c) / r, (gt - c) / r, (v - c) / r
    pg2, gp2 = _nn_ref(pred, gt), _nn_ref(gt, pred)
    d2, face = mesh_distance_ref(v, f, pred)
    p2f = np.sqrt(d2)
    a, b, cc = v[f[face, 0]], v[f[face, 1]], v[f[face, 2]]
    out = {"cd": np.sqrt(pg2).mean() + np.sqrt(gp2).mean(), "cd_sq": pg2.mean() + gp2.mean(),
           "hd": max(np.sqrt(pg2).max(), np.sqrt(gp2).max()), "p2f_mean": p2f.mean(), "p2f_std": p2f.std()}
    out.update(M.normal_stats(normals, np.cross(b - a, cc - a)))
    return out


def _assert_eval(got, exp):
    assert set(got) == set(exp)
    for k in ("p2f_mean", "p2f_std", "hd", "angle_mean", "angle_median", "angle_max", "flipped"):
        assert got[k] == exp[k], k                                     # same arrays, same host reductions
    for k in ("cd", "cd_sq"):
        np.testing.assert_allclose(got[k], exp[k], rtol=1e-12)          # device means


@pytest.mark.gpu
def test_evaluate_upsampled_sphere(lib):
    from sapcu_b200.generation import Generator3D6
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 2, seed=1)
    gen = Generator3D6(*_models(), DEV, k_neighbors=100)
    pts, nrm = gen.upsample(np.expand_dims(cloud, 0), seeds=seeds, return_normals=True)
    v, f = syn.sphere_mesh(5)
    got = M.evaluate(pts, cloud, v, f, normals=nrm)
    _assert_eval(got, _evaluate_ref(pts, cloud, v, f, nrm))
    plain = M.evaluate(pts, cloud, normalize=False)
    assert set(plain) == {"cd", "cd_sq", "hd"}


@pytest.mark.gpu
def test_cli_on_process_file_output(lib, tmp_path):
    from sapcu_b200.generation import Generator3D6
    from sapcu_b200.generate import process_file
    cloud = syn.cloud(512, seed=3, shape="sphere")
    for d in ("in", "pred", "gt", "mesh"):
        (tmp_path / d).mkdir()
    np.savetxt(tmp_path / "in" / "ball.xyz", cloud, fmt="%.8f")
    np.savetxt(tmp_path / "gt" / "ball.xyz", cloud, fmt="%.8f")
    np.savetxt(tmp_path / "gt" / "other.xyz", cloud[:100], fmt="%.8f")
    v, f = syn.sphere_mesh(4)
    _write_off(tmp_path / "mesh" / "ball.off", v, f)
    gen = Generator3D6(*_models(), DEV, k_neighbors=100, dense_spacing=0.02)
    process_file(str(tmp_path / "in" / "ball.xyz"), str(tmp_path / "pred" / "ball.xyz"), gen, 1024, with_normals=True)
    out = tmp_path / "res.json"
    env = dict(os.environ, PYTHONPATH=ROOT)
    proc = subprocess.run([sys.executable, "-m", "sapcu_b200.metrics", str(tmp_path / "pred"), str(tmp_path / "gt"),
                           "--mesh-dir", str(tmp_path / "mesh"), "--json", str(out)], cwd=ROOT, env=env, capture_output=True,
                          text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    lines = proc.stdout.strip().splitlines()
    assert lines[0].startswith("ball ") and lines[-1].startswith("mean (1 files)")
    res = json.loads(out.read_text())
    pred = np.loadtxt(tmp_path / "pred" / "ball.xyz")
    exp = M.evaluate(pred[:, :3], np.loadtxt(tmp_path / "gt" / "ball.xyz"), v, f, normals=pred[:, 3:])
    assert res["files"]["ball"] == exp and res["mean"] == exp
