"""Consistently oriented normals: sapcu_orient_normals against a host restatement of its contract, and the opt-in
return_normals path of Generator3D6 / upsample_batch / process_file.

The restatement (orient_reference) is independent of the kernels' Boruvka rounds: numpy computes the edge keys,
scipy's minimum_spanning_tree runs on each edge's rank in the strict order (so its tree is the unique forest Kruskal
builds), connected_components gives the per-component roots and breadth_first_order's predecessors the path parities.
"""
import ctypes
import os

import numpy as np
import pytest
import torch
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import breadth_first_order, connected_components, minimum_spanning_tree

import sapcu_b200
import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N

DEV = "cuda:0"
SAPCU_EINVAL, SAPCU_EWORKSPACE = -1, -3


def orient_reference(points, idx, normals):
    """Host restatement of sapcu_orient_normals (include/sapcu_b200.h) -> (oriented normals [S,3] f32, root [S] int64)."""
    S, k = idx.shape
    normals = np.ascontiguousarray(normals, dtype=np.float32)
    i = np.repeat(np.arange(S, dtype=np.int64), k)
    j = idx.reshape(-1).astype(np.int64)
    m = i != j
    a, b = np.minimum(i[m], j[m]), np.maximum(i[m], j[m])
    _, first = np.unique(a * S + b, return_index=True)
    a, b = a[first], b[first]
    n = normals.astype(np.float64)
    dot = ((n[a, 0] * n[b, 0]) + (n[a, 1] * n[b, 1])) + n[a, 2] * n[b, 2]
    order = np.lexsort((b, a, -np.abs(dot)))          # larger |dot| first, then the smaller (min, max) pair
    rank = np.empty(len(order))
    rank[order] = np.arange(1, len(order) + 1)
    tree = minimum_spanning_tree(coo_matrix((rank, (a, b)), shape=(S, S)).tocsr()).tocoo()
    e = order[tree.data.astype(np.int64) - 1]
    ta, tb, tflip = a[e], b[e], (dot[e] < 0).astype(np.int64)
    ncomp, label = connected_components(coo_matrix((np.ones(len(e)), (ta, tb)), shape=(S, S)), directed=False)
    z = np.ascontiguousarray(points, dtype=np.float64)[:, 2] + 0.0      # -0.0 ties with +0.0
    o = np.lexsort((np.arange(S), -z, label))                           # per label: largest z, then lowest index
    comp_root = o[np.searchsorted(label[o], np.arange(ncomp))]
    # one BFS over the forest from a virtual node S joined to every root; edge data = flip + 1 (zero means no edge)
    g = coo_matrix((np.concatenate([tflip + 1, np.ones(ncomp, np.int64)]),
                    (np.concatenate([ta, np.full(ncomp, S)]), np.concatenate([tb, comp_root]))), shape=(S + 1, S + 1)).tocsr()
    g = (g + g.T).tocsr()
    _, pred = breadth_first_order(g, S, directed=False, return_predecessors=True)
    pred[S] = S
    par = np.zeros(S + 1, np.int64)
    par[:S] = np.asarray(g[pred[:S], np.arange(S)]).ravel() - 1
    anc = pred.astype(np.int64)
    while (anc != S).any():                                             # parity to the root by pointer doubling
        par, anc = par ^ par[anc], anc[anc]
    root = comp_root[label]
    neg = (normals[root, 2] < 0) ^ (par[:S] == 1)
    return np.where(neg[:, None], -normals, normals), root


def _sphere(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.normal(size=(n, 3))
    p /= np.linalg.norm(p, axis=1, keepdims=True)
    return p, rng


def _random_signs(n, rng):
    return np.where(rng.random(len(n))[:, None] < 0.5, -n, n).astype(np.float32)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _is_pm(out, inp):
    """every row bitwise its input or the input with all three sign bits flipped"""
    o, i = _bits(out), _bits(inp)
    return bool(((o == i).all(1) | (o == (i ^ np.uint32(0x80000000))).all(1)).all())


# ----------------------------------------------------------------------------------------- the restatement on its own (CPU)
def test_reference_orients_sphere_outward_and_ignores_input_signs():
    from scipy.spatial import cKDTree
    p, rng = _sphere(3000, 3)
    _, idx = cKDTree(p).query(p, 11)
    radial = p.astype(np.float32)
    out, root = orient_reference(p, idx, _random_signs(radial, rng))
    assert _is_pm(out, radial)
    assert ((out.astype(np.float64) * p).sum(1) > 0).all()              # outward everywhere
    assert (root == np.argmax(p[:, 2])).all()                           # one component, rooted at the top
    for _ in range(3):
        again, root2 = orient_reference(p, idx, _random_signs(radial, rng))
        assert np.array_equal(_bits(again), _bits(out)) and np.array_equal(root2, root)


def test_reference_two_components_two_roots():
    from scipy.spatial import cKDTree
    p, rng = _sphere(1000, 4)
    q = np.concatenate([p, p[::-1] * 0.5 + np.array([10.0, 0.0, -3.0])])
    _, idx = cKDTree(q).query(q, 9)
    out, root = orient_reference(q, idx, _random_signs(np.concatenate([p, -p[::-1]]).astype(np.float32), rng))
    assert set(root[:1000]) == {int(np.argmax(q[:1000, 2]))} and set(root[1000:]) == {1000 + int(np.argmax(q[1000:, 2]))}
    c = np.where(np.arange(2000)[:, None] < 1000, 0.0, np.array([10.0, 0.0, -3.0]))
    assert ((out.astype(np.float64) * (q - c)).sum(1) > 0).all()


def test_orient_normals_refuses_cpu_tensors():
    from sapcu_b200.generation import orient_normals
    with pytest.raises(N.SapcuError):
        orient_normals(torch.zeros(4, 3, dtype=torch.float64), torch.zeros(4, 3))
    with pytest.raises(ValueError):
        orient_normals(torch.zeros(4, 3), torch.zeros(4, 3))


# ----------------------------------------------------------------------------------------- the operator (GPU)
@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


def _knn_self(points, K):
    L = N.lib()
    d = torch.from_numpy(np.ascontiguousarray(points, dtype=np.float64)).to(DEV)
    idx = torch.empty(d.shape[0], K, dtype=torch.int32, device=DEV)
    ws = torch.empty(L.sapcu_knn_workspace_bytes(d.shape[0]), dtype=torch.uint8, device=DEV)
    N.check(L.sapcu_knn(N.ptr(d), d.shape[0], N.ptr(d), d.shape[0], K, N.ptr(idx), N.ptr(ws), ws.numel(), N.stream_ptr(DEV)))
    return idx.cpu().numpy()


def _gpu_orient(points, idx, normals, stream=None):
    L = N.lib()
    S, k = idx.shape
    d_p = torch.from_numpy(np.ascontiguousarray(points, dtype=np.float64)).to(DEV)
    d_i = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32)).to(DEV)
    d_n = torch.from_numpy(np.ascontiguousarray(normals, dtype=np.float32)).to(DEV)
    root = torch.full((S,), -1, dtype=torch.int32, device=DEV)
    ws = torch.empty(L.sapcu_orient_normals_workspace_bytes(S, k), dtype=torch.uint8, device=DEV)
    st = stream or torch.cuda.current_stream(DEV)
    st.wait_stream(torch.cuda.current_stream(DEV))
    N.check(L.sapcu_orient_normals(N.ptr(d_p), S, N.ptr(d_i), k, N.ptr(d_n), N.ptr(root), N.ptr(ws), ws.numel(),
                                   ctypes.c_void_p(st.cuda_stream)), "sapcu_orient_normals")
    st.synchronize()
    N.check_device("orient")
    return d_n.cpu().numpy(), root.cpu().numpy()


def _check_operator(points, idx, normals):
    got, root = _gpu_orient(points, idx, normals)
    ref, ref_root = orient_reference(points, idx, normals)
    assert _is_pm(got, normals)
    assert np.array_equal(_bits(got), _bits(ref))
    assert np.array_equal(root, ref_root)
    return got, root


@pytest.mark.gpu
def test_operator_sphere_random_signs(lib):
    p, rng = _sphere(20000, 5)
    p *= 0.5
    idx = _knn_self(p, 11)
    radial = (p / np.linalg.norm(p, axis=1, keepdims=True)).astype(np.float32)
    got, root = _check_operator(p, idx, _random_signs(radial, rng))
    assert ((got.astype(np.float64) * p).sum(1) > 0).all()
    # input signs do not matter; repeated runs and another stream give the same bits
    again, _ = _gpu_orient(p, idx, _random_signs(radial, rng))
    assert np.array_equal(_bits(again), _bits(got))
    n = _random_signs(radial, rng)
    first, _ = _gpu_orient(p, idx, n)
    assert np.array_equal(_bits(_gpu_orient(p, idx, n)[0]), _bits(first))
    assert np.array_equal(_bits(_gpu_orient(p, idx, n, stream=torch.cuda.Stream(device=DEV))[0]), _bits(first))


@pytest.mark.gpu
def test_operator_random_normals_sign_invariance(lib):
    p, rng = _sphere(5000, 6)
    n = rng.normal(size=(5000, 3))
    n = (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32)
    idx = _knn_self(p, 11)
    got, _ = _check_operator(p, idx, n)
    flipped = n.copy()
    sel = rng.random(5000) < 0.3
    flipped[sel] = -flipped[sel]
    assert np.array_equal(_bits(_gpu_orient(p, idx, flipped)[0]), _bits(got))


def _models():
    from sapcu_b200.fn import config as fc
    from sapcu_b200.fd import config as dc
    mfn = fc.get_model(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    mfd = dc.get_model(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")), None)
    syn.init_weights(mfn, seed=100, stress=True)
    syn.init_weights(mfd, seed=200, stress=True)
    return mfn.to(DEV), mfd.to(DEV)


@pytest.mark.gpu
def test_operator_pipeline_normals_on_boxes(lib):
    from sapcu_b200.generation import Generator3D6
    cloud = syn.cloud(2048, seed=9, shape="boxes")
    seeds = syn.seeds(cloud, 3, seed=10)
    mfn, mfd = _models()
    mfn.set_mode("tc"), mfd.set_mode("tc")
    gen = Generator3D6(mfn, mfd, DEV, k_neighbors=100, remove_outliers=False)
    out, _, n, _ = gen.displace_device(torch.from_numpy(cloud).to(DEV), torch.from_numpy(seeds).to(DEV), return_parts=True)
    pts, n = out.cpu().numpy(), n.cpu().numpy()
    _check_operator(pts, _knn_self(pts, 11), n)


@pytest.mark.gpu
def test_operator_two_components(lib):
    p, rng = _sphere(4000, 7)
    q = np.concatenate([p * 0.5, p[::-1] * 0.3 + np.array([5.0, -2.0, 1.0])])
    n = _random_signs(np.concatenate([p, p[::-1]]).astype(np.float32), rng)
    _, root = _check_operator(q, _knn_self(q, 11), n)
    assert sorted(set(root.tolist())) == [int(np.argmax(q[:4000, 2])), 4000 + int(np.argmax(q[4000:, 2]))]


@pytest.mark.gpu
def test_operator_duplicated_points(lib):
    p, rng = _sphere(3000, 8)
    q = np.concatenate([p, p[:600], p[:200]])
    n = rng.normal(size=(3800, 3))
    n = (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32)
    idx = _knn_self(q, 11)
    assert (idx[:, 0] != np.arange(3800)).any()                       # self is not always in column 0
    _check_operator(q, idx, n)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["k1_self_only", "k1_nearest_other", "k128", "S1", "S2"])
def test_operator_extreme_sizes(lib, case):
    p, rng = _sphere(3000, 11)
    n = rng.normal(size=(3000, 3)).astype(np.float32)
    if case == "k1_self_only":
        idx = _knn_self(p, 1)
    elif case == "k1_nearest_other":                                  # a forest of many small components
        idx = np.ascontiguousarray(_knn_self(p, 2)[:, 1:])
    elif case == "k128":
        idx = _knn_self(p, 128)
    else:
        s = 1 if case == "S1" else 2
        p, n = p[:s], n[:s]
        idx = _knn_self(p, s)
    got, root = _check_operator(p, idx, n)
    if case == "k1_self_only" or case == "S1":
        assert np.array_equal(root, np.arange(len(p))) and (got[:, 2] >= 0).all()


@pytest.mark.gpu
def test_operator_skips_out_of_range_entries(lib):
    p, rng = _sphere(2000, 12)
    n = rng.normal(size=(2000, 3)).astype(np.float32)
    idx = _knn_self(p, 11)
    bad = idx.copy()
    sel = rng.random(bad.shape) < 0.2
    bad[sel] = rng.choice(np.array([-1, 2000, 2 ** 31 - 1, -2 ** 31], dtype=np.int64), size=int(sel.sum()))
    same = np.where(sel, np.arange(2000)[:, None], idx)                # skipped exactly like self entries
    got, root = _gpu_orient(p, bad, n)
    ref, ref_root = orient_reference(p, same, n)
    assert np.array_equal(_bits(got), _bits(ref)) and np.array_equal(root, ref_root)


@pytest.mark.gpu
def test_operator_error_codes(lib):
    L = N.lib()
    S = 64
    d_p = torch.zeros(S, 3, dtype=torch.float64, device=DEV)
    d_n = torch.ones(S, 3, dtype=torch.float32, device=DEV)
    d_i = torch.zeros(S, 129, dtype=torch.int32, device=DEV)
    ws = torch.empty(L.sapcu_orient_normals_workspace_bytes(S, 128), dtype=torch.uint8, device=DEV)
    st = N.stream_ptr(DEV)
    before = L.sapcu_launch_count()
    for k in (0, 129):
        assert L.sapcu_orient_normals(N.ptr(d_p), S, N.ptr(d_i), k, N.ptr(d_n), None, N.ptr(ws), ws.numel(), st) == SAPCU_EINVAL
        assert L.sapcu_orient_normals_workspace_bytes(S, k) == 0
    need = L.sapcu_orient_normals_workspace_bytes(S, 10)
    assert 0 < need <= ws.numel()
    assert L.sapcu_orient_normals(N.ptr(d_p), S, N.ptr(d_i), 10, N.ptr(d_n), None, N.ptr(ws), need - 1, st) == SAPCU_EWORKSPACE
    assert L.sapcu_orient_normals(N.ptr(d_p), 0, N.ptr(d_i), 10, N.ptr(d_n), None, N.ptr(ws), ws.numel(), st) == SAPCU_EINVAL
    assert L.sapcu_launch_count() == before
    assert torch.equal(d_n, torch.ones_like(d_n))


# ----------------------------------------------------------------------------------------- the public API (GPU)
def _expected(gen, cloud, seeds, batch=None):
    """Per problem: the points and raw fn normals of return_parts with the outlier mask applied, and the restatement's
    orientation of those normals over those points (k = 10 -> 11 self-neighbours)."""
    out, _, raw, _ = gen.displace_device(torch.from_numpy(cloud).to(DEV), torch.from_numpy(seeds).to(DEV),
                                         return_parts=True, batch=batch)
    so = (0, seeds.shape[0]) if batch is None else batch[1]
    res = []
    for b in range(len(so) - 1):
        p, n = out[so[b]:so[b + 1]], raw[so[b]:so[b + 1]]
        if gen.remove_outliers:
            with torch.cuda.device(gen.device):
                keep = gen._outlier_keep(p).bool()
            p, n = p[keep], n[keep]
        p, n = p.cpu().numpy(), n.cpu().numpy()
        res.append((p, n, orient_reference(p, _knn_self(p, min(11, len(p))), n)[0]))
    return res


def _check_api(pts, nrm, plain, expected):
    p, raw, oriented = expected
    assert pts.dtype == np.float64 and nrm.dtype == np.float32 and nrm.shape == pts.shape
    assert np.array_equal(pts, plain)            # the points of return_normals=False, bit for bit
    assert np.array_equal(pts, p)
    assert _is_pm(nrm, raw)                      # the pipeline's own normals, only signs changed
    assert np.array_equal(_bits(nrm), _bits(oriented))


@pytest.mark.gpu
@pytest.mark.parametrize("remove_outliers", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "tc", "fast"])
def test_upsample_return_normals(lib, mode, remove_outliers):
    from sapcu_b200.generation import Generator3D6
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 1.5, seed=1)
    mfn, mfd = _models()
    mfn.set_mode(mode), mfd.set_mode(mode)
    gen = Generator3D6(mfn, mfd, DEV, k_neighbors=100, remove_outliers=remove_outliers)
    data = np.expand_dims(cloud, 0)
    pts, nrm = gen.upsample(data, seeds=seeds, return_normals=True)
    _check_api(pts, nrm, gen.upsample(data, seeds=seeds), _expected(gen, cloud, seeds)[0])
    # several workers on the device list: normals gathered on the primary device, oriented there over the whole cloud
    multi = Generator3D6(mfn, mfd, [DEV] * 3, k_neighbors=100, remove_outliers=remove_outliers)
    mp, mn = multi.upsample(data, seeds=seeds, return_normals=True)
    _check_api(mp, mn, multi.upsample(data, seeds=seeds), _expected(multi, cloud, seeds)[0])
    if mode == "fp32":                           # split-invariant: the same arrays as one device
        assert np.array_equal(mp, pts) and np.array_equal(_bits(mn), _bits(nrm))
    # a batch: each cloud's normals oriented on its own points
    clouds = [syn.cloud(n, seed=40 + b, shape="boxes") for b, n in enumerate((1024, 700, 1500))]
    sds = [syn.seeds(c, r, seed=50 + b) for b, (c, r) in enumerate(zip(clouds, (1.0, 0.5, 0.8)))]
    res = gen.upsample_batch(clouds, sds, return_normals=True)
    plain = gen.upsample_batch(clouds, sds)
    co = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    so = np.concatenate([[0], np.cumsum([s.shape[0] for s in sds])]).astype(np.int64)
    exp = _expected(gen, np.concatenate(clouds), np.concatenate(sds), batch=(co, so))
    assert len(res) == 3
    for b in range(3):
        _check_api(res[b][0], res[b][1], plain[b], exp[b])
    N.check_device("upsample(return_normals=True)")


@pytest.mark.gpu
def test_process_file_with_normals(lib, tmp_path):
    from sapcu_b200.generation import Generator3D6
    from sapcu_b200.generate import process_file
    mfn, mfd = _models()
    mfn.set_mode("tc"), mfd.set_mode("tc")
    cloud = syn.cloud(256, seed=5, shape="sphere") * 3.0 + np.array([1.0, -2.0, 0.5])
    np.savetxt(tmp_path / "in.xyz", cloud, fmt="%.8f")
    gen = Generator3D6(mfn, mfd, DEV, k_neighbors=100, dense_spacing=0.02)
    process_file(str(tmp_path / "in.xyz"), str(tmp_path / "plain.xyz"), gen, 1024)
    process_file(str(tmp_path / "in.xyz"), str(tmp_path / "normals.xyz"), gen, 1024, with_normals=True)
    plain = (tmp_path / "plain.xyz").read_text().splitlines()
    six = (tmp_path / "normals.xyz").read_text().splitlines()
    assert len(six) == len(plain) == 1024
    assert all(len(r.split()) == 6 for r in six)
    assert [" ".join(r.split()[:3]) for r in six] == plain
    n = np.loadtxt(tmp_path / "normals.xyz")[:, 3:]
    np.testing.assert_allclose(np.linalg.norm(n, axis=1), 1.0, atol=2e-6)
