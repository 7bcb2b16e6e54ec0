"""Earth Mover's Distance: sapcu_emd against scipy's exact assignment and a numpy restatement of its costs, and the
sapcu_b200.metrics API (emd_match, emd, evaluate(emd=True), the CLI's --emd).

cost_ref restates c_ij = sqrt(((dx*dx)+(dy*dy))+(dz*dz)) in fp64 (numpy rounds every operation and never contracts, like
the -fmad=false build of csrc/emd.cu), so every returned per-point cost is checked bit for bit.  phase1_rounds restates the
first auction phase (same constants, same arithmetic, same tie rules) to place the round cap of the cap tests.
"""
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
from sapcu_b200 import metrics as M

DEV = "cuda:0"
SAPCU_EINVAL, SAPCU_EWORKSPACE = -1, -3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_N = 131072


# ----------------------------------------------------------------------------------------- the restatement
def cost_ref(a, b):
    """c of every row of a with the same row of b ([n] f64)."""
    d = np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)
    return np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])


def cost_matrix(a, b):
    d = a[:, None, :] - b[None, :, :]
    return np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])


def phase1_rounds(a, b):
    """Rounds of the first auction phase and whether its bounds already certify the result at rel_tol = 1e-6."""
    C = cost_matrix(a, b)
    n = len(a)
    cmax = float(C.max())
    eps_min = (cmax if cmax > 0 else 1.0) * 2.0 ** -40
    eps = max(cmax * 0.25, eps_min)
    p = np.zeros(n)
    owner, assign = np.full(n, -1), np.full(n, -1)
    unas = np.arange(n)
    rounds = 0
    while len(unas):
        rounds += 1
        V = C[unas] + p[None, :]
        j1 = np.argmin(V, 1)
        v1 = V[np.arange(len(unas)), j1]
        V[np.arange(len(unas)), j1] = np.inf
        v2 = V.min(1)
        bid = (p[j1] + (v2 - v1)) + eps
        order = np.lexsort((unas, -bid, j1))                     # per object: highest bid, then lowest person
        first = np.ones(len(order), bool)
        first[1:] = j1[order][1:] != j1[order][:-1]
        win = order[first]
        objs, who = j1[win], unas[win]
        prev = owner[objs]
        p[objs] = bid[win]
        owner[objs] = who
        assign[who] = objs
        assign[prev[prev >= 0]] = -1
        unas = np.flatnonzero(assign < 0)
    primal = C[np.arange(n), assign].sum()
    dual = (C + p[None, :]).min(1).sum() - p.sum()
    return rounds, primal - dual > 2 * (1e-6 * primal + n * eps_min)


def shell(n, seed, r_lo=0.49, r_hi=0.51):
    rng = np.random.default_rng(seed)
    q = rng.normal(size=(n, 3))
    return q * (r_lo + (r_hi - r_lo) * rng.random((n, 1))) / np.linalg.norm(q, axis=1, keepdims=True)


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


# ----------------------------------------------------------------------------------------- CPU
def test_workspace_bytes_limits_and_linear_growth():
    L = N.lib()
    for n in (0, -1, MAX_N + 1, 1 << 40):
        assert L.sapcu_emd_workspace_bytes(n) == 0
    assert 0 < L.sapcu_emd_workspace_bytes(1) < L.sapcu_emd_workspace_bytes(MAX_N)
    per_point = [(L.sapcu_emd_workspace_bytes(2 * n) - L.sapcu_emd_workspace_bytes(n)) / n for n in (4096, 16384, 65536)]
    assert all(76 <= x <= 77 for x in per_point), per_point              # 76 bytes per point plus a constant
    assert L.sapcu_emd_workspace_bytes(MAX_N) < 80 * MAX_N + (1 << 20)


def test_emd_match_rejects_bad_input_before_any_device_call():
    a = np.zeros((5, 3))
    for b in (np.zeros((4, 3)), np.zeros((6, 3))):
        with pytest.raises(ValueError, match="differ in size"):
            M.emd_match(a, b)
    with pytest.raises(ValueError, match="non-finite"):
        M.emd_match(a, np.array([[0.0, np.nan, 0.0]] * 5))
    with pytest.raises(ValueError, match="non-finite"):
        M.emd(np.array([[np.inf, 0.0, 0.0]] * 5), a)
    with pytest.raises(ValueError):
        M.emd_match(np.zeros((0, 3)), np.zeros((0, 3)))
    with pytest.raises(ValueError):
        M.emd_match(a[:, :2], a[:, :2])
    with pytest.raises(ValueError):
        M.emd_match(a, a, rel_tol=-1.0)


def test_phase1_restatement_on_hand_cases():
    # two rows that want different objects: one round; identical clouds: one round
    a = np.array([[0.0, 0, 0], [10.0, 0, 0]])
    assert phase1_rounds(a, a + [1.0, 0, 0])[0] == 1
    assert phase1_rounds(shell(64, 1), shell(64, 1)[::-1].copy())[0] == 1


# ----------------------------------------------------------------------------------------- GPU: the operator
@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return N.lib()


def _emd_gpu(a, b, rel_tol=1e-6, stream=None, ws_bytes=None):
    """(assign [n] int32, cost [n] f64, stats [6] f64) of one sapcu_emd call."""
    L = N.lib()
    d_a = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(DEV)
    d_b = torch.from_numpy(np.ascontiguousarray(b, dtype=np.float64)).to(DEV)
    n = d_a.shape[0]
    assign = torch.full((n,), -7, dtype=torch.int32, device=DEV)
    cost = torch.full((n,), -1.0, dtype=torch.float64, device=DEV)
    stats = torch.full((6,), -1.0, dtype=torch.float64, device=DEV)
    ws = torch.full((L.sapcu_emd_workspace_bytes(n),), 0xA5, dtype=torch.uint8, device=DEV)   # no state may leak in
    st = stream or torch.cuda.current_stream(DEV)
    st.wait_stream(torch.cuda.current_stream(DEV))
    N.check(L.sapcu_emd(N.ptr(d_a), N.ptr(d_b), n, rel_tol, N.ptr(assign), N.ptr(cost), N.ptr(stats), N.ptr(ws),
                        ws.numel() if ws_bytes is None else ws_bytes, ctypes.c_void_p(st.cuda_stream)), "sapcu_emd")
    st.synchronize()
    N.check_device("sapcu_emd")
    return assign.cpu().numpy(), cost.cpu().numpy(), stats.cpu().numpy()


def _eps_min(a, b):
    cmax = max(float(cost_matrix(a[i:i + 512], b).max()) for i in range(0, len(a), 512))
    return (cmax if cmax > 0 else 1.0) * 2.0 ** -40


def _check_certified(a, b, assign, cost, stats, rel_tol=1e-6):
    n = len(a)
    assert np.array_equal(np.sort(assign), np.arange(n))                    # a permutation
    assert np.array_equal(_bits(cost), _bits(cost_ref(a, b[assign])))
    primal, dual = stats[0], stats[1]
    assert stats[5] == 1.0 and stats[3] >= 1 and stats[4] >= 1
    assert primal - dual <= (rel_tol * primal + n * _eps_min(a, b)) * (1 + 1e-9)
    assert primal == pytest.approx(math.fsum(cost), rel=1e-13, abs=1e-300)
    return primal, dual


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 17, 512, 2048, 4096])
@pytest.mark.parametrize("kind", ["shells", "gauss"])
def test_against_the_exact_optimum(lib, n, kind):
    from scipy.optimize import linear_sum_assignment
    from scipy.spatial.distance import cdist
    if kind == "shells":
        a, b = shell(n, 100 + n), shell(n, 200 + n)
    else:
        rng = np.random.default_rng(300 + n)
        a, b = rng.normal(size=(n, 3)), rng.normal(size=(n, 3)) * 0.7 + 0.1
    assign, cost, stats = _emd_gpu(a, b)
    primal, dual = _check_certified(a, b, assign, cost, stats)
    _, col = linear_sum_assignment(cdist(a, b))
    opt = math.fsum(cost_ref(a, b[col]))
    assert dual <= opt * (1 + 1e-12) and opt <= primal * (1 + 1e-12)


@pytest.mark.gpu
def test_ties_on_a_lattice_with_duplicates(lib):
    from scipy.optimize import linear_sum_assignment
    rng = np.random.default_rng(7)
    g = np.stack(np.meshgrid(*[np.arange(4.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
    a, b = g[rng.integers(0, 64, 1024)], g[rng.integers(0, 64, 1024)]
    assign, cost, stats = _emd_gpu(a, b)
    primal, dual = _check_certified(a, b, assign, cost, stats)
    _, col = linear_sum_assignment(cost_matrix(a, b))
    opt = math.fsum(cost_ref(a, b[col]))
    assert dual <= opt * (1 + 1e-12) and opt <= primal * (1 + 1e-12)


@pytest.mark.gpu
def test_identity_under_a_permutation(lib):
    n = 8192
    a = shell(n, 11)
    perm = np.random.default_rng(12).permutation(n)
    b = a[perm]
    assign, cost, stats = _emd_gpu(a, b)
    inv = np.empty(n, np.int64)
    inv[perm] = np.arange(n)
    assert np.array_equal(assign, inv)
    assert stats[5] == 1.0 and stats[0] <= n * _eps_min(a, b) and (cost == 0).all()


@pytest.mark.gpu
def test_translation_is_the_shift_length(lib):
    # For unsquared Euclidean costs the identity matching is optimal under a translation: sum_i |a_i + t - b_s(i)| >=
    # |sum_i (a_i + t - a_s(i))| = n |t|.  rel_tol = 0 certifies to the 2^-40 floor, |t| / max c > 0.96 keeps that below 1e-12.
    n = 32768
    a = shell(n, 13)
    t = np.array([12.0, -9.0, 20.0])
    assign, cost, stats = _emd_gpu(a, a + t, rel_tol=0.0)
    assert np.array_equal(np.sort(assign), np.arange(n)) and stats[5] == 1.0
    assert np.array_equal(_bits(cost), _bits(cost_ref(a, (a + t)[assign])))
    assert stats[0] / n == pytest.approx(np.linalg.norm(t), rel=1e-12)


@pytest.mark.gpu
def test_repeat_and_second_stream_are_bitwise_equal(lib):
    a, b = shell(4096, 21), shell(4096, 22)
    first = _emd_gpu(a, b)
    again = _emd_gpu(a, b)
    other = _emd_gpu(a, b, stream=torch.cuda.Stream(device=DEV))
    for x in (again, other):
        assert np.array_equal(x[0], first[0])
        assert np.array_equal(_bits(x[1]), _bits(first[1])) and np.array_equal(_bits(x[2]), _bits(first[2]))


@pytest.mark.gpu
def test_limits_and_errors(lib):
    L = N.lib()
    n = 16
    a = torch.zeros(n, 3, dtype=torch.float64, device=DEV)
    assign = torch.full((n,), -7, dtype=torch.int32, device=DEV)
    cost = torch.zeros(n, dtype=torch.float64, device=DEV)
    stats = torch.zeros(6, dtype=torch.float64, device=DEV)
    need = L.sapcu_emd_workspace_bytes(n)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    st = N.stream_ptr(DEV)
    p = [N.ptr(a), N.ptr(a), N.ptr(assign), N.ptr(cost), N.ptr(stats), N.ptr(ws)]
    before = L.sapcu_launch_count()

    def call(n_, tol, ptrs, nbytes):
        return L.sapcu_emd(ptrs[0], ptrs[1], n_, tol, ptrs[2], ptrs[3], ptrs[4], ptrs[5], nbytes, st)
    for n_, tol in ((0, 1e-6), (MAX_N + 1, 1e-6), (n, -1e-9), (n, float("nan"))):
        assert call(n_, tol, p, need) == SAPCU_EINVAL
    for k in range(6):
        assert call(n, 1e-6, p[:k] + [None] + p[k + 1:], need) == SAPCU_EINVAL
    assert call(n, 1e-6, p, need - 1) == SAPCU_EWORKSPACE
    assert L.sapcu_launch_count() == before and (assign == -7).all()
    # the largest n converges: only the certificate and the permutation are checked
    big_a, big_b = shell(MAX_N, 31), shell(MAX_N, 32)
    r = M.emd_match(big_a, big_b)
    assert r["converged"] and np.array_equal(np.sort(r["assignment"]), np.arange(MAX_N))
    assert r["emd"] - r["emd_lower"] <= 1e-6 * r["emd"] + 1.1 * 2.0 ** -40          # max c <= 1.02 on these shells


_CAP_SCRIPT = r"""
import json, sys
import numpy as np, torch
sys.path.insert(0, sys.argv[1])
from sapcu_b200 import _native as N
from sapcu_b200 import metrics as M
d = np.load(sys.argv[2])
torch.cuda.set_device(0)
r = M.emd_match(d["a"], d["b"])
torch.cuda.synchronize()
try:
    M.emd(d["a"], d["b"])
    raised = False
except N.SapcuError:
    raised = True
torch.cuda.synchronize()
print(json.dumps({"assign": r["assignment"].tolist(), "cost": r["cost"].tolist(), "emd": r["emd"], "lower": r["emd_lower"],
                  "phases": r["phases"], "rounds": r["rounds"], "converged": r["converged"], "raised": raised,
                  "status": N.lib().sapcu_device_status()}))
"""


@pytest.mark.gpu
def test_round_cap(lib, tmp_path):
    a, b = shell(64, 41), shell(64, 42)
    r1, uncertified = phase1_rounds(a, b)
    assert r1 >= 2 and uncertified                               # the input needs a second phase
    np.savez(tmp_path / "ab.npz", a=a, b=b)
    (tmp_path / "cap.py").write_text(_CAP_SCRIPT)

    def run(cap):
        env = dict(os.environ, SAPCU_EMD_MAX_ROUNDS=str(cap))
        proc = subprocess.run([sys.executable, str(tmp_path / "cap.py"), ROOT, str(tmp_path / "ab.npz")], env=env,
                              capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stdout + proc.stderr
        return json.loads(proc.stdout.strip().splitlines()[-1])

    below = run(r1 - 1)                                          # phase 1 never completes
    assert below["status"] == 0 and not below["converged"] and below["raised"]
    assert below["assign"] == [-1] * 64 and below["emd"] == float("inf") and below["phases"] == 0
    between = run(r1)                                            # phase 1 completes, phase 2 is cut
    assert between["status"] == 0 and not between["converged"] and between["raised"]
    assert between["phases"] == 1 and between["rounds"] == r1
    assign, cost = np.array(between["assign"]), np.array(between["cost"])
    assert np.array_equal(np.sort(assign), np.arange(64))
    assert np.array_equal(_bits(cost), _bits(cost_ref(a, b[assign])))
    from scipy.optimize import linear_sum_assignment
    _, col = linear_sum_assignment(cost_matrix(a, b))
    opt = math.fsum(cost_ref(a, b[col])) / 64
    assert between["lower"] <= opt * (1 + 1e-12) and opt <= between["emd"] * (1 + 1e-12)
    # this process kept the default cap
    _, _, stats = _emd_gpu(a, b)
    assert stats[5] == 1.0 and stats[3] >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2])
def test_overflowing_costs_return_no_phase(lib, n):
    # |a - b| = 2e200: the squared distance overflows, so c_max = +inf and no finite bid exists
    a = np.array([[1e200, 0.0, 0.0], [0.0, 1.0, 0.0]])[:n]
    b = np.array([[-1e200, 0.0, 0.0], [0.0, 2.0, 0.0]])[:n]
    assign, cost, stats = _emd_gpu(a, b)
    assert (assign == -1).all() and np.isinf(cost).all()
    assert stats[0] == np.inf and stats[5] == 0.0 and stats[3] == 0.0
    assert N.lib().sapcu_device_status() == 0
    with pytest.raises(ValueError, match="overflow"):
        M.emd_match(a, b)
    # far apart but representable: solved as usual, and the next call on the device is unaffected
    a, b = a * 1e-50, b * 1e-50
    assign, cost, stats = _emd_gpu(a, b)
    assert stats[5] == 1.0 and np.array_equal(_bits(cost), _bits(cost_ref(a, b[assign])))
    best = min(math.fsum(cost_ref(a, b[list(p)])) for p in ([[0]] if n == 1 else [[0, 1], [1, 0]]))
    assert stats[1] <= best * (1 + 1e-12) and best <= stats[0] * (1 + 1e-12)
    assert _emd_gpu(shell(256, 61), shell(256, 62))[2][5] == 1.0


# ----------------------------------------------------------------------------------------- GPU: the Python API
@pytest.mark.gpu
def test_emd_match_and_emd(lib):
    a, b = shell(1000, 51), shell(1000, 52)
    r = M.emd_match(a, b)
    assign, cost, stats = _emd_gpu(a, b)
    assert np.array_equal(r["assignment"], assign) and np.array_equal(_bits(r["cost"]), _bits(cost))
    assert r["emd"] == stats[0] / 1000 and r["emd_lower"] == stats[1] / 1000 and r["converged"]
    assert (r["phases"], r["rounds"]) == (int(stats[3]), int(stats[4]))
    assert M.emd(a, b) == r["emd"]
    assert M.emd(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)) == r["emd"]
    with pytest.raises(ValueError):
        M.emd_match(torch.from_numpy(a).to(DEV), torch.from_numpy(b[:999]).to(DEV))


@pytest.mark.gpu
def test_evaluate_with_emd_on_an_upsampled_sphere(lib):
    from test_metrics import _models
    from sapcu_b200.generation import Generator3D6
    cloud = syn.cloud(2048, seed=0, shape="sphere")
    seeds = syn.seeds(cloud, 2, seed=1)
    gen = Generator3D6(*_models(), DEV, k_neighbors=100)
    pts = gen.upsample(np.expand_dims(cloud, 0), seeds=seeds)
    gt = syn.cloud(len(pts), seed=5, shape="sphere")
    plain = M.evaluate(pts, gt)
    got = M.evaluate(pts, gt, emd=True)
    assert set(plain) == {"cd", "cd_sq", "hd"} and set(got) == {"cd", "cd_sq", "hd", "emd"}
    for k in plain:
        assert _bits(got[k]) == _bits(plain[k]), k
    c, r = M.unit_ball(gt)
    assert got["emd"] == M.emd((pts - c) / r, (gt - c) / r)
    assert got["emd"] >= got["cd"] / 2                            # EMD >= each direction's mean nearest distance
    with pytest.raises(ValueError):
        M.evaluate(pts, gt[:-1], emd=True)


@pytest.mark.gpu
def test_cli_emd_on_process_file_output(lib, tmp_path):
    from test_metrics import _models
    from sapcu_b200.generation import Generator3D6
    from sapcu_b200.generate import process_file
    cloud = syn.cloud(512, seed=3, shape="sphere")
    for d in ("in", "pred", "gt"):
        (tmp_path / d).mkdir()
    np.savetxt(tmp_path / "in" / "ball.xyz", cloud, fmt="%.8f")
    gen = Generator3D6(*_models(), DEV, k_neighbors=100, dense_spacing=0.02)
    process_file(str(tmp_path / "in" / "ball.xyz"), str(tmp_path / "pred" / "ball.xyz"), gen, 1024, with_normals=True)
    pred = np.loadtxt(tmp_path / "pred" / "ball.xyz")
    np.savetxt(tmp_path / "pred" / "other.xyz", pred, fmt="%.8f")
    np.savetxt(tmp_path / "gt" / "ball.xyz", syn.cloud(len(pred), seed=4, shape="sphere"), fmt="%.8f")
    np.savetxt(tmp_path / "gt" / "other.xyz", cloud, fmt="%.8f")                   # 512 points against 1024: skipped
    out = tmp_path / "res.json"
    env = dict(os.environ, PYTHONPATH=ROOT)
    proc = subprocess.run([sys.executable, "-m", "sapcu_b200.metrics", str(tmp_path / "pred"), str(tmp_path / "gt"), "--emd",
                           "--json", str(out)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    lines = proc.stdout.strip().splitlines()
    assert any(ln.startswith("other: EMD skipped") for ln in lines), lines
    assert lines[-1].startswith("mean (2 files)")
    res = json.loads(out.read_text())
    gt = np.loadtxt(tmp_path / "gt" / "ball.xyz")
    assert res["files"]["ball"] == M.evaluate(pred[:, :3], gt, normals=pred[:, 3:], emd=True)
    assert set(res["files"]["other"]) == {"cd", "cd_sq", "hd"}
    assert res["mean"]["emd"] == res["files"]["ball"]["emd"]
