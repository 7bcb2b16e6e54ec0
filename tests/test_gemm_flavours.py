"""Every tensor-core GEMM flavour on its own, against a float64 reference of the same contraction.

sapcu_gemm_case runs ONE contraction through the forwards' dispatcher (engine choice, fast-mode switches, fallbacks), with
weights split and LIF tables built by the code of sapcu_model_finalize.  Each GPU case asserts the exact kernel instantiation
it targets (a silent fall-back to another engine fails) and an error bound stated per flavour:

  contraction   |y - y64| <= eps_op * S + eps_acc(K) * S (+ eps_abs * sum|x|),   S = sum_k |x_k| |w_k|
                  3xTF32 (HM 0)       eps_op = 2^-20 (dropped lo*lo product, tf32 lo planes)
                  fp16x3 (HM 1, 2)    eps_op = 2^-20, eps_abs = 2^-25 * winv (the fp16 weight split's absolute floor for
                                      weights far below the matrix maximum, model.cu split_weights)
                  one fp16 plane (3)  eps_op = 2^-11 (x * 2^13 and w * 2^e each rounded to fp16), eps_abs as above
                  single-pass TF32(4) eps_op = 2^-9 (both operands truncated to 10 mantissa bits)
                  SIMT (fp32 FFMA)    eps_op = (K + 2) * 2^-24 (one rounding per k step, worst case)
                  eps_acc(K) = 4 * sqrt(K / k_step) * 2^-24: fp32 accumulation over K / k_step MMA steps (k_step 8 for
                  tf32, 16 for fp16), a probabilistic rounding bound with margin 4
  epilogue      |u - u64| <= |scale| * (contraction bound + 2^-22 |acc + bias + edge|) + 2^-22 |shift|
  LIF outputs   eps_chain + |dF/du| * eps_u, dF/du by central differences of the fp64 chain per element; eps_chain =
                  LT_BOUND = 5e-5 for tables (the fit meets LT_TOL = 4e-5 at its acceptance points, up to 4.4e-5
                  between), EPS_MUFU for the exact recurrence of the parity-grade epilogues, EPS_FAST_MUFU
                  for the fast mode's reduced recurrence, plus the output format's rounding (fp16 planes of y * 2^13)
  pool          the max of the pooled elements' bounds (max is 1-Lipschitz)
  attention     sum_j a_j |vp_j - Y| eps_y_j / at_sqrt + 2^-20 * sum_j a_j |vp_j| (softmax, fp32 sums)

CPU tests restate the reference against the oracle's own layer compositions and show that every bound is tight enough to
catch a dropped lo product, a T-1 step chain and a pool over pool_M - 1 points.
"""
import json
import math
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest
import torch

import sapcu_oracle as orc

LT_TOL = 4e-5            # the table fit's acceptance bound at its acceptance points
LT_BOUND = 5e-5          # |table - exact chain| anywhere, as test_lif_table_host_selftest asserts for the host restatement
EPS_MUFU = 4e-6          # exact-recurrence LIF^T epilogue (fp32 with MUFU exp / rcp)
EPS_FAST_MUFU = 6e-5     # SAPCU_MODE_FAST's reduced-MUFU recurrence
ACT_NONE, ACT_LEAKY, ACT_GELU, ACT_LIF = 0, 1, 2, 3
A_PLAIN, A_EDGECAT, A_ATTNIN = 0, 1, 2
MODES = {"fp32": 0, "tc": 1, "tf32": 2, "fast": 3}
EPS_OP = {0: 2.0 ** -20, 1: 2.0 ** -20, 2: 2.0 ** -20, 3: 2.0 ** -11, 4: 2.0 ** -9}
DEV = "cuda:0"


# ----------------------------------------------------------------------------------------- float64 reference
def weight_split16(w):
    """winv of the fp16 weight split (model.cu split_weights): max |w| * 2^e in [2^13, 2^14), winv = 2^-e."""
    mx = float(np.abs(w[np.isfinite(w)]).max()) if w.size else 0.0
    if mx == 0.0:
        return 1.0
    return 2.0 ** -(14 - math.frexp(mx)[1])


def hi_only(w, hm):
    """The operand a flavour would use if it dropped its lo products: tf32 hi (HM 0) or fp16 hi of w * 2^e (HM 1, 2)."""
    w = np.asarray(w, np.float32)
    if hm == 0:
        b = w.view(np.uint32).astype(np.uint64)
        b = ((b + 0x1000) & 0xFFFFE000).astype(np.uint32)
        return b.view(np.float32).astype(np.float64)
    inv = weight_split16(w)
    return (w / inv).astype(np.float16).astype(np.float64) * inv


def lif64(u, prm, T):
    """fp64 LIF^T chain from the zero state of the pre-activation u [R, N]; prm = [4, N] clamped."""
    p = {k: torch.from_numpy(prm[i].astype(np.float64)) for i, k in
         enumerate(("membrane_decay", "threshold_adapt", "refractory_decay", "threshold_base"))}
    return orc.lif_chain(torch.from_numpy(np.asarray(u, np.float64)), p, T).numpy()


def lif_slope(u, prm, T, h=1e-5):
    return np.abs(lif64(u + h, prm, T) - lif64(u - h, prm, T)) / (2 * h)


def gelu64(u):
    return 0.5 * u * (1.0 + np.vectorize(math.erf)(u / math.sqrt(2.0)))


def edge_rows(c):
    """Per edge row r = pt * kk + j: the point row and the global neighbour row (patch0 + idx[pt, j])."""
    R, kk, M = c["R"], c["kk"], c["mpts"]
    r = c["rows"] if c.get("rows") is not None else np.arange(R)
    pt = r // kk
    nb = (pt // M) * M + c["idx"][pt, r % kk]
    return pt, nb


def reference(c, w=None):
    """float64 result and bound of case c (numpy arrays; w overrides the weights, for the sensitivity tests)."""
    w = np.asarray(c["w"] if w is None else w, np.float64)
    x = np.asarray(c["x"], np.float64)
    R, K, N = c["R"], c["K"], c["N"]
    if c.get("amode", A_PLAIN) == A_EDGECAT:
        pt, nb = edge_rows(c)
        F = np.asarray(c["F"], np.float64)
        x = np.concatenate([F[nb] - F[pt], F[nb]], 1)
    elif c.get("amode", A_PLAIN) == A_ATTNIN:
        pt, nb = edge_rows(c)
        x = np.asarray(c["q"], np.float64)[pt] - np.asarray(c["kf"], np.float64)[nb] + x
    acc = x @ w.T
    S = np.abs(x) @ np.abs(w).T
    hm = c["hm"]
    kstep = 16 if hm in (1, 2, 3) else 8
    # SIMT engine: fp32 FFMA, one rounding per k step: the worst-case sequential-sum bound (K + 2) * 2^-24
    eps_op = (K + 2) * 2.0 ** -24 if hm == "simt" else EPS_OP[hm]
    eps = (eps_op + 4.0 * math.sqrt(K / kstep) * 2.0 ** -24) * S
    if hm in (1, 2, 3):
        eps = eps + 2.0 ** -25 * weight_split16(np.asarray(c["w"], np.float32)) * np.abs(x).sum(1, keepdims=True)
    if c.get("edge_bias"):
        pt, nb = edge_rows(c)
        eb = np.asarray(c["q"], np.float64)[pt] - np.asarray(c["kf"], np.float64)[nb]
        acc = acc + eb
        eps = eps + 2.0 ** -23 * (np.abs(np.asarray(c["q"], np.float64)[pt]) + np.abs(np.asarray(c["kf"], np.float64)[nb]))
    if c.get("bias") is not None:
        acc = acc + c["bias"]
    scale = np.ones(N) if c.get("scale") is None else np.asarray(c["scale"], np.float64)
    shift = np.zeros(N) if c.get("shift") is None else np.asarray(c["shift"], np.float64)
    u = acc * scale + shift
    eps_u = np.abs(scale) * (eps + 2.0 ** -22 * np.abs(acc)) + 2.0 ** -22 * np.abs(shift)
    act = c["act"]
    if act == ACT_LIF:
        y = lif64(u, c["prm"], c["T"])
        chain = LT_BOUND if c.get("table") else (EPS_FAST_MUFU if c.get("fast_chain") else EPS_MUFU)
        tol = chain + lif_slope(u, c["prm"], c["T"]) * eps_u
    elif act == ACT_LEAKY:
        y = np.where(u >= 0, u, 0.2 * u)
        tol = eps_u + 2.0 ** -23 * np.abs(u)
    elif act == ACT_GELU:
        y = gelu64(u)
        tol = 1.2 * eps_u + 2.0 ** -21 * np.abs(u) + 1e-7
    else:
        y = u
        tol = eps_u
    if c.get("residual") is not None:
        y = y + c["residual"]
        tol = tol + 2.0 ** -23 * np.abs(y)
    tol = tol + 2.0 ** -24 * np.abs(y)                    # fp32 store
    if c.get("out_fmt"):                                  # fp16 plane(s) of y * 2^13: rounding of the stored format
        tol = tol + (2.0 ** -11 * np.abs(y) if c["out_fmt"] == 2 else 2.0 ** -22 * np.abs(y))
    if c.get("group"):
        g = c["group"]
        y, tol = y.reshape(-1, g, N).max(1), tol.reshape(-1, g, N).max(1)
    if c.get("pool_M"):
        pT, pM = c["pool_T"], c["pool_M"]
        y = y.reshape(-1, pM, pT, N).max(1).reshape(-1, N)
        tol = tol.reshape(-1, pM, pT, N).max(1).reshape(-1, N)
    if c.get("at_pos") is not None:
        y, tol = attention_tail(c, y, tol)
    return y, tol


def attention_tail(c, y, eps_y):
    """softmax over each point's kk edges of y / at_sqrt, then sum_j a_j (v[nb_j] + pos[e_j])."""
    kk, N = c["kk"], c["N"]
    P = c["R"] // kk
    pt, nb = edge_rows(c)
    e = c["rows"] if c.get("rows") is not None else np.arange(c["R"])
    if c.get("at_pid") is not None:
        e = c["at_pid"][e]
    vp = np.asarray(c["at_v"], np.float64)[nb, :N] + np.asarray(c["at_pos"], np.float64)[e]
    z = (y / c["at_sqrt"]).reshape(P, kk, N)
    a = np.exp(z - z.max(1, keepdims=True))
    a /= a.sum(1, keepdims=True)
    vp = vp.reshape(P, kk, N)
    out = (a * vp).sum(1)
    tol = (a * np.abs(vp - out[:, None, :]) * eps_y.reshape(P, kk, N)).sum(1) / c["at_sqrt"] + 2.0 ** -20 * (a * np.abs(vp)).sum(1)
    return out, tol


# ----------------------------------------------------------------------------------------- case builders (host, seeded)
def neuron_params(N, rng):
    """Distinct clamped parameters per channel, thresholds spread over [0.3, 1.5]."""
    return np.stack([rng.uniform(0.1, 0.99, N), rng.uniform(0.001, 0.1, N), rng.uniform(0.1, 0.95, N),
                     rng.uniform(0.3, 1.5, N)]).astype(np.float32)


def spikes(R, K, rng):
    """Soft-spike inputs in [0, 0.6995]: exact zeros and the maximum included."""
    x = rng.uniform(0.0, 0.6995, (R, K)).astype(np.float32)
    x[rng.random((R, K)) < 0.1] = 0.0
    x[rng.random((R, K)) < 0.02] = np.float32(0.6995)
    return x


def weights(N, K, rng, span=True):
    """Rows scaled over 2^0 .. 2^-20 and one all-zero row, so the fp16 split meets weights far below the maximum."""
    w = rng.standard_normal((N, K)) / math.sqrt(K)
    if span:
        w *= 2.0 ** -(np.arange(N) % 21)[:, None].astype(np.float64)
        w[min(5, N - 1)] = 0.0
    return w.astype(np.float32)


def boundary_sweep(R, K, rng):
    """Offsets from theta0 that hit every table cell boundary y = 2|x| + 2 = 2^(e+1) and its fp32 neighbours, x = 0 +-, and
    |x| >= 255 (the exact-chain fallback)."""
    v = [0.0, -0.0, 1e-30, -1e-30, 254.99998, -254.99998, 255.0, -256.0, 400.0, -1000.0]
    for e in range(8):
        b = np.float32(2.0 ** e - 1.0)
        for s in (1.0, -1.0):
            v += [s * b, s * np.nextafter(b, np.float32(1e9))]
            if b > 0:
                v.append(s * np.nextafter(b, np.float32(0.0)))
    v = np.array(v, np.float32)
    x = rng.choice(v, size=(R, K)).astype(np.float32)
    x[: len(v) * 2 // K + 1].flat[: len(v)] = v
    return x


def graph(P, M, kk, ldi, rng):
    """Patch-local neighbour lists with duplicates and neighbours at both patch ends."""
    idx = rng.integers(0, M, (P, ldi)).astype(np.int32)
    idx[:, 0] = np.arange(P) % M
    idx[::3, 1] = 0
    idx[::3, 2] = M - 1
    idx[1::3, 1:4] = idx[1::3, 1:2]
    return idx


def make_case(name, seed=0):
    """The cases of CASES by name (inputs and expected instantiation)."""
    spec = dict(CASES[name])
    rng = np.random.default_rng(zlib.crc32(name.encode()) + seed)
    R, K, N = spec["R"], spec["K"], spec["N"]
    c = dict(spec, name=name)
    unit = spec.get("x_unit", False)
    c["x"] = spikes(R, K, rng) if unit else rng.standard_normal((R, K)).astype(np.float32)
    c["w"] = weights(N, K, rng, span=spec.get("span", True))
    c["bias"] = rng.standard_normal(N).astype(np.float32) * 0.1
    c["scale"] = rng.uniform(0.5, 2.0, N).astype(np.float32)
    c["shift"] = rng.standard_normal(N).astype(np.float32) * 0.1
    if spec["act"] == ACT_LIF:
        c["prm"] = neuron_params(N, rng)
        c["shift"] = c["shift"] + c["prm"][3]              # pre-activations around the thresholds
    if spec.get("sweep"):                                 # identity-like weights: u = x[r, n % K] + theta0[n]
        c["w"] = np.zeros((N, K), np.float32)
        c["w"][np.arange(N), np.arange(N) % K] = 1.0
        c["x"] = boundary_sweep(R, K, rng)
        c["bias"] = None
        c["scale"] = np.ones(N, np.float32)
        c["shift"] = c["prm"][3].copy()
    if spec.get("residual"):
        c["residual"] = rng.standard_normal((R, N)).astype(np.float32)
    if spec.get("kk"):
        kk, M = spec["kk"], spec["mpts"]
        P = R // kk
        c["idx"] = graph(P, M, kk, spec.get("ldi", kk), rng)
        c["ldi"] = spec.get("ldi", kk)
        if spec.get("edge_bias") or spec.get("amode") == A_ATTNIN:
            c["q"] = rng.standard_normal((P, N)).astype(np.float32) * 0.5
            c["kf"] = rng.standard_normal((P, N)).astype(np.float32) * 0.5
        if spec.get("amode") == A_EDGECAT:
            c["F"] = rng.standard_normal((P, K // 2)).astype(np.float32)
        if spec.get("attn"):
            c["act"] = ACT_NONE
            c["at_v"] = rng.standard_normal((P, N)).astype(np.float32)
            pos = spikes(R, N, rng)
            pf = spec.get("pos_fmt", 2 if spec.get("fast") else 0)
            if pf:                                    # the reference reads the value the planes encode
                pos = planes_decode(planes_encode(pos, pf), pf, R, N)
            if spec.get("pid"):                       # pos held once per distinct pair: U rows, read through at_pid
                U = R // 3
                c["at_pid"] = rng.integers(0, U, R).astype(np.int32)
                c["at_pid"][1::5] = c["at_pid"][::5][: len(c["at_pid"][1::5])]     # duplicates, also within a point
                pos[U:] = np.nan                      # rows past the pairs: never read
            c["at_pos"] = pos
            c["at_sqrt"] = math.sqrt(N / 8)
    if spec.get("x_fmt"):
        c["x"] = planes_decode(planes_encode(c["x"], spec["x_fmt"]), spec["x_fmt"], R, K)
    return c


def planes_encode(x, fmt):
    """fp16 hi (and lo) planes of x * 2^13, hi plane first."""
    xs = np.asarray(x, np.float64) * 8192.0
    hi = xs.astype(np.float16)
    if fmt == 2:
        return hi
    lo = (xs - hi.astype(np.float64)).astype(np.float16)
    return np.concatenate([hi.ravel(), lo.ravel()])


def planes_decode(h, fmt, R, C):
    h = np.asarray(h, np.float16).ravel()
    v = h[: R * C].astype(np.float64)
    if fmt == 1:
        v = v + h[R * C: 2 * R * C].astype(np.float64)
    return (v / 8192.0).reshape(R, C).astype(np.float32)


# name -> (mode, shapes, flavour switches, expected instantiation).  hm: operand format of the bound (see the module doc).
T2 = "gemm_tc2_kernel<%s>"
CASES = {
    # ---- 2-CTA engine, 3xTF32 (splitter) path
    "tc2_plain_3xtf32": dict(mode="tc", R=4096 + 77, K=960, N=256, act=ACT_NONE, hm=0, lda=968, ldc=264, kernel=T2 % "0,0,1,0,0,2"),
    "tc2_residual": dict(mode="tc", R=4096, K=64, N=512, act=ACT_NONE, hm=0, residual=True, kernel=T2 % "0,1,1,0,0,2"),
    "tc2_leaky": dict(mode="tc", R=5000, K=192, N=256, act=ACT_LEAKY, hm=0, kernel=T2 % "1,0,1,0,0,2"),
    "tc2_lif_mufu": dict(mode="tc", R=4096 * 5 + 5, K=512, N=768, act=ACT_LIF, T=4, hm=0, ldc=776, kernel=T2 % "3,0,1,0,0,2"),
    "tc2_lif_table_sweep": dict(mode="tc", R=8192, K=64, N=768, act=ACT_LIF, T=4, hm=0, table=True, sweep=True,
                                kernel=T2 % "3,0,1,0,1,2"),
    "tc2_pool_3xtf32": dict(mode="tc", R=7 * 100 * 8, K=960, N=256, act=ACT_LEAKY, hm=0, pool_T=7, pool_M=100, kernel=T2 % "1,4,1,0,0,2"),
    "tc2_attn_3xtf32_k12": dict(mode="tc", R=12 * 100 * 4, K=128, N=256, act=ACT_NONE, hm=0, kk=12, mpts=100, ldi=24, attn=True,
                                kernel=T2 % "0,3,12,0,0,2"),
    # ---- fp16x3, split in the kernel (HM 1): fp32 spike inputs
    "tc2_hm1_plain": dict(mode="tc", R=4096, K=256, N=256, act=ACT_NONE, hm=1, x_unit=True, kernel=T2 % "0,0,1,1,0,2"),
    "tc2_hm1_lif": dict(mode="tc", R=4096 + 200, K=512, N=1536, act=ACT_LIF, T=4, hm=1, x_unit=True, kernel=T2 % "3,0,1,1,0,2"),
    "tc2_hm1_lif_edge": dict(mode="tc", R=18 * 100 * 3, K=256, N=256, act=ACT_LIF, T=4, hm=1, x_unit=True, kk=18, mpts=100,
                             edge_bias=True, kernel=T2 % "3,2,1,1,0,2"),
    "tc2_hm1_pool": dict(mode="tc", R=7 * 100 * 8, K=960, N=768, act=ACT_LEAKY, hm=1, x_unit=True, pool_T=7, pool_M=100,
                         kernel=T2 % "1,4,1,1,0,2"),
    "tc2_hm1_attn_k18": dict(mode="tc", R=18 * 100 * 3, K=256, N=256, act=ACT_NONE, hm=1, x_unit=True, kk=18, mpts=100, attn=True,
                             kernel=T2 % "0,3,18,1,0,2"),
    # ---- fp16 (hi, lo) planes in (HM 2)
    "tc2_hm2_plain": dict(mode="tc", R=4096, K=256, N=512, act=ACT_NONE, hm=2, x_unit=True, x_fmt=1, tc2_any_rows=True,
                          kernel=T2 % "0,0,1,2,0,2"),
    "tc2_hm2_lif_planes_out": dict(mode="tc", R=1024, K=512, N=1536, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1,
                                   y2=True, tc2_any_rows=True, kernel=T2 % "3,0,1,2,0,2"),
    "tc2_hm2_lif_table": dict(mode="tc", R=4095, K=256, N=768, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1, table=True,
                              tc2_any_rows=True, kernel=T2 % "3,0,1,2,1,2"),
    "tc2_hm2_lif_edge": dict(mode="tc", R=24 * 100 * 2, K=256, N=256, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, kk=24, mpts=100,
                             edge_bias=True, kernel=T2 % "3,2,1,2,0,2"),
    "tc2_hm2_lif_edge_table": dict(mode="tc", R=12 * 100 * 4, K=512, N=512, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1,
                                   kk=12, mpts=100, edge_bias=True, table=True, kernel=T2 % "3,2,1,2,1,2"),
    "tc2_hm2_pool": dict(mode="tc", R=7 * 100 * 8, K=960, N=256, act=ACT_LEAKY, hm=2, x_unit=True, x_fmt=1, pool_T=7, pool_M=100,
                         kernel=T2 % "1,4,1,2,0,2"),
    "tc2_hm2_attn_k24_pos_planes": dict(mode="tc", R=24 * 100 * 2, K=256, N=256, act=ACT_NONE, hm=2, x_unit=True, x_fmt=1, kk=24,
                                        mpts=100, attn=True, pos_fmt=1, kernel=T2 % "0,3,24,2,0,2"),
    "tc2_hm2_rdev_in_tile": dict(mode="tc", R=8192, K=256, N=256, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1, table=True,
                                 R_dev=5000, kernel=T2 % "3,0,1,2,1,2"),
    "tc2_hm2_rdev_tile_short": dict(mode="tc", R=8192, K=256, N=256, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1,
                                    R_dev=8192 - 256, kernel=T2 % "3,0,1,2,0,2"),
    # ---- single-CTA flavour (N = 128) on planes
    "tc2_cg1_lif": dict(mode="tc", R=1024 + 100, K=128, N=128, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1,
                        tc2_any_rows=True, kernel=T2 % "3,0,1,2,0,1"),
    "tc2_cg1_lif_table": dict(mode="tc", R=4096, K=128, N=128, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1, table=True,
                              tc2_any_rows=True, kernel=T2 % "3,0,1,2,1,1"),
    "tc2_cg1_plain": dict(mode="tc", R=4096, K=128, N=128, act=ACT_NONE, hm=2, x_unit=True, x_fmt=1, kernel=T2 % "0,0,1,2,0,1"),
    "tc2_cg1_lif_edge_table": dict(mode="tc", R=12 * 100 * 4, K=128, N=128, act=ACT_LIF, T=4, hm=2, x_unit=True, x_fmt=1, out_fmt=1,
                                   kk=12, mpts=100, edge_bias=True, table=True, kernel=T2 % "3,2,1,2,1,1"),
    "tc2_cg1_attn_k12": dict(mode="tc", R=12 * 100 * 4, K=128, N=128, act=ACT_NONE, hm=2, x_unit=True, x_fmt=1, kk=12, mpts=100,
                             attn=True, pos_fmt=1, kernel=T2 % "0,3,12,2,0,1"),
    # ---- fast mode: one fp16 plane (HM 3), compact single-pass TF32 (HM 4)
    "fast_hm3_lif_table": dict(mode="fast", R=4096 * 2, K=256, N=512, act=ACT_LIF, T=4, hm=3, x_unit=True, x_fmt=2, out_fmt=2,
                               fast=True, table=True, kernel=T2 % "3,0,1,3,1,2"),
    "fast_hm3_lif_mufu": dict(mode="fast", R=4096, K=256, N=256, act=ACT_LIF, T=4, hm=3, x_unit=True, x_fmt=2, out_fmt=2,
                              fast=True, fast_chain=True, kernel=T2 % "3,0,1,3,0,2"),
    "fast_hm3_edge_table_cg1": dict(mode="fast", R=18 * 100 * 3, K=128, N=128, act=ACT_LIF, T=4, hm=3, x_unit=True, x_fmt=2, out_fmt=2,
                                    fast=True, table=True, kk=18, mpts=100, edge_bias=True, kernel=T2 % "3,2,1,3,1,1"),
    "fast_hm3_pool": dict(mode="fast", R=7 * 100 * 8, K=960, N=768, act=ACT_LEAKY, hm=3, x_unit=True, x_fmt=2, fast=True, pool_T=7,
                          pool_M=100, kernel=T2 % "1,4,1,3,0,2"),
    "fast_hm3_attn_k24": dict(mode="fast", R=24 * 100 * 2, K=256, N=256, act=ACT_NONE, hm=3, x_unit=True, x_fmt=2, fast=True, kk=24,
                              mpts=100, attn=True, kernel=T2 % "0,3,24,3,0,2"),
    "fast_hm4_lif_table": dict(mode="fast", R=4096 + 3, K=64, N=768, act=ACT_LIF, T=6, hm=4, fast=True, table=True,
                               kernel=T2 % "3,0,1,4,1,2"),
    "fast_hm4_lif_cg1": dict(mode="fast", R=4096, K=64, N=128, act=ACT_LIF, T=4, hm=4, fast=True, fast_chain=True,
                             kernel=T2 % "3,0,1,4,0,1"),
    "fast_hm4_plain": dict(mode="fast", R=4096, K=2048, N=1024, act=ACT_NONE, hm=4, lda=2056, kernel=T2 % "0,0,1,4,0,2"),
    # ---- single-CTA tensor-core engine (gemm_tc): row counts below the 2-CTA engine's, N = 128, GELU
    "tc_lif_n128": dict(mode="tc", R=1500, K=192, N=128, act=ACT_LIF, T=4, hm=0, kernel="gemm_tc_kernel<3,0,1>"),
    "tc_gelu": dict(mode="tc", R=2048, K=512, N=384, act=ACT_GELU, hm=0, kernel="gemm_tc_kernel<2,0,1>"),
    "tc_plain_tf32": dict(mode="tf32", R=1024, K=64, N=128, act=ACT_NONE, hm=4, ldc=136, kernel="gemm_tc_kernel<0,0,1>"),
    "tc_lif_edge": dict(mode="tc", R=12 * 100 * 2, K=128, N=128, act=ACT_LIF, T=4, hm=0, kk=12, mpts=100, edge_bias=True,
                        kernel="gemm_tc_kernel<3,2,1>"),
    # ---- SIMT only where SIMT is the only engine for the flavour
    "simt_edgecat_group32": dict(mode="tc", R=32 * 64, K=128, N=128, act=ACT_LEAKY, hm="simt", amode=A_EDGECAT, kk=32, mpts=64,
                                 group=32, kernel="gemm_simt_kernel<1,1,32,1>"),
    "simt_attnin_lif": dict(mode="fp32", R=16 * 100, K=128, N=128, act=ACT_LIF, T=4, hm="simt", amode=A_ATTNIN, kk=16, mpts=100,
                            x_unit=True, kernel="gemm_simt_kernel<2,3,0,1>"),
}


def _more_cases():
    """The remaining instantiations, one case each: every fused-attention (neighbour count, operand format, CTA group), the
    edge-bias and LIF flavours of the fast formats, the single-CTA engine's other epilogues and the SIMT engine's."""
    out = {}
    rows = {12: 4800, 18: 5400, 24: 4800}
    fmt = {0: dict(mode="tc"), 1: dict(mode="tc", x_unit=True), 2: dict(mode="tc", x_unit=True, x_fmt=1, pos_fmt=1),
           3: dict(mode="fast", x_unit=True, x_fmt=2, fast=True)}
    for kk in (12, 18, 24):
        for hm in (0, 1, 2, 3):
            for cg in ((2, 1) if hm >= 2 else (2,)):
                key = T2 % "0,3,%d,%d,0,%d" % (kk, hm, cg)
                out["tc2_attn_k%d_hm%d_cg%d" % (kk, hm, cg)] = dict(fmt[hm], R=rows[kk], K=128, N=128 * cg, act=ACT_NONE, hm=hm, kk=kk,
                                                                    mpts=100, ldi=24, attn=True, kernel=key)
        out["tc_attn_k%d" % kk] = dict(mode="tc", R=kk * 100 * (1 if kk == 24 else 2), K=128, N=256, act=ACT_NONE, hm=0, kk=kk, mpts=100,
                                       attn=True, kernel="gemm_tc_kernel<0,3,%d>" % kk)
    lif = dict(act=ACT_LIF, T=4)
    edge = dict(kk=12, mpts=100, edge_bias=True, R=4800)
    f3 = dict(mode="fast", hm=3, x_unit=True, x_fmt=2, out_fmt=2, fast=True, K=128)
    out.update({
        "tc2_edge_3xtf32": dict(**lif, **edge, mode="tc", K=256, N=256, hm=0, kernel=T2 % "3,2,1,0,0,2"),
        "tc2_cg1_edge_planes": dict(**lif, **edge, mode="tc", K=128, N=128, hm=2, x_unit=True, x_fmt=1, kernel=T2 % "3,2,1,2,0,1"),
        "fast_edge_cg1_mufu": dict(**lif, **edge, **f3, N=128, fast_chain=True, kernel=T2 % "3,2,1,3,0,1"),
        "fast_edge_mufu": dict(**lif, **edge, **f3, N=256, fast_chain=True, kernel=T2 % "3,2,1,3,0,2"),
        "fast_edge_table": dict(**lif, **edge, **f3, N=256, table=True, kernel=T2 % "3,2,1,3,1,2"),
        "fast_hm3_cg1_mufu": dict(**lif, **f3, R=4096, N=128, fast_chain=True, kernel=T2 % "3,0,1,3,0,1"),
        "fast_hm3_cg1_table": dict(**lif, **f3, R=4096 + 31, N=128, table=True, kernel=T2 % "3,0,1,3,1,1"),
        "fast_hm4_mufu": dict(**lif, mode="fast", R=4096, K=64, N=256, hm=4, fast=True, fast_chain=True, kernel=T2 % "3,0,1,4,0,2"),
        "fast_hm4_cg1_table": dict(**lif, mode="fast", R=4096, K=64, N=128, hm=4, fast=True, table=True, kernel=T2 % "3,0,1,4,1,1"),
        "tc_residual": dict(mode="tc", R=2048, K=128, N=256, act=ACT_NONE, hm=0, residual=True, kernel="gemm_tc_kernel<0,1,1>"),
        "tc_leaky": dict(mode="tc", R=2048 + 7, K=128, N=384, act=ACT_LEAKY, hm=0, kernel="gemm_tc_kernel<1,0,1>"),
        "simt_plain": dict(mode="tc", R=500, K=256, N=2048, act=ACT_NONE, hm="simt", kernel="gemm_simt_kernel<0,0,0,1>"),
        "simt_leaky": dict(mode="tc", R=300, K=64, N=256, act=ACT_LEAKY, hm="simt", kernel="gemm_simt_kernel<0,1,0,1>"),
        "simt_gelu": dict(mode="tc", R=200, K=512, N=256, act=ACT_GELU, hm="simt", kernel="gemm_simt_kernel<0,2,0,1>"),
        "simt_lif_precise": dict(**lif, mode="fp32", R=700, K=192, N=128, hm="simt", kernel="gemm_simt_kernel<0,3,0,1>"),
        "simt_lif_reduced": dict(**lif, mode="tc", R=700, K=192, N=128, hm="simt", fast_chain=True, kernel="gemm_simt_kernel<0,3,0,0>"),
        "simt_edgecat_any_k": dict(mode="fp32", R=18 * 100, K=128, N=128, act=ACT_LEAKY, hm="simt", amode=A_EDGECAT, kk=18, mpts=100,
                                   kernel="gemm_simt_kernel<1,1,0,1>"),
        "simt_attnin_reduced": dict(**lif, mode="tc", R=16 * 100, K=128, N=128, hm="simt", amode=A_ATTNIN, kk=16, mpts=100,
                                    fast_chain=True, kernel="gemm_simt_kernel<2,3,0,0>"),
    })
    return out


CASES.update(_more_cases())
CASES["tc2_attn_pid_k24_hm2"] = dict(mode="tc", R=4800, K=128, N=256, act=ACT_NONE, hm=2, x_unit=True, x_fmt=1, pos_fmt=1, kk=24,
                                     mpts=100, attn=True, pid=True, kernel=T2 % "0,3,24,2,0,2")

NUM_SMS = 148


def tc2_grid(spec, R=None):
    """(tile rows, channel tiles, total tiles, CTA pairs) of a 2-CTA-engine case, by launch_gemm_tc2's rules: tile rows 256
    (whole points for the fused attention tail), grid = min(tiles, 148 / CG) pairs, rounded down to a multiple of the channel
    tiles when the layer's LIF table is loaded (a pair then keeps one channel block)."""
    R = spec["R"] if R is None else R
    cg = 2 if spec["N"] % 256 == 0 else 1
    tr = (256 // spec["kk"]) * spec["kk"] if spec.get("attn") else 256
    m_tiles = spec["N"] // (128 * cg)
    total = -(-R // tr) * m_tiles
    pairs = min(total, NUM_SMS // cg)
    if spec.get("table"):
        pairs = pairs // m_tiles * m_tiles
    return tr, m_tiles, total, pairs


def _walk_cases():
    """Each 2-CTA-engine case again at a row count where every CTA (pair) walks >= 3 tiles: both accumulator buffers, both
    barrier parities and the next-tile prefetch of the persistent loop.  A partial last tile where the rows allow it."""
    out = {}
    for name, spec in CASES.items():
        if not spec["kernel"].startswith("gemm_tc2") or spec.get("R_dev"):
            continue
        tr, m_tiles, _, _ = tc2_grid(spec)
        cg = 2 if spec["N"] % 256 == 0 else 1
        pairs = NUM_SMS // cg
        if spec.get("table"):
            pairs = pairs // m_tiles * m_tiles
        rows = (-(-3 * pairs // m_tiles) + 1) * tr
        unit = spec["kk"] * spec["mpts"] if spec.get("kk") else (spec["pool_T"] * spec["pool_M"] if spec.get("pool_M") else 1)
        rows = -(-rows // unit) * unit - (37 if unit == 1 else 0)
        out[name + "_walk"] = dict(spec, R=rows)
    return out


CASES.update(_walk_cases())


# ----------------------------------------------------------------------------------------- CPU: the reference and its sensitivity
def _oracle_fn_block_pieces(seed=3):
    """lif_chain(bn(conv(x))) of the oracle's fn block, on one small random block."""
    g = torch.Generator().manual_seed(seed)
    D, Cin, M = 128, 64, 20
    sd = {"t.fc1.0.weight": torch.randn(D, Cin, 1, generator=g) / 8, "t.fc1.0.bias": torch.randn(D, generator=g) * 0.1,
          "t.fc1.1.weight": torch.rand(D, generator=g) + 0.5, "t.fc1.1.bias": torch.randn(D, generator=g) * 0.1,
          "t.fc1.1.running_mean": torch.randn(D, generator=g) * 0.1, "t.fc1.1.running_var": torch.rand(D, generator=g) + 0.5,
          "t.snn1.membrane_decay": torch.rand(D, generator=g), "t.snn1.threshold_adapt": torch.rand(D, generator=g) * 0.2,
          "t.snn1.refractory_decay": torch.rand(D, generator=g), "t.snn1.threshold_base": torch.rand(D, generator=g) + 0.3}
    sd = {k: v.double() for k, v in sd.items()}
    f = torch.randn(2, Cin, M, generator=g).double()
    out = orc.lif_chain(orc._conv_bn(sd, "t.fc1", f), orc.neuron_params(sd, "t.snn1"), 4)
    return sd, f, out


def test_reference_matches_oracle_conv_bn_lif():
    sd, f, out = _oracle_fn_block_pieces()
    inv = 1.0 / torch.sqrt(sd["t.fc1.1.running_var"] + 1e-5)
    sc = (sd["t.fc1.1.weight"] * inv).numpy()
    sh = (sd["t.fc1.1.bias"] - sd["t.fc1.1.running_mean"] * sd["t.fc1.1.weight"] * inv).numpy()
    prm = np.stack([np.clip(sd["t.snn1.membrane_decay"].numpy(), 0.1, 0.99), np.clip(sd["t.snn1.threshold_adapt"].numpy(), 0.001, 0.1),
                    np.clip(sd["t.snn1.refractory_decay"].numpy(), 0.1, 0.95), sd["t.snn1.threshold_base"].numpy()])
    x = f.permute(0, 2, 1).reshape(-1, 64).numpy()
    c = dict(x=x, w=sd["t.fc1.0.weight"][:, :, 0].numpy(), R=x.shape[0], K=64, N=128, hm=0, act=ACT_LIF, T=4,
             bias=sd["t.fc1.0.bias"].numpy(), scale=sc, shift=sh, prm=prm)
    y, _ = reference(c)
    np.testing.assert_allclose(y, out.permute(0, 2, 1).reshape(-1, 128).numpy(), rtol=0, atol=1e-12)


def test_reference_matches_oracle_attention_and_edgeconv():
    """The attention tail and the EdgeConv loader restated against the oracle's fn_block / graph_feature formulas."""
    rng = np.random.default_rng(4)
    B, M, kk, D = 2, 20, 6, 16
    idx = torch.from_numpy(rng.integers(0, M, (B, M, kk)))
    logits = torch.from_numpy(rng.standard_normal((B, D, M, kk)))
    v = torch.from_numpy(rng.standard_normal((B, D, M)))
    pos = torch.from_numpy(rng.standard_normal((B, D, M, kk)))
    H = 1
    vg = orc.gather_points(v.permute(0, 2, 1).contiguous(), idx).permute(0, 3, 1, 2)
    attn = torch.softmax(logits.view(B, H, D, M, kk) / np.sqrt(D), dim=-1)
    want = torch.einsum("bhcnk,bhcnk->bhcn", attn, vg.reshape(B, H, D, M, kk) + pos.view(B, H, D, M, kk)).reshape(B, D, M)
    c = dict(R=B * M * kk, N=D, kk=kk, mpts=M, idx=idx.reshape(B * M, kk).numpy().astype(np.int32), at_sqrt=math.sqrt(D),
             at_v=v.permute(0, 2, 1).reshape(B * M, D).numpy(), at_pos=pos.permute(0, 2, 3, 1).reshape(-1, D).numpy())
    y = logits.permute(0, 2, 3, 1).reshape(-1, D).numpy()
    got, _ = attention_tail(c, y, np.zeros_like(y))
    np.testing.assert_allclose(got, want.permute(0, 2, 1).reshape(-1, D).numpy(), rtol=0, atol=1e-12)
    # EdgeConv input cat(x_j - x_i, x_j) of graph_feature through edge_rows
    F = torch.from_numpy(rng.standard_normal((B, 8, M)))
    gf, _ = orc.graph_feature(F, kk, idx)
    pt, nb = edge_rows(c)
    Fr = F.permute(0, 2, 1).reshape(B * M, 8).numpy()
    mine = np.concatenate([Fr[nb] - Fr[pt], Fr[nb]], 1)
    np.testing.assert_allclose(mine, gf.permute(0, 2, 3, 1).reshape(-1, 16).numpy(), rtol=0, atol=0)


@pytest.mark.parametrize("name", ["tc2_lif_mufu", "tc2_hm1_lif", "tc2_hm2_lif_edge", "tc2_plain_3xtf32", "tc2_hm2_pool"])
def test_bound_catches_dropped_lo_products(name):
    """Every 3-product flavour: the same case computed with the hi product only deviates beyond the stated bound."""
    c = make_case(name)
    sl = slice(0, 512 if not c.get("pool_M") else 700 * 2)
    c = _rows(c, sl)
    ref, tol = reference(c)
    bad, _ = reference(c, w=hi_only(c["w"], c["hm"] if c["hm"] != 2 else 1))
    assert (np.abs(bad - ref) > tol).any(), (name, float((np.abs(bad - ref) / tol).max()))


@pytest.mark.parametrize("name", ["tc2_lif_mufu", "tc2_hm2_lif_table", "fast_hm3_lif_table", "fast_hm4_lif_table"])
def test_bound_catches_a_short_chain(name):
    c = _rows(make_case(name), slice(0, 256))
    ref, tol = reference(c)
    short, _ = reference(dict(c, T=c["T"] - 1))
    assert (np.abs(short - ref) > tol).any()


@pytest.mark.parametrize("name", ["tc2_pool_3xtf32", "tc2_hm1_pool", "fast_hm3_pool"])
def test_bound_catches_a_short_pool(name):
    c = _rows(make_case(name), slice(0, 7 * 100 * 2))
    ref, tol = reference(c)
    y, _ = reference(dict(c, pool_M=None))
    pT, pM = c["pool_T"], c["pool_M"]
    short = y.reshape(-1, pM, pT, c["N"])[:, : pM - 1].max(1).reshape(-1, c["N"])
    assert (np.abs(short - ref) > tol).any()


def _rows(c, sl):
    """The first rows of a case (whole patches / points for the row-structured flavours)."""
    c = dict(c)
    n = sl.stop
    for k in ("x", "residual", "at_pos"):
        if c.get(k) is not None:
            c[k] = c[k][:n]
    c["R"] = n
    return c


def test_every_two_cta_flavour_walks_three_tiles_per_pair():
    """Each 2-CTA-engine case has a twin on which every CTA pair of the persistent grid walks at least three tiles."""
    for name, spec in CASES.items():
        if spec["kernel"].startswith("gemm_tc2") and not spec.get("R_dev") and not name.endswith("_walk"):
            _, _, total, pairs = tc2_grid(CASES[name + "_walk"])
            assert total >= 3 * pairs, (name, total, pairs)


def test_sampled_rows_cover_every_tile():
    c = make_case("tc2_hm2_lif_edge_table_walk")
    sel, sub = checked_rows(c)
    tr = tc2_grid(c)[0]
    assert set(range(0, c["R"], tr)) <= set(sel.tolist()) and c["R"] - 1 in sel
    pt, nb = edge_rows(sub)
    np.testing.assert_array_equal(pt, sel // c["kk"])


def test_table_sweep_hits_every_cell_boundary():
    c = make_case("tc2_lif_table_sweep")
    off = np.unique(c["x"])
    for e in range(8):
        b = np.float32(2.0 ** e - 1.0)
        assert b in off and -b in off and np.nextafter(b, np.float32(1e9)) in off
    assert (np.abs(off) >= 255).any() and (off == 0).any()


# ----------------------------------------------------------------------------------------- GPU
KERNEL_FAMILIES = ("gemm_tc2_kernel", "gemm_tc_kernel", "gemm_simt_kernel")


def kernel_key(name):
    """'gemm_tc2_kernel<3,0,1,2,1,2>' from a demangled or mangled kernel name (None for other kernels)."""
    import re
    m = re.search(r"(gemm_(?:tc2|tc|simt)_kernel)<([^>]*)>", name)
    if m:
        args = [a.strip() for a in m.group(2).split(",")]
        args = ["1" if a == "true" else "0" if a == "false" else a.rstrip("u") for a in args]
        return "%s<%s>" % (m.group(1), ",".join(args))
    m = re.search(r"(gemm_(?:tc2|tc|simt)_kernel)I((?:L[ib]\d+E)+)E", name)
    if m:
        return "%s<%s>" % (m.group(1), ",".join(re.findall(r"L[ib](\d+)E", m.group(2))))
    return None


def profiled_kernels(run):
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    with tempfile.NamedTemporaryFile(suffix=".json") as f:
        prof.export_chrome_trace(f.name)
        ev = json.load(open(f.name))["traceEvents"]
    return [k for k in (kernel_key(e["name"]) for e in ev if e.get("cat") == "kernel") if k]


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    from sapcu_b200 import _native as N
    return N.lib()


def _dev(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV) if a is not None else None


def run_case(lib, c):
    """Launch case c through sapcu_gemm_case; returns (result rows as float64 numpy, kernels, output buffers for checks)."""
    from sapcu_b200 import _native as N
    R, K, N_ = c["R"], c["K"], c["N"]
    a = N.GemmCaseArgs()
    keep = []
    hp = lambda arr: (keep.append(np.ascontiguousarray(arr, np.float32)), keep[-1].ctypes.data)[1] if arr is not None else None
    a.amode, a.act, a.T, a.use_table = c.get("amode", A_PLAIN), c["act"], c.get("T", 0), int(bool(c.get("table")))
    a.R, a.K, a.N = R, K, N_
    a.h_w, a.h_bias, a.h_scale, a.h_shift = hp(c["w"]), hp(c.get("bias")), hp(c.get("scale")), hp(c.get("shift"))
    a.h_params4 = hp(c.get("prm"))
    xf = c.get("x_fmt", 0)
    lda = c.get("lda", K)
    if xf:
        xbuf = _dev(planes_encode(c["x"], xf))
        lda = K
    else:
        xp = np.full((R, lda), np.nan, np.float32)
        xp[:, :K] = c["x"]
        xbuf = _dev(xp)
    a.d_x, a.lda, a.x_format, a.x_unit, a.fast = xbuf.data_ptr(), lda, xf, int(bool(c.get("x_unit"))), int(bool(c.get("fast")))
    of = c.get("out_fmt", 0)
    ldc = c.get("ldc", N_)
    pad = 64
    if c.get("attn"):
        ybuf = torch.full(((R // c["kk"]) + pad, ldc), float("nan"), device=DEV)
    elif of:
        ybuf = torch.full((R * N_ * (2 if of == 1 else 1) + 2 * pad,), float("nan"), dtype=torch.float16, device=DEV)
        ldc = N_
    elif c.get("group"):
        ybuf = torch.full((R // c["group"] + pad, ldc), float("nan"), device=DEV)
    else:
        ybuf = torch.full((R + pad, ldc), float("nan"), device=DEV)
    a.d_y, a.ldc, a.out_h2 = ybuf.data_ptr(), ldc, int(bool(of))
    y2 = torch.full((R + pad, N_), float("nan"), device=DEV) if c.get("y2") else None
    a.d_y2 = y2.data_ptr() if y2 is not None else None
    res = _dev(c.get("residual"))
    a.d_residual, a.ldr = (res.data_ptr(), N_) if res is not None else (None, 0)
    bufs = [xbuf, ybuf, y2, res]
    if c.get("kk"):
        idx = _dev(c["idx"]); bufs.append(idx)
        a.d_idx, a.ldi, a.kk, a.mpts = idx.data_ptr(), c["ldi"], c["kk"], c["mpts"]
        if c.get("q") is not None:
            q, kf = _dev(c["q"]), _dev(c["kf"]); bufs += [q, kf]
            a.d_q, a.d_kf, a.ldq = q.data_ptr(), kf.data_ptr(), N_
        a.edge_bias = int(bool(c.get("edge_bias")))
        if c.get("F") is not None:
            F = _dev(c["F"]); bufs.append(F)
            a.d_f, a.ldf, a.C = F.data_ptr(), K // 2, K // 2
        if c.get("attn"):
            v = _dev(c["at_v"]); bufs.append(v)
            pf = c.get("pos_fmt", 2 if c.get("fast") else 0)
            pos = _dev(planes_encode(c["at_pos"], pf)) if pf else _dev(c["at_pos"])
            bufs.append(pos)
            a.d_at_pos, a.d_at_v, a.at_ldv, a.at_sqrt, a.pos_h2 = pos.data_ptr(), v.data_ptr(), N_, c["at_sqrt"], int(bool(pf))
            if c.get("at_pid") is not None:
                pid = _dev(c["at_pid"]); bufs.append(pid)
                a.d_at_pid = pid.data_ptr()
    pool = None
    if c.get("pool_M"):
        pool = torch.full((R // c["pool_M"] + pad, N_), float("-inf"), device=DEV)
        a.d_pool, a.pool_T, a.pool_M = pool.data_ptr(), c["pool_T"], c["pool_M"]
    rdev = None
    if c.get("R_dev"):
        rdev = torch.tensor([c["R_dev"]], dtype=torch.int32, device=DEV)
        a.d_R_dev = rdev.data_ptr()
    a.tc2_any_rows, a.group = int(bool(c.get("tc2_any_rows"))), c.get("group", 0)
    nb = lib.sapcu_gemm_case_workspace_bytes(a)
    assert nb > 0
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    rc = []
    kern = profiled_kernels(lambda: rc.append(lib.sapcu_gemm_case(a, ws.data_ptr(), nb, MODES[c["mode"]], None)))
    N.check(rc[0], "gemm_case " + c["name"])
    torch.cuda.synchronize()
    assert lib.sapcu_device_status() == 0
    return dict(y=ybuf, y2=y2, pool=pool, kernels=kern, ldc=ldc, pad=pad, bufs=bufs)


def decode_output(c, out):
    R, N_ = c["R"], c["N"]
    if c.get("pool_M"):
        p = out["pool"].cpu().numpy()
        return p[: R // c["pool_M"]].astype(np.float64), p[R // c["pool_M"]:]
    y = out["y"]
    if c.get("out_fmt"):
        h = y.cpu().numpy()
        n = R * N_ * (2 if c["out_fmt"] == 1 else 1)
        return planes_decode(h[:n], c["out_fmt"], R, N_).astype(np.float64), h[n:]
    rows = R // c["kk"] if c.get("attn") else (R // c["group"] if c.get("group") else R)
    yy = y.cpu().numpy()
    tail = np.concatenate([yy[:rows, N_:].ravel(), yy[rows:].ravel()])
    return yy[:rows, :N_].astype(np.float64), tail


def checked_rows(c, n_rand=768, seed=0):
    """Output rows the fp64 reference is evaluated on, and the case restricted to the inputs they need.  Every output row for
    cases up to 20,000 rows; beyond that the first and last row of every tile, the last row and n_rand random rows (the
    sentinels around the output are checked in full either way)."""
    R = c["R"]
    if R <= 20000:
        return None, c
    tr = tc2_grid(c)[0]
    rng = np.random.default_rng(seed)
    starts = np.arange(0, R, tr)
    sel = np.unique(np.concatenate([starts, np.minimum(starts + tr - 1, R - 1), [R - 1], rng.integers(0, R, n_rand)]))
    if c.get("attn"):                                     # whole points: output row = point
        kk = c["kk"]
        out = np.unique(sel // kk)
        rows = (out[:, None] * kk + np.arange(kk)).ravel()
    elif c.get("pool_M"):                                 # whole patches: output rows = (patch, t)
        blk = c["pool_T"] * c["pool_M"]
        patches = np.unique(sel // blk)
        rows = (patches[:, None] * blk + np.arange(blk)).ravel()
        out = (patches[:, None] * c["pool_T"] + np.arange(c["pool_T"])).ravel()
    else:
        out = rows = sel
    sub = dict(c, R=len(rows), rows=rows, x=c["x"][rows])
    if c.get("residual") is not None:
        sub["residual"] = c["residual"][rows]
    return out, sub


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_flavour_against_fp64(lib, parity_log, name):
    c = make_case(name)
    out = run_case(lib, c)
    assert c["kernel"] in out["kernels"], (name, out["kernels"])
    assert all(k == c["kernel"] for k in out["kernels"]), (name, out["kernels"])
    got, tail = decode_output(c, out)
    if c.get("R_dev"):
        # the tiles that hold rows < R_dev are computed in full (from the capacity rows, like any other row); no later tile
        # is touched
        done = -(-c["R_dev"] // tc2_grid(c)[0]) * tc2_grid(c)[0]
        assert np.isnan(got[done:]).all(), "tiles past R_dev were written"
        got = got[:done]
        c = dict(c, R=done, x=c["x"][:done])
    sel, sub = checked_rows(c)
    if sel is not None:
        got = got[sel]
    ref, tol = reference(sub)
    if c.get("pool_M"):
        assert np.isneginf(tail).all(), "store outside the pooled rows"
    else:
        assert np.isnan(tail.astype(np.float32)).all(), "store outside the output"
    err = np.abs(got - ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(err == 0, 0.0, np.nan_to_num(err / tol, nan=np.inf))
    worst = np.unravel_index(np.argmax(ratio), ratio.shape)
    parity_log.record("gemm_flavours", **{name: dict(kernel=c["kernel"], max_abs=float(err.max()), max_err_over_tol=float(ratio.max()),
                                                     tol_at_max_abs=float(tol.flat[np.argmax(err)]))})
    assert ratio.max() <= 1.0, (name, "row %d col %d: got %r want %r tol %r" % (worst[0], worst[1], got[worst], ref[worst], tol[worst]),
                                "rows > tol: %s" % np.unique(np.nonzero(ratio > 1)[0])[:20])
    if c.get("y2"):
        y2 = out["y2"].cpu().numpy()
        assert np.isnan(y2[c["R"]:]).all()
        # the fp32 copy holds the spikes the planes encode, before the plane rounding
        np.testing.assert_allclose(y2[: c["R"]] if sel is None else y2[sel], got, rtol=0, atol=2.0 ** -22)


# Instantiations that no GemmArgs the forwards build can reach (listed, not deleted: removing them is a separate change)
UNREACHED = {}
COVERED = {spec["kernel"] for spec in CASES.values()}

_CHILD = r'''
import json, os, sys, copy
sys.path[:0] = [sys.argv[1], os.path.join(sys.argv[1], "oracle"), os.path.join(sys.argv[1], "tests")]
import torch
import sapcu_b200, sapcu_b200.synthetic as syn
from sapcu_b200 import _native as N
from sapcu_b200.fn import config as fc
from sapcu_b200.fd import config as dc
import sapcu_oracle as orc, oracle_c
from test_gemm_flavours import profiled_kernels
dev = "cuda:0"
cloud = syn.cloud(2048, seed=0, shape="sphere")
seeds = syn.seeds(cloud, 4, seed=1)
def models(yaml):
    cfn = copy.deepcopy(fc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fn.yaml")))
    cfd = copy.deepcopy(dc.load_config(os.path.join(sapcu_b200.CONFIG_DIR, "fd.yaml")))
    if not yaml:
        cfn["model"].update(k_values=[16, 10, 6], time_steps_enc=4)
        cfd["model"].update(k=18, k_scales=[4, 8, 12, 20], time_steps_enc=5)
    mfn, mfd = fc.get_model(cfn), dc.get_model(cfd, None)
    syn.init_weights(mfn, seed=100, stress=True); syn.init_weights(mfd, seed=200, stress=True)
    return mfn.to(dev), mfd.to(dev)
seen = set()
c64 = torch.from_numpy(cloud.astype("float64")).to(dev)
for yaml in (True, False):
    mfn, mfd = models(yaml)
    for B, M in ((48, 100), (48, 64)):
        gi = oracle_c.knn(cloud, seeds[:B], M)
        p = torch.from_numpy(orc.gather_center(cloud, seeds[:B], gi)).to(dev)
        gidx = torch.from_numpy(gi.astype("int32")).to(dev)
        for mode in sys.argv[2].split(","):
            for m in (mfn, mfd):
                m.set_mode(mode)
                seen.update(profiled_kernels(lambda: m(p)))
            # the pair schedule of the parity-grade mode (pair-row launches with device row counts, pid-indexed attention)
            seen.update(profiled_kernels(lambda: mfn.forward_indexed(p, c64, gidx)))
            N.check_device(mode)
json.dump(sorted(seen), open(sys.argv[3], "w"))
'''


@pytest.mark.gpu
def test_every_forward_instantiation_is_covered(lib, tmp_path):
    """fn (patch and cloud-indexed forwards) and fd in tc, fast and tf32 (yaml and non-yaml configs, M = 100 and 64; fast also
    without LIF tables): every GEMM
    instantiation they launch is one a case above targets, or is listed as unreached with a reason."""
    script = tmp_path / "child.py"
    script.write_text(_CHILD)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    seen = set()
    for modes, env in (("tc,fast,tf32", {}), ("fast", {"SAPCU_FAST_LIF_TABLES": "0"})):
        out = tmp_path / ("seen_%d.json" % len(seen))
        r = subprocess.run([sys.executable, str(script), root, modes, str(out)], capture_output=True, text=True,
                           env=dict(os.environ, **env), timeout=900)
        assert r.returncode == 0, r.stdout + r.stderr
        seen.update(json.load(open(out)))
    assert seen, "no GEMM kernel recorded"
    missing = sorted(k for k in seen if k not in COVERED)
    assert not missing, "launched by the forwards, no case: " + ", ".join(missing)
    assert not (set(UNREACHED) & seen), sorted(set(UNREACHED) & seen)
