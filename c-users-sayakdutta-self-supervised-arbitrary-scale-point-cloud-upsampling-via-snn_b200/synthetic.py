"""Seeded synthetic inputs for the parity suite and the benchmark (SURVEY.md section 8d).

  cloud(n, seed, shape)   points on a closed surface, bbox-normalised like generate.py:43-53 (fp64)
  seeds(cloud, ratio, seed)  S = ceil(ratio*N) seeds in the 0.011-0.015 band dense.cpp emits around the surface
  init_weights(model, seed, stress)  deterministic random weights for an fn/fd module (state_dict in place)
  sphere_mesh(level)      the icosphere of radius 0.5 that cloud(shape="sphere") samples (metrics tests and benchmark)

Everything is generated from numpy / torch CPU generators so the GPU box reproduces the same bits
without the reference checkout.
"""
import math

import numpy as np
import torch


def normalize_pointcloud(cloud):
    lo, hi = cloud.min(axis=0), cloud.max(axis=0)
    loc = (lo + hi) / 2
    scale = (hi - lo).max()
    return (cloud - loc) * (1.0 / scale if scale > 0 else 1.0), loc, scale


def cloud(n, seed=0, shape="sphere"):
    rng = np.random.default_rng(seed)
    if shape == "sphere":
        v = rng.normal(size=(n, 3))
        pts = 0.5 * v / np.linalg.norm(v, axis=1, keepdims=True)
    elif shape == "boxes":          # "ShapeNet-shaped": union of three boxes and a cylinder, surface samples
        parts = []
        per = [n // 4, n // 4, n // 4, n - 3 * (n // 4)]
        boxes = [((-0.5, -0.2, -0.1), (0.5, 0.2, 0.1)), ((-0.4, -0.15, 0.1), (-0.1, 0.15, 0.5)),
                 ((0.1, -0.15, 0.1), (0.4, 0.15, 0.35))]
        for (lo, hi), m in zip(boxes, per[:3]):
            lo, hi = np.array(lo), np.array(hi)
            p = rng.uniform(lo, hi, size=(m, 3))
            face = rng.integers(0, 6, size=m)
            ax = face % 3
            p[np.arange(m), ax] = np.where(face < 3, lo[ax], hi[ax])
            parts.append(p)
        m = per[3]
        th = rng.uniform(0, 2 * math.pi, size=m)
        z = rng.uniform(-0.45, 0.45, size=m)
        parts.append(np.stack([0.08 * np.cos(th), 0.3 + 0.08 * np.sin(th), z], axis=1))
        pts = np.concatenate(parts, axis=0)
    else:
        raise ValueError(shape)
    pts, _, _ = normalize_pointcloud(pts.astype(np.float64))
    return np.ascontiguousarray(pts)


def seeds(cloud_pts, ratio, seed=1):
    n = cloud_pts.shape[0]
    s = int(math.ceil(ratio * n))
    rng = np.random.default_rng(seed)
    u = rng.normal(size=(s, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    rho = rng.uniform(0.011, 0.015, size=(s, 1))
    return np.ascontiguousarray(cloud_pts[np.arange(s) % n] + u * rho)


def sphere_mesh(level=3):
    """Icosahedron subdivided `level` times (20 * 4**level faces), vertices on the sphere of radius 0.5 centred at the
    origin -> (vertices [V,3] float64, faces [F,3] int32).  Every face is wound counter-clockwise seen from outside, so
    (b-a)x(c-a) points outward.  cloud(n, shape="sphere") samples this sphere (up to its bounding-box normalisation, which
    moves the points by well under 1e-2 for n >= 1000)."""
    t = (1.0 + math.sqrt(5.0)) / 2.0
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], dtype=np.float64)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6],
                  [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10],
                  [8, 6, 7], [9, 8, 1]], dtype=np.int64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    for _ in range(level):
        nv, nf = v.shape[0], f.shape[0]
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
        e.sort(axis=1)
        uniq, inv = np.unique(e[:, 0] * nv + e[:, 1], return_inverse=True)
        mid = v[uniq // nv] + v[uniq % nv]
        v = np.concatenate([v, mid / np.linalg.norm(mid, axis=1, keepdims=True)])
        m01, m12, m20 = (nv + inv.reshape(3, nf))
        a, b, c = f[:, 0], f[:, 1], f[:, 2]
        f = np.concatenate([np.stack(x, axis=1) for x in ((a, m01, m20), (b, m12, m01), (c, m20, m12), (m01, m12, m20))])
    return np.ascontiguousarray(0.5 * v), np.ascontiguousarray(f, dtype=np.int32)


def _gen(seed):
    g = torch.Generator(device="cpu")
    g.manual_seed(int(seed))
    return g


@torch.no_grad()
def init_weights(model, seed=0, stress=False):
    """Deterministic weights written in place through the module's state_dict (so the same call works on the
    shim modules and on the reference modules, which share key names and shapes).

    stress=False: PyTorch-default-like init (uniform +-1/sqrt(fan_in) conv/linear, identity BatchNorm statistics,
                  constructor neuron constants) -- the "random-init" of the configs.
    stress=True : SURVEY.md section 7 hard-part 5 -- first-layer weights x40, other weights x3, randomised BatchNorm
                  affine/statistics and neuron parameters spread over their clamp ranges, so that neurons cross
                  threshold and outputs depend on the patch.
    """
    sd = model.state_dict()
    g = _gen(seed)
    first_layers = ("encoder.conv1.0.", "fc_delta.0.", "encoder.multi_scale_first_conv.")
    for name in sorted(sd.keys()):
        t = sd[name]
        if not t.dtype.is_floating_point:
            continue
        leaf = name.rsplit(".", 1)[-1]
        new = None
        if leaf in ("weight", "bias") and _is_norm(name, sd):
            if leaf == "weight":
                new = torch.empty(t.shape).uniform_(0.5, 1.5, generator=g) if stress else torch.ones(t.shape)
            else:
                new = torch.empty(t.shape).normal_(0.0, 0.3, generator=g) if stress else torch.zeros(t.shape)
        elif leaf == "running_mean":
            new = torch.empty(t.shape).normal_(0.0, 0.2, generator=g) if stress else torch.zeros(t.shape)
        elif leaf == "running_var":
            new = torch.empty(t.shape).uniform_(0.5, 1.5, generator=g) if stress else torch.ones(t.shape)
        elif leaf == "weight":
            fan_in = int(np.prod(t.shape[1:])) if t.ndim > 1 else t.shape[0]
            bound = 1.0 / math.sqrt(max(fan_in, 1))
            new = torch.empty(t.shape).uniform_(-bound, bound, generator=g)
            if stress:
                new *= 40.0 if any(f in name for f in first_layers) else 3.0
        elif leaf == "bias":
            wkey = name[:-4] + "weight"
            fan_in = int(np.prod(sd[wkey].shape[1:])) if wkey in sd and sd[wkey].ndim > 1 else t.shape[0]
            bound = 1.0 / math.sqrt(max(fan_in, 1))
            new = torch.empty(t.shape).uniform_(-bound, bound, generator=g)
            if stress and name.endswith("fc_distance.bias"):
                new = torch.full(t.shape, 0.5)      # keep stress-init distances out of the Softplus tail
        elif leaf == "membrane_decay":
            new = torch.empty(t.shape).uniform_(0.1, 0.99, generator=g) if stress else torch.full(t.shape, 0.9)
        elif leaf == "threshold_adapt":
            new = torch.empty(t.shape).uniform_(0.001, 0.1, generator=g) if stress else torch.full(t.shape, 0.01)
        elif leaf == "refractory_decay":
            new = torch.empty(t.shape).uniform_(0.1, 0.95, generator=g) if stress else torch.full(t.shape, 0.5)
        elif leaf == "threshold_base":
            new = torch.empty(t.shape).uniform_(0.5, 1.5, generator=g) if stress else torch.ones(t.shape)
        elif leaf == "delta_T":
            new = torch.empty(t.shape).uniform_(0.5, 2.0, generator=g) if stress else torch.full(t.shape, 1.0)
        elif leaf == "theta_rh":
            new = torch.empty(t.shape).uniform_(0.3, 1.5, generator=g) if stress else torch.full(t.shape, 0.8)
        elif leaf == "weights":          # fd temporal integration
            new = torch.empty(t.shape).normal_(0.0, 0.5, generator=g) if stress else torch.ones(t.shape)
        if new is None:
            raise KeyError("init_weights: no rule for state_dict entry %r" % name)
        t.copy_(new.to(t.dtype))
    return model


def _is_norm(name, sd):
    """BatchNorm entries have a sibling running_mean; LayerNorm entries are named norm / norm_out."""
    stem = name.rsplit(".", 1)[0]
    if stem + ".running_mean" in sd:
        return True
    last = stem.rsplit(".", 1)[-1]
    return last in ("norm", "norm_out")
