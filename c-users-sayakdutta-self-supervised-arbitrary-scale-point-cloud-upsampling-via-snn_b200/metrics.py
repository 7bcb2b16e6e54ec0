"""Quality metrics of upsampled clouds on the GPU: Chamfer (CD), Hausdorff (HD), point-to-mesh (P2F) distances and the
normal error against the closest mesh face.

    read_off(path)                              -> vertices [V,3] f64, faces [F,3] int32 (plain-text OFF, triangles only)
    nn_distances(a, b)                          -> [len(a)] f64, distance from each row of a to its nearest row of b
    chamfer_hausdorff(pred, gt)                 -> {"cd", "cd_sq", "hd"}
    point_to_mesh(points, vertices, faces)      -> [S] f64 exact distance to the mesh (and the closest face)
    normal_errors(points, normals, vertices, faces)
    evaluate(pred, gt, vertices, faces, normals, normalize)

The nearest neighbours come from sapcu_knn with K = 1 (exact fp64), the point-to-mesh distances from sapcu_mesh_distance (an
LBVH built and queried on the device, bitwise the brute-force minimum; include/sapcu_b200.h).  Point arrays may be numpy
arrays or CUDA tensors; numpy inputs go to the current CUDA device.  Results are host (numpy / float) values.

    python -m sapcu_b200.metrics PRED_DIR GT_DIR [--mesh-dir DIR] [--json OUT]

pairs PRED_DIR/<stem>.xyz with GT_DIR/<stem>.xyz (and MESH_DIR/<stem>.off), prints one line per file and the means.  A
prediction with six columns (generate.process_file(..., with_normals=True)) is graded on its normals too.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

from . import _native as N


# ----------------------------------------------------------------------------------------------------------------- inputs
def read_off(path):
    """Plain-text OFF -> (vertices [V,3] float64, faces [F,3] int32).  '#' starts a comment; extra per-vertex or per-face
    values (colours) after the coordinates / indices are ignored.  A missing 'OFF' header, wrong counts, a face that is not a
    triangle or an index outside [0, V) raise ValueError: nothing is triangulated or repaired silently."""
    with open(path) as fh:
        rows = [ln.split("#", 1)[0].split() for ln in fh]
    rows = [r for r in rows if r]
    if not rows or rows[0][0] != "OFF":
        raise ValueError("%s: not an OFF file (first token %r)" % (path, rows[0][0] if rows else None))
    head = rows[0][1:] if len(rows[0]) > 1 else (rows[1] if len(rows) > 1 else [])
    body = rows[1:] if len(rows[0]) > 1 else rows[2:]
    try:
        nv, nf = int(head[0]), int(head[1])
    except (IndexError, ValueError):
        raise ValueError("%s: bad OFF counts line %r" % (path, head)) from None
    if nv < 0 or nf < 0 or len(body) != nv + nf:
        raise ValueError("%s: header announces %d vertices and %d faces, the file has %d data rows" % (path, nv, nf, len(body)))
    try:
        vertices = np.array([[float(x) for x in r[:3]] for r in body[:nv]], dtype=np.float64).reshape(nv, 3)
        face_rows = [[int(x) for x in r[:4]] for r in body[nv:]]
    except ValueError as e:
        raise ValueError("%s: %s" % (path, e)) from None
    if any(len(r) < 4 or r[0] != 3 for r in face_rows) or any(len(r) < 3 for r in body[:nv]):
        raise ValueError("%s: only triangle faces ('3 i j k') and 3-coordinate vertices are accepted" % path)
    faces = np.array([r[1:] for r in face_rows], dtype=np.int64).reshape(nf, 3)
    if faces.size and (faces.min() < 0 or faces.max() >= nv):
        raise ValueError("%s: face index outside [0, %d)" % (path, nv))
    return vertices, faces.astype(np.int32)


def _device_f64(x, name, device=None):
    """[n,3] float64 contiguous CUDA tensor of a numpy array or tensor; non-finite values raise."""
    if isinstance(x, torch.Tensor):
        if x.device.type != "cuda":
            raise N.SapcuError("%s: CPU tensors are not accepted (no CPU fallback); pass numpy or a CUDA tensor" % name)
        t = x.detach().to(device or x.device, torch.float64)
    else:
        t = torch.from_numpy(np.asarray(x, dtype=np.float64)).to(device or torch.device("cuda", torch.cuda.current_device()))
    if t.ndim != 2 or t.shape[1] != 3:
        raise ValueError("%s: [n,3] coordinates expected, got shape %s" % (name, tuple(t.shape)))
    if not bool(torch.isfinite(t).all()):
        raise ValueError("%s: non-finite coordinates" % name)
    return t.contiguous()


# ----------------------------------------------------------------------------------------------------------------- CD / HD
def _nn_dist2(d_a, d_b):
    """((dx*dx)+(dy*dy))+(dz*dz) from each row of d_a to its nearest row of d_b (both [n,3] f64 on one CUDA device)."""
    S, M = d_a.shape[0], d_b.shape[0]
    if S == 0:
        return torch.empty(0, dtype=torch.float64, device=d_a.device)
    if M == 0:
        raise ValueError("nn_distances: the second cloud is empty")
    L = N.lib()
    dev = d_a.device
    with torch.cuda.device(dev):
        idx = torch.empty(S, 1, dtype=torch.int32, device=dev)
        ws = torch.empty(L.sapcu_knn_workspace_bytes(M), dtype=torch.uint8, device=dev)
        N.check(L.sapcu_knn(N.ptr(d_b), M, N.ptr(d_a), S, 1, N.ptr(idx), N.ptr(ws), ws.numel(), N.stream_ptr(dev)), "sapcu_knn(K=1)")
        d = d_a - d_b[idx[:, 0].long()]
        return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]      # separate rounded ops, no contraction


def nn_distances(a, b):
    """Euclidean distance from each row of `a` to its nearest row of `b` ([len(a)] float64, numpy): sapcu_knn(cloud=b,
    seeds=a, K=1), then sqrt(((dx*dx)+(dy*dy))+(dz*dz)) of the returned neighbour."""
    d_a = _device_f64(a, "a")
    return torch.sqrt(_nn_dist2(d_a, _device_f64(b, "b", d_a.device))).cpu().numpy()


def chamfer_hausdorff(pred, gt):
    """With d_pg(p) = min_g |p - g| over gt for every p in pred, and d_gp the same from gt to pred:

        cd    = mean(d_pg) + mean(d_gp)
        cd_sq = mean(d_pg^2) + mean(d_gp^2)       (squared distances as computed, not squares of the roots)
        hd    = max(max(d_pg), max(d_gp))

    Means are fp64 sums over the whole cloud.  Evaluation scripts of the upsampling literature differ in whether CD is
    summed or averaged over the two directions and whether it uses squared distances; cd and cd_sq above are both sums of the
    two directions' means.  Which convention external/Meta-PU_evaluation uses has not been checked against it here: that needs
    a SAPCU_REFERENCE checkout."""
    d_p = _device_f64(pred, "pred")
    d_g = _device_f64(gt, "gt", d_p.device)
    return cd_hd_from_dist2(_nn_dist2(d_p, d_g), _nn_dist2(d_g, d_p))


def cd_hd_from_dist2(pg2, gp2):
    """chamfer_hausdorff's formulas from the squared nearest-neighbour distances of both directions (tensors)."""
    pg, gp = torch.sqrt(pg2), torch.sqrt(gp2)
    return {"cd": float(pg.mean() + gp.mean()), "cd_sq": float(pg2.mean() + gp2.mean()),
            "hd": float(torch.maximum(pg.max(), gp.max()))}


# ----------------------------------------------------------------------------------------------------------------- P2F
def _mesh_arrays(vertices, faces, device):
    d_v = _device_f64(vertices, "vertices", device)
    f = faces.detach().cpu().numpy() if isinstance(faces, torch.Tensor) else np.asarray(faces)
    if f.ndim != 2 or f.shape[1] != 3 or f.shape[0] < 1:
        raise ValueError("faces: [F,3] indices expected (F >= 1), got shape %s" % (f.shape,))
    if f.min() < 0 or f.max() >= d_v.shape[0]:
        raise ValueError("faces: index outside [0, %d)" % d_v.shape[0])
    return d_v, torch.from_numpy(np.ascontiguousarray(f, dtype=np.int32)).to(device)


def _point_to_mesh(d_p, d_v, d_f):
    """(dist2 [S] f64, face [S] int32) on the device of d_p."""
    L = N.lib()
    S, V, F = d_p.shape[0], d_v.shape[0], d_f.shape[0]
    dev = d_p.device
    with torch.cuda.device(dev):
        d2 = torch.empty(S, dtype=torch.float64, device=dev)
        face = torch.empty(S, dtype=torch.int32, device=dev)
        ws = torch.empty(max(L.sapcu_mesh_distance_workspace_bytes(V, F), 1), dtype=torch.uint8, device=dev)
        N.check(L.sapcu_mesh_distance(N.ptr(d_v), V, N.ptr(d_f), F, N.ptr(d_p), S, N.ptr(d2), N.ptr(face), N.ptr(ws), ws.numel(),
                                      N.stream_ptr(dev)), "sapcu_mesh_distance")
    return d2, face


def point_to_mesh(points, vertices, faces, return_face=False):
    """Exact distance ([S] float64, numpy) from every point to the triangle mesh (vertices [V,3], faces [F,3]):
    sqrt of sapcu_mesh_distance's D (include/sapcu_b200.h).  return_face: also the index of the closest face ([S] int32;
    ties go to the lowest index).  Faces must index [0, V); non-finite coordinates raise."""
    d_p = _device_f64(points, "points")
    d2, face = _point_to_mesh(d_p, *_mesh_arrays(vertices, faces, d_p.device))
    dist = torch.sqrt(d2).cpu().numpy()
    return (dist, face.cpu().numpy()) if return_face else dist


def _face_normals(vertices, faces):
    v = np.asarray(vertices, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    return np.cross(b - a, c - a)


def normal_errors(points, normals, vertices, faces):
    """Normals graded against the geometric normal (b-a)x(c-a) of each point's closest face:

        angle_*      unoriented angle in degrees, acos(|cos|) -- mean, median, max
        flipped      share of normals with cos < 0: the orientation error, meaningful on a closed, consistently wound mesh
                     (outward normals of an outward-wound mesh give 0)

    A zero-area closest face or a zero normal counts as 90 degrees and not flipped."""
    d_p = _device_f64(points, "points")
    _, face = _point_to_mesh(d_p, *_mesh_arrays(vertices, faces, d_p.device))
    fn = _face_normals(vertices.detach().cpu().numpy() if isinstance(vertices, torch.Tensor) else vertices,
                       faces.detach().cpu().numpy() if isinstance(faces, torch.Tensor) else faces)[face.cpu().numpy()]
    n = normals.detach().cpu().numpy() if isinstance(normals, torch.Tensor) else np.asarray(normals)
    n = n.astype(np.float64).reshape(-1, 3)
    if n.shape[0] != d_p.shape[0]:
        raise ValueError("normal_errors: one normal per point expected")
    return normal_stats(n, fn)


def normal_stats(normals, face_normals):
    """normal_errors' numbers from per-point normals and the (unnormalised) normals of their closest faces ([n,3] each)."""
    n, fn = np.asarray(normals, dtype=np.float64), np.asarray(face_normals, dtype=np.float64)
    if len(n) == 0:
        return {"angle_mean": float("nan"), "angle_median": float("nan"), "angle_max": float("nan"), "flipped": float("nan")}
    den = np.linalg.norm(n, axis=1) * np.linalg.norm(fn, axis=1)
    cos = np.divide((n * fn).sum(1), den, out=np.zeros(len(n)), where=den > 0)
    ang = np.degrees(np.arccos(np.clip(np.abs(cos), 0.0, 1.0)))
    return {"angle_mean": float(ang.mean()), "angle_median": float(np.median(ang)), "angle_max": float(ang.max()),
            "flipped": float((cos < 0).mean())}


# ----------------------------------------------------------------------------------------------------------------- one shape
def _host(x):
    return x.detach().cpu().numpy().astype(np.float64) if isinstance(x, torch.Tensor) else np.asarray(x, dtype=np.float64)


def unit_ball(gt):
    """(centroid, furthest-point distance from it) of a cloud: evaluate's normalisation x -> (x - c) / r (r = 1 when 0)."""
    gt = np.asarray(gt, dtype=np.float64)
    c = gt.mean(axis=0)
    r = float(np.sqrt(((gt - c) ** 2).sum(1)).max()) if len(gt) else 0.0
    return c, (r if r > 0 else 1.0)


def evaluate(pred, gt, vertices=None, faces=None, normals=None, normalize=True):
    """CD / HD between pred and gt and, given a mesh, P2F (mean and std of the point-to-mesh distances of pred) and, given
    normals of pred, normal_errors.  normalize: pred, gt and the mesh are first mapped by x -> (x - c) / r with c the gt
    cloud's centroid and r its largest distance from c (the gt then lies in the unit ball), so numbers of differently
    scaled shapes are comparable; normals are unchanged by that map."""
    pred, gt = _host(pred)[:, :3], _host(gt)[:, :3]
    if vertices is not None:
        vertices = _host(vertices)
    if normalize:
        c, r = unit_ball(gt)
        pred, gt = (pred - c) / r, (gt - c) / r
        if vertices is not None:
            vertices = (vertices - c) / r
    out = chamfer_hausdorff(pred, gt)
    if vertices is not None and faces is not None:
        p2f = point_to_mesh(pred, vertices, faces)
        out["p2f_mean"], out["p2f_std"] = float(p2f.mean()), float(p2f.std())
        if normals is not None:
            out.update(normal_errors(pred, normals, vertices, faces))
    return out


# ----------------------------------------------------------------------------------------------------------------- CLI
def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m sapcu_b200.metrics", description=__doc__.split("\n\n")[0])
    ap.add_argument("pred_dir")
    ap.add_argument("gt_dir")
    ap.add_argument("--mesh-dir", default=None, help="<stem>.off meshes for P2F (and normals, when pred has six columns)")
    ap.add_argument("--json", default=None, help="write the per-file results and the means here")
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        sys.exit("sapcu_b200.metrics needs a CUDA device (no CPU fallback)")
    stems = sorted(os.path.splitext(f)[0] for f in os.listdir(a.pred_dir) if f.endswith(".xyz"))
    rows = {}
    for stem in stems:
        gt_path = os.path.join(a.gt_dir, stem + ".xyz")
        if not os.path.exists(gt_path):
            print("%s: no ground truth %s, skipped" % (stem, gt_path))
            continue
        pred = np.loadtxt(os.path.join(a.pred_dir, stem + ".xyz"), ndmin=2)
        gt = np.loadtxt(gt_path, ndmin=2)
        mesh = None
        if a.mesh_dir:
            off = os.path.join(a.mesh_dir, stem + ".off")
            if os.path.exists(off):
                mesh = read_off(off)
        r = evaluate(pred[:, :3], gt, *(mesh or (None, None)), normals=pred[:, 3:6] if pred.shape[1] >= 6 else None)
        rows[stem] = r
        print(stem + "  " + "  ".join("%s %.6g" % kv for kv in r.items()))
    keys = sorted({k for r in rows.values() for k in r})
    mean = {k: float(np.mean([r[k] for r in rows.values() if k in r])) for k in keys}
    print("mean (%d files)  " % len(rows) + "  ".join("%s %.6g" % (k, mean[k]) for k in keys))
    if a.json:
        with open(a.json, "w") as fh:
            json.dump({"files": rows, "mean": mean}, fh, indent=1, sort_keys=True)
    return 0 if rows else 1


if __name__ == "__main__":
    sys.exit(main())
