"""Utilities of the reference's generate.py (the CLI driver around Generator3D6) on the device:

  normalize_pointcloud      generate.py:43-53   bbox centre / max-extent scale (host, trivial)
  farthest_point_sample     generate.py:56-74   one cooperative CUDA kernel (csrc/post_ops.cu) instead of `npoint` torch
                                                 round trips; same fp32 arithmetic, start index N // 2, lowest-index ties
  process_file              generate.py:81-101  load .xyz -> normalise -> upsample -> denormalise -> FPS -> save
                                                 (with_normals=True: six columns, point and oriented normal)
"""
import numpy as np
import torch

from . import _native as N


def normalize_pointcloud(cloud):
    bbox = np.zeros((2, 3))
    bbox[0] = np.min(cloud, axis=0)
    bbox[1] = np.max(cloud, axis=0)
    loc = (bbox[0] + bbox[1]) / 2
    scale = (bbox[1] - bbox[0]).max()
    scale_inv = 1.0 / scale if scale > 0 else 1.0
    return (cloud - loc) * scale_inv, loc, scale


def farthest_point_sample(xyz, npoint, device="cuda"):
    """Return the indices (numpy int64) of `npoint` farthest-point samples of xyz [N,3]."""
    L = N.lib()
    d = torch.from_numpy(np.ascontiguousarray(xyz)).float().to(device).contiguous()
    n = d.shape[0]
    out = torch.empty(int(npoint), dtype=torch.int32, device=d.device)
    ws = torch.zeros(32, dtype=torch.uint8, device=d.device)
    with torch.cuda.device(d.device):
        N.check(L.sapcu_fps(N.ptr(d), n, int(npoint), n // 2, N.ptr(out), N.ptr(ws), ws.numel(), N.stream_ptr(d.device)), "sapcu_fps")
    return out.cpu().numpy().astype(np.int64)


def process_file(input_path, output_path, generator, target_points, with_normals=False):
    """with_normals: six columns per row, the point and its oriented normal (Generator3D6.upsample(return_normals=True));
    the uniform scale and translation of the denormalisation leave normals unchanged."""
    cloud = np.loadtxt(input_path)[:, :3]
    cloud, loc, scale = normalize_pointcloud(cloud)
    if with_normals:
        upsampled, normals = generator.upsample(np.expand_dims(cloud, 0), return_normals=True)
    else:
        upsampled = np.array(generator.upsample(np.expand_dims(cloud, 0)))
    upsampled = upsampled * scale + loc
    assert upsampled.shape[0] >= target_points, f"Generated {upsampled.shape[0]} points, expected >= {target_points}"
    indices = farthest_point_sample(upsampled, target_points, device=generator.device)
    rows = upsampled[indices]
    if with_normals:
        rows = np.concatenate([rows, normals[indices]], axis=1)
    np.savetxt(output_path, rows, fmt="%.6f")
