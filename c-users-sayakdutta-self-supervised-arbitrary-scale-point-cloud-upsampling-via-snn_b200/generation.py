"""Generator3D6 -- B200-native drop-in for the reference upsampling pipeline (reference: generation.py:51-187).

Same constructor and `upsample(data[1,N,3]) -> ndarray[M,3] float64` contract.  The hot loop of the reference
(`generateiopoint`, generation.py:122-172: per-chunk KDTree query, gather/centre, fn forward, normalise,
second KDTree query, per-seed Rodrigues python loop, fd forward, `seed + n*d`) becomes one device pipeline:

    H2D(cloud, seeds) -> sapcu_knn -> sapcu_gather_center_rotate -> sapcu_fn_forward -> sapcu_renormalize
                      -> sapcu_gather_center_rotate(normals) -> sapcu_fd_forward -> sapcu_displace -> D2H

The kNN is computed once (the reference queries the same tree twice with identical results) and nothing
round-trips through the host between stages.  Seeds come from `./dense` exactly as in the reference unless the
caller injects them with `seeds=` (needed for synthetic benchmarks; SURVEY.md section 8b).

`upsample(..., return_normals=True)` also returns the fn normals of the output points, oriented consistently on the device
(`orient_normals`: self-kNN + sapcu_orient_normals); without it every path and result is the reference contract above.

`device` may also be a sequence of devices: the flat seed list is then split with `sharding.shard_bounds` (the split of the
torch.distributed path), every shard runs the same pipeline on its device in a host thread of its own, and the results are
gathered in shard order.  A repeated device is one more worker on that device, with its own stream.
"""
import os
import threading

import numpy as np
import torch

from . import _native as N
from .sharding import shard_batch_offsets, shard_bounds


def rotation_matrix_from_vectors(vec1, vec2):
    """Host utility with the reference's signature (generation.py:30-47).  The pipeline itself builds the
    rotations on the device (csrc/patch_ops.cu); this exists for callers that import the helper."""
    a = (vec1 / np.linalg.norm(vec1)).reshape(3)
    b = (vec2 / np.linalg.norm(vec2)).reshape(3)
    v = np.cross(a, b)
    if not any(v):
        return np.eye(3)
    c, s = np.dot(a, b), np.linalg.norm(v)
    k = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    return np.eye(3) + k + k.dot(k) * ((1 - c) / (s ** 2))


def morton_order(d_pts, bits=10):
    """Permutation that sorts points [S,3] (cuda, f64) along a 3-D Morton curve (`bits` per axis).  Seeds are independent
    units, so the pipeline may visit them in any order; in the thread-per-seed kNN of large clouds (N >= 2^20) the 32 seeds
    of a warp then share their filter survivors (the exact fp64 re-rank runs convergent instead of one lane at a time) and
    the patch gathers hit the same cache lines.  torch is plumbing here: three quantisations, a bit interleave, one argsort."""
    lo = d_pts.min(dim=0).values
    span = (d_pts.max(dim=0).values - lo).clamp_min(1e-300)
    q = ((d_pts - lo) / span * ((1 << bits) - 1)).to(torch.int64)
    key = torch.zeros(d_pts.shape[0], dtype=torch.int64, device=d_pts.device)
    for b in range(bits):
        for a in range(3):
            key |= ((q[:, a] >> b) & 1) << (3 * b + a)
    return torch.argsort(key)


@torch.no_grad()
def orient_normals(d_points, d_normals, k=10):
    """Consistently oriented copy of unit normals [S,3] f32 at points [S,3] f64 (both cuda): the self-kNN (sapcu_knn,
    K = min(k + 1, S), the +1 for the point itself) and the spanning-forest propagation of sapcu_orient_normals.  Every row
    of the result is bitwise its input or its negation; per connected component of the kNN graph the topmost point's normal
    points up (include/sapcu_b200.h gives the exact rule)."""
    S = d_points.shape[0]
    if d_points.shape != (S, 3) or d_normals.shape != (S, 3) or d_points.dtype != torch.float64 or d_normals.dtype != torch.float32:
        raise ValueError("orient_normals: points [S,3] float64 and normals [S,3] float32 expected")
    if d_points.device.type != "cuda" or d_normals.device != d_points.device:
        raise N.SapcuError("orient_normals needs both tensors on one CUDA device (no CPU fallback)")
    if k < 1:
        raise ValueError("orient_normals: k must be at least 1")
    out = d_normals.clone(memory_format=torch.contiguous_format)
    if S == 0:
        return out
    L = N.lib()
    dev = d_points.device
    K = min(k + 1, S)
    with torch.cuda.device(dev):
        st = N.stream_ptr(dev)
        pts = d_points.contiguous()
        idx = torch.empty(S, K, dtype=torch.int32, device=dev)
        kws = torch.empty(L.sapcu_knn_workspace_bytes(S), dtype=torch.uint8, device=dev)
        N.check(L.sapcu_knn(N.ptr(pts), S, N.ptr(pts), S, K, N.ptr(idx), N.ptr(kws), kws.numel(), st), "sapcu_knn(self)")
        ws = torch.empty(L.sapcu_orient_normals_workspace_bytes(S, K), dtype=torch.uint8, device=dev)
        N.check(L.sapcu_orient_normals(N.ptr(pts), S, N.ptr(idx), K, N.ptr(out), None, N.ptr(ws), ws.numel(), st),
                "sapcu_orient_normals")
    return out


def _on_device(fn):
    """Run a Generator3D6 method with the generator's CUDA device current (launches, allocations and the stream the
    C ABI receives all belong to that device, whichever device the calling thread had selected)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **kw):
        if self.device.type != "cuda":
            raise N.SapcuError("Generator3D6 needs a CUDA device (no CPU fallback)")
        with torch.cuda.device(self.device):
            return fn(self, *a, **kw)
    return wrapper


class Generator3D6(object):
    def __init__(self, model1, model2, device, k_neighbors=100, dense_spacing=0.004,
                 outlier_threshold=1.5, batch_size=400, seeds_per_pass=None, remove_outliers=True, seed_source="gpu",
                 normal_neighbors=10):
        self.model1, self.model2 = model1, model2          # fn (normals), fd (distances)
        self.devices = [torch.device(d) for d in ([device] if isinstance(device, (str, int, torch.device)) else device)]
        if not self.devices:
            raise ValueError("Generator3D6: empty device list")
        self.device = self.devices[0]                      # primary device: seeds, outlier filter, gathered results
        self.k_neighbors = k_neighbors
        self.dense_spacing = dense_spacing
        self.outlier_threshold = outlier_threshold
        self.batch_size = batch_size                       # kept for API compatibility; results are per-seed
        self.seeds_per_pass = seeds_per_pass               # device-side pass size (None: everything at once)
        self.remove_outliers = remove_outliers
        self.seed_source = seed_source                     # "gpu": sapcu_seedgen; "dense": the reference's ./dense process
        self.sort_seeds = True                             # Morton-order the seeds of large clouds (N >= 2^20) before the pipeline
        self.normal_neighbors = normal_neighbors           # k of the graph that orients returned normals (return_normals=True)
        self.model1.eval()
        self.model2.eval()
        self._bufs = {}
        self._streams = {}                                 # worker index -> its stream (several devices only)

    # ------------------------------------------------------------------ reference API
    def upsample(self, data, seeds=None, return_normals=False):
        return self.generateiopoint(data, seeds=seeds, return_normals=return_normals)

    def generateiopoint(self, data, seeds=None, return_normals=False):
        """-> points [M,3] f64; with return_normals: (points, normals [M,3] f32), the fn normals of the same rows, oriented
        consistently over the surviving points (orient_normals, k = normal_neighbors)."""
        data = np.asarray(data, dtype=np.float64)
        if data.ndim == 3:
            data = np.squeeze(data, 0)
        if seeds is None:
            seeds = self._dense_seeds(data)
        seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.float64)[:, :3])
        if return_normals:
            return self._points_and_normals(np.ascontiguousarray(data), seeds)[0]
        out = self.displace_host(data, seeds)
        if self.remove_outliers:
            out = self._outlier_filter(out)
        return out

    @_on_device
    def _points_and_normals(self, cloud, seeds, batch=None):
        """The pipeline with its normals kept, per problem of `batch` (one problem without): the outlier mask selects points
        and normals alike, then the normals are oriented on the surviving points, on the primary device.  Returns a list of
        (points [M_b,3] f64, normals [M_b,3] f32) host arrays."""
        d_out, _, d_normals, _ = self.displace_device(torch.from_numpy(cloud).to(self.device),
                                                      torch.from_numpy(seeds).to(self.device), return_parts=True, batch=batch)
        so = (0, seeds.shape[0]) if batch is None else batch[1]
        res = []
        for b in range(len(so) - 1):
            pts, nrm = d_out[so[b]:so[b + 1]], d_normals[so[b]:so[b + 1]]
            if self.remove_outliers:
                keep = self._outlier_keep(pts).bool()
                pts, nrm = pts[keep], nrm[keep]
            nrm = orient_normals(pts, nrm, self.normal_neighbors)
            res.append((pts.cpu().numpy(), nrm.cpu().numpy()))
        N.check_device("upsample(return_normals=True)")
        return res

    # ------------------------------------------------------------------ host <-> device pipeline
    def _pinned(self, key, shape, dtype):
        n = int(np.prod(shape))
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < n or buf.dtype != dtype:
            buf = torch.empty(max(n, 1), dtype=dtype, pin_memory=True)
            self._bufs[key] = buf
        return buf[:n].view(*shape)

    @_on_device
    def displace_host(self, cloud, seeds, batch=None):
        """cloud [N,3] f64, seeds [S,3] f64 (host) -> displaced points [S,3] f64 (host).
        Timed end to end by bench.py: includes the H2D copies of its inputs and the D2H copy of the result."""
        if self.device.type != "cuda":
            raise N.SapcuError("Generator3D6 needs a CUDA device (no CPU fallback)")
        h_cloud = self._pinned("cloud", cloud.shape, torch.float64)
        h_cloud.copy_(torch.from_numpy(np.ascontiguousarray(cloud)))
        h_seeds = self._pinned("seeds", seeds.shape, torch.float64)
        h_seeds.copy_(torch.from_numpy(seeds))
        if len(self.devices) > 1 and seeds.shape[0]:
            return self._displace_host_sharded(h_cloud, h_seeds, batch)
        d_cloud = h_cloud.to(self.device, non_blocking=True)
        d_seeds = h_seeds.to(self.device, non_blocking=True)
        d_out = self.displace_device(d_cloud, d_seeds, batch=batch)
        h_out = self._pinned("out", seeds.shape, torch.float64)
        with torch.cuda.device(self.device):
            h_out.copy_(d_out, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            N.check_device("displace_host")
        return h_out.numpy().copy()

    @torch.no_grad()
    def displace_device(self, d_cloud, d_seeds, return_parts=False, batch=None, sort=True):
        """Device-resident pipeline: cloud [N,3] f64, seeds [S,3] f64 (cuda) -> [S,3] f64 (cuda).
        batch = (cloud_off, seed_off): host prefix tables ([B+1] ints) when d_cloud / d_seeds are the concatenation of
        B independent (cloud, seed set) problems -- one batched kNN launch, then the same per-seed pipeline.
        With several devices the seeds are sharded over them and the results (with return_parts: also idx, normals, dist)
        are gathered on the primary device; with one device everything stays on the inputs' device."""
        if len(self.devices) > 1 and d_seeds.shape[0]:
            return self._displace_device_sharded(d_cloud, d_seeds, return_parts, batch, sort)
        return self._displace_local(d_cloud, d_seeds, return_parts, batch, sort)

    def _displace_local(self, d_cloud, d_seeds, return_parts=False, batch=None, sort=True):
        L = N.lib()
        K = self.k_neighbors
        Ncl, S = d_cloud.shape[0], d_seeds.shape[0]
        dev = d_cloud.device
        if sort and batch is None and self.sort_seeds and Ncl >= (1 << 20) and S > 1 and not return_parts:
            # large clouds: visit the seeds along a Morton curve (results are per-seed, so only the order of the work changes)
            with torch.cuda.device(dev):
                perm = morton_order(d_seeds)
                res = self._displace_local(d_cloud, d_seeds[perm].contiguous(), sort=False)
                out = torch.empty_like(res)
                out[perm] = res
            return out
        with torch.cuda.device(dev):              # every launch below goes to the tensors' device and its current stream
            st = N.stream_ptr(dev)
            out = torch.empty(S, 3, dtype=torch.float64, device=dev)
            normals = torch.empty(S, 3, dtype=torch.float32, device=dev)
            dist = torch.empty(S, dtype=torch.float32, device=dev)
            idx = torch.empty(S, K, dtype=torch.int32, device=dev)
            if batch is None:
                kws = torch.empty(L.sapcu_knn_workspace_bytes(Ncl), dtype=torch.uint8, device=dev)
                N.check(L.sapcu_knn(N.ptr(d_cloud), Ncl, N.ptr(d_seeds), S, K, N.ptr(idx), N.ptr(kws), kws.numel(), st), "sapcu_knn")
            else:
                co = np.ascontiguousarray(batch[0], dtype=np.int64)
                so = np.ascontiguousarray(batch[1], dtype=np.int64)
                B = co.shape[0] - 1
                if so.shape[0] != B + 1 or co[-1] != Ncl or so[-1] != S:
                    raise ValueError("batch offsets do not match the concatenated arrays")
                kws = torch.empty(L.sapcu_knn_batched_workspace_bytes(Ncl, B), dtype=torch.uint8, device=dev)
                N.check(L.sapcu_knn_batched(N.ptr(d_cloud), co.ctypes.data, N.ptr(d_seeds), so.ctypes.data, B, K, N.ptr(idx),
                                            N.ptr(kws), kws.numel(), st), "sapcu_knn_batched")
            step = S if not self.seeds_per_pass else int(self.seeds_per_pass)
            step = max(step, 1)
            patches = torch.empty(min(S, step), K, 3, dtype=torch.float32, device=dev)
            for s0 in range(0, S, step):
                s1 = min(S, s0 + step)
                n = s1 - s0
                p = patches[:n]
                N.check(L.sapcu_gather_center_rotate(N.ptr(d_cloud), Ncl, N.ptr(d_seeds[s0:]), N.ptr(idx[s0:]), n, K, None,
                                                     N.ptr(p), st), "gather_center")
                normals[s0:s1] = self.model1(p)
                N.check(L.sapcu_renormalize(N.ptr(normals[s0:]), n, st), "renormalize")
                N.check(L.sapcu_gather_center_rotate(N.ptr(d_cloud), Ncl, N.ptr(d_seeds[s0:]), N.ptr(idx[s0:]), n, K,
                                                     N.ptr(normals[s0:]), N.ptr(p), st), "gather_center_rotate")
                dist[s0:s1] = self.model2(p)
            N.check(L.sapcu_displace(N.ptr(d_seeds), N.ptr(normals), N.ptr(dist), S, N.ptr(out), st), "displace")
        if return_parts:
            return out, idx, normals, dist
        return out

    # ------------------------------------------------------------------ several devices in one process
    def _run_shards(self, S, work, after=None):
        """work(device, lo, hi) for every entry of self.devices and its seed range shard_bounds(S, n)[i], each in a host thread of
        its own (created here, always joined) with its device current and its own stream as the current stream.  `after`: an
        event every worker stream waits for before its first launch.  Returns (results in shard order, streams); an exception in
        a worker is raised here once every worker has finished."""
        n = len(self.devices)
        for d in self.devices:
            if d.type != "cuda":
                raise N.SapcuError("Generator3D6 needs CUDA devices (no CPU fallback); got %s" % d)
        for i in range(n):
            if i not in self._streams:
                self._streams[i] = torch.cuda.Stream(device=self.devices[i])
        streams = [self._streams[i] for i in range(n)]
        results, errors = [None] * n, [None] * n

        def run(i, lo, hi):
            try:
                with torch.no_grad(), torch.cuda.device(streams[i].device), torch.cuda.stream(streams[i]):
                    if after is not None:
                        streams[i].wait_event(after)
                    results[i] = work(streams[i].device, lo, hi) if hi > lo else None
            except BaseException as e:      # noqa: BLE001 -- re-raised in the caller below
                errors[i] = e

        threads = [threading.Thread(target=run, args=(i, lo, hi), name="Generator3D6-%d" % i)
                   for i, (lo, hi) in enumerate(shard_bounds(S, n))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for e in errors:
            if e is not None:
                raise e
        return results, streams

    def _displace_device_sharded(self, d_cloud, d_seeds, return_parts, batch, sort):
        def work(dev, lo, hi):
            b = None if batch is None else (batch[0], shard_batch_offsets(batch[1], lo, hi))
            c = d_cloud.to(dev, non_blocking=True)                     # the cloud is replicated to every device
            s = d_seeds[lo:hi].to(dev, non_blocking=True).contiguous()
            res = self._displace_local(c, s, return_parts, b, sort)
            return res if return_parts else (res,)

        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(d_seeds.device))            # the inputs are complete on the caller's stream
        parts, streams = self._run_shards(d_seeds.shape[0], work, after=ready)
        parts = [p for p in parts if p is not None]
        home = torch.cuda.current_stream(self.device)
        for st in streams:
            home.wait_stream(st)
        for p in parts:
            for t in p:      # made on a worker stream, read by the gather on the caller's stream of its device
                t.record_stream(torch.cuda.current_stream(t.device))
        with torch.cuda.device(self.device):
            out = tuple(torch.cat([p[j].to(self.device, non_blocking=True) for p in parts]) for j in range(len(parts[0])))
        return out if return_parts else out[0]

    def _displace_host_sharded(self, h_cloud, h_seeds, batch):
        """displace_host over several devices: every worker copies the pinned cloud and its seed rows to its device, runs the
        pipeline, copies its points into its rows of one pinned output and synchronises its stream.  Only this (calling)
        thread allocates and fills the pinned buffers, so the workers never race on them."""
        h_out = self._pinned("out", tuple(h_seeds.shape), torch.float64)

        def work(dev, lo, hi):
            b = None if batch is None else (batch[0], shard_batch_offsets(batch[1], lo, hi))
            c = h_cloud.to(dev, non_blocking=True)
            s = h_seeds[lo:hi].to(dev, non_blocking=True)
            h_out[lo:hi].copy_(self._displace_local(c, s, batch=b), non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()

        _, streams = self._run_shards(h_seeds.shape[0], work)
        for d in dict.fromkeys(st.device for st in streams):
            with torch.cuda.device(d):
                N.check_device("displace_host")
        return h_out.numpy().copy()

    def upsample_batch(self, clouds, seeds, return_normals=False):
        """A batch of independent clouds in one device pipeline (the per-file loop of the reference's generate.py:135-160
        as ONE call): clouds / seeds are lists of [N_b,3] / [S_b,3] arrays; returns the list of displaced [S_b,3] f64
        arrays (outlier-filtered per cloud when remove_outliers is set).  return_normals: a list of (points, normals) pairs,
        each cloud's normals oriented on its own points as in upsample."""
        clouds = [np.ascontiguousarray(np.asarray(c, dtype=np.float64).reshape(-1, 3)) for c in clouds]
        seeds = [np.ascontiguousarray(np.asarray(s, dtype=np.float64)[:, :3]) for s in seeds]
        if len(clouds) != len(seeds):
            raise ValueError("upsample_batch: one seed array per cloud")
        co = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
        so = np.concatenate([[0], np.cumsum([s.shape[0] for s in seeds])]).astype(np.int64)
        if return_normals:
            return self._points_and_normals(np.concatenate(clouds, 0), np.concatenate(seeds, 0), batch=(co, so))
        out = self.displace_host(np.concatenate(clouds, 0), np.concatenate(seeds, 0), batch=(co, so))
        res = [out[so[b]:so[b + 1]] for b in range(len(clouds))]
        if self.remove_outliers:
            res = [self._outlier_filter(r) for r in res]
        return res

    # ------------------------------------------------------------------ host-side steps outside the hot path
    @_on_device
    def gpu_seeds(self, data, cap=None, quirk_origin=True, round6=True):
        """Seeds of dense.cpp computed on the device (csrc/seedgen.cu): same set, same order as `./dense`."""
        import ctypes
        L = N.lib()
        d_cloud = torch.from_numpy(np.ascontiguousarray(data, dtype=np.float64)).to(self.device)
        n = d_cloud.shape[0]
        cap = int(cap or max(400 * n, 1 << 20))
        while True:
            ws = torch.empty(L.sapcu_seedgen_workspace_bytes(n, float(self.dense_spacing), cap), dtype=torch.uint8, device=self.device)
            out = torch.empty(cap, 3, dtype=torch.float64, device=self.device)
            cnt = ctypes.c_int64(0)
            N.check(L.sapcu_seedgen(N.ptr(d_cloud), n, float(self.dense_spacing), int(quirk_origin), int(round6), N.ptr(out), cap,
                                    ctypes.byref(cnt), N.ptr(ws), ws.numel(), N.stream_ptr(self.device)), "sapcu_seedgen")
            if cnt.value <= cap:
                return out[:cnt.value].cpu().numpy()
            cap = int(cnt.value)

    def _dense_seeds(self, data):
        """Seed generation: on the device by default; seed_source="dense" shells out to ./dense exactly as the
        reference does (generation.py:113-118; needs a ./test.xyz that the reference never writes)."""
        if self.seed_source == "gpu":
            return self.gpu_seeds(data)
        cmd = f"./dense {self.dense_spacing} {data.shape[0]}"
        print(cmd)
        os.system(cmd)
        return np.loadtxt("target.xyz")[:, 0:3]

    @_on_device
    def _outlier_filter(self, xyz):
        """generation.py:176-183 on the device: self-kNN (k = 30) with sapcu_knn, mean neighbour distance per point,
        keep the points below outlier_threshold x the global mean."""
        d_pts = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float64)).to(self.device)
        return xyz[self._outlier_keep(d_pts).cpu().numpy().astype(bool), :]

    def _outlier_keep(self, d_pts):
        """uint8 [S] keep mask of the outlier filter for points [S,3] f64 on self.device (which must be current)."""
        L = N.lib()
        S = d_pts.shape[0]
        if S < 30:
            raise ValueError("k must be less than or equal to the number of training points")   # as sklearn does
        st = N.stream_ptr(self.device)
        d_pts = d_pts.contiguous()
        idx = torch.empty(S, 30, dtype=torch.int32, device=self.device)
        kws = torch.empty(L.sapcu_knn_workspace_bytes(S), dtype=torch.uint8, device=self.device)
        N.check(L.sapcu_knn(N.ptr(d_pts), S, N.ptr(d_pts), S, 30, N.ptr(idx), N.ptr(kws), kws.numel(), st), "sapcu_knn(self)")
        keep = torch.empty(S, dtype=torch.uint8, device=self.device)
        ows = torch.empty(L.sapcu_outlier_workspace_bytes(S), dtype=torch.uint8, device=self.device)
        N.check(L.sapcu_outlier_mask(N.ptr(d_pts), S, N.ptr(idx), 30, float(self.outlier_threshold), N.ptr(keep), N.ptr(ows),
                                     ows.numel(), st), "sapcu_outlier_mask")
        return keep


class SNNPointCloudGenerator(Generator3D6):
    """Multi-pass variant (reference generation.py:191-220)."""

    def __init__(self, model1, model2, device, **kwargs):
        self.upsampling_ratio = kwargs.pop("upsampling_ratio", 4)
        super().__init__(model1, model2, device, **kwargs)

    def multi_scale_upsample(self, data, num_passes=1):
        result = data
        for _ in range(num_passes):
            result = self.upsample(np.expand_dims(result, 0) if result.ndim == 2 else result)
        return result
