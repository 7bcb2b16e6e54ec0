"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product package.

CPU restatement (torch CPU tensors used as the fp32 array library, exactly the numerical library the
reference itself runs on) of the reference's inference hot path.  Only tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py may import this file.

Parity status: PINNED.  oracle/make_golden.py imports the real reference from /root/reference, runs it on seeded
inputs and (1) asserts this restatement reproduces it, (2) writes tests/golden/*.npz which
tests/test_oracle_golden.py re-checks without the reference checkout.  The reference itself ships no tests or
golden vectors (SURVEY.md section 4); its third-party arithmetic is torch (unpinned in the reference, README.md:293;
2.11.0 here) and scikit-learn's KDTree (unpinned, README.md:294; 1.9.0 here).

Each function cites the reference lines it restates.  Functions take a plain `sd` dict (state_dict: name -> tensor)
instead of nn.Modules.  The schedule is the reference's FAITHFUL one (every time step recomputes every layer);
`schedule="dce"` skips the work whose result is multiplied by the closed refractory gate (SURVEY.md fact 4) and is
asserted bit-identical to the faithful schedule in tests/test_oracle_golden.py.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

SQRT_2PI = float(np.sqrt(2 * np.pi))


# ----------------------------------------------------------------------------- neurons
def spike_function(x):
    """Eval-mode soft spike (fn/snn_coder.py:135-153, fd/snn_coder.py:143-155, :263-275)."""
    xc = torch.clamp(x, -10.0, 10.0)
    gaussian = torch.exp(-(xc ** 2) / 2) / SQRT_2PI
    sigmoid = torch.sigmoid(10.0 * xc)
    return 0.5 * gaussian + 0.5 * sigmoid


def _expand(p, x):
    """Per-channel parameter broadcast over [B,C], [B,C,M] or [B,C,M,k] (fn/snn_coder.py:99-107)."""
    return p.view(1, -1, *([1] * (x.dim() - 2)))


def lif_step(x, prm, state=None):
    """One LIF step (fn/snn_coder.py:109-133 == fd/snn_coder.py:117-141).  prm: dict of the four raw parameters."""
    d = _expand(torch.clamp(prm["membrane_decay"], 0.1, 0.99), x)
    a = _expand(torch.clamp(prm["threshold_adapt"], 0.001, 0.1), x)
    r = _expand(torch.clamp(prm["refractory_decay"], 0.1, 0.95), x)
    th0 = _expand(prm["threshold_base"], x)
    if state is None:
        m, th, rho = torch.zeros_like(x), th0.expand_as(x), torch.zeros_like(x)
    else:
        m, th, rho = state
    x = x * (rho <= 0).float()
    m = m * d * (1 - rho) + x
    s = spike_function(m - th)
    m = m * (1 - s)
    rho = rho * r + s
    th = th + a * s
    th = th0 + (th - th0) * 0.95
    return s, (m, th, rho)


def eif_step(x, prm, state=None):
    """One EIF step (fd/snn_coder.py:223-261): LIF plus delta_T*exp((m_prev-theta_rh)/(delta_T+1e-6))."""
    d = _expand(torch.clamp(prm["membrane_decay"], 0.1, 0.99), x)
    a = _expand(torch.clamp(prm["threshold_adapt"], 0.001, 0.1), x)
    r = _expand(torch.clamp(prm["refractory_decay"], 0.1, 0.95), x)
    th0 = _expand(prm["threshold_base"], x)
    dT = _expand(torch.clamp(prm["delta_T"], 0.1, 5.0), x)
    thrh = _expand(torch.clamp(prm["theta_rh"], 0.1, 2.0), x)
    if state is None:
        m, th, rho = torch.zeros_like(x), th0.expand_as(x), torch.zeros_like(x)
    else:
        m, th, rho = state
    ex = dT * torch.exp(torch.clamp((m - thrh) / (dT + 1e-6), -5.0, 5.0))
    x = x * (rho <= 0).float()
    m = m * d * (1 - rho) + x + ex
    s = spike_function(m - th)
    m = m * (1 - s)
    rho = rho * r + s
    th = th + a * s
    th = th0 + (th - th0) * 0.95
    return s, (m, th, rho)


def neuron_params(sd, prefix):
    keys = ("membrane_decay", "threshold_adapt", "refractory_decay", "threshold_base", "delta_T", "theta_rh")
    return {k: sd[prefix + "." + k] for k in keys if prefix + "." + k in sd}


def lif_chain(x, prm, T, all_steps=False):
    """`for t in range(T): x, *st = lif(x, *st)` -- the fed-back chain used all over fn (e.g. fn/snn_coder.py:318-320)."""
    st, outs = None, []
    step = eif_step if "delta_T" in prm else lif_step
    for _ in range(T):
        x, st = step(x, prm, st)
        outs.append(x)
    return torch.stack(outs, 0) if all_steps else x


# ----------------------------------------------------------------------------- graph utilities
def intra_knn(x, k):
    """`knn(x, k)` (fn/snn_coder.py:31-39 == fd/snn_coder.py:25-32): x [B,C,N] -> idx [B,N,k]."""
    k = min(k, x.shape[2])
    inner = -2 * torch.matmul(x.transpose(2, 1), x)
    xx = torch.sum(x ** 2, dim=1, keepdim=True)
    pd = -xx - inner - xx.transpose(2, 1)
    return pd.topk(k=k, dim=-1)[1]


def gather_points(points, idx):
    """`index_points` (fn/snn_coder.py:19-29): points [B,N,C], idx [B,N,k] -> [B,N,k,C]."""
    B = points.shape[0]
    bidx = torch.arange(B, device=idx.device).view(B, *([1] * (idx.dim() - 1))).expand_as(idx)
    return points[bidx, idx, :]


def graph_feature(x, k, idx=None):
    """`get_graph_feature` (fd/snn_coder.py:52-68): x [B,C,N] -> cat(x_j - x_i, x_j) as [B,2C,N,k]."""
    B, C, Np = x.shape
    k = min(k, Np)
    if idx is None:
        idx = intra_knn(x, k)
    xt = x.transpose(2, 1).contiguous()
    nb = gather_points(xt, idx)                                   # [B,N,k,C]
    ctr = xt.unsqueeze(2).expand(-1, -1, k, -1)
    return torch.cat((nb - ctr, nb), dim=-1).permute(0, 3, 1, 2).contiguous(), idx


def _bn(sd, p, x):
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"],
                        False, 0.0, 1e-5)


def _conv_bn(sd, p, x):
    """nn.Sequential(ConvNd(k=1), BatchNormNd) in eval mode; conv bias is optional."""
    w, b = sd[p + ".0.weight"], sd.get(p + ".0.bias")
    y = F.conv2d(x, w, b) if w.dim() == 4 else F.conv1d(x, w, b)
    return _bn(sd, p + ".1", y)


# ----------------------------------------------------------------------------- fn
def fn_block(sd, p, xyz, feats, k, heads, T=4, taps=None):
    """MultiHeadSNNTransformerBlock.forward (fn/snn_coder.py:294-396).  xyz [B,N,3], feats [B,N,64]."""
    B, Np, _ = xyz.shape
    k = min(k, Np)
    idx = intra_knn(xyz.permute(0, 2, 1).contiguous(), k)                   # :307 (cache neutralised: always fresh)
    pos_diff = xyz[:, :, None, :] - gather_points(xyz, idx)                 # :308-310
    f = feats.permute(0, 2, 1).contiguous()
    pre = f
    x = lif_chain(_conv_bn(sd, p + ".fc1", f), neuron_params(sd, p + ".snn1"), T)          # :317-320
    q = lif_chain(_conv_bn(sd, p + ".w_qs", x), neuron_params(sd, p + ".snn_q"), T)        # :322-325
    kf = lif_chain(_conv_bn(sd, p + ".w_ks", x), neuron_params(sd, p + ".snn_k"), T)       # :327-330
    v = lif_chain(_conv_bn(sd, p + ".w_vs", x), neuron_params(sd, p + ".snn_v"), T)        # :332-335
    D = q.shape[1]
    hd = D // heads
    # :337-353 -- gather k and v at the neighbour lists, channel-first [B,D,N,k]
    kg = gather_points(kf.permute(0, 2, 1).contiguous(), idx).permute(0, 3, 1, 2)
    vg = gather_points(v.permute(0, 2, 1).contiguous(), idx).permute(0, 3, 1, 2)
    pos = lif_chain(_conv_bn(sd, p + ".fc_delta", pos_diff.permute(0, 3, 1, 2).contiguous()),
                    neuron_params(sd, p + ".snn_delta"), T)                                 # :355-358
    pos = lif_chain(_conv_bn(sd, p + ".fc_delta2", pos), neuron_params(sd, p + ".snn_delta2"), T)   # :360-363
    attn_in = q.unsqueeze(-1) - kg + pos                                                    # :367-371
    a1 = lif_chain(_conv_bn(sd, p + ".fc_gamma", attn_in), neuron_params(sd, p + ".snn_gamma"), T)  # :373-376
    logits = _conv_bn(sd, p + ".fc_gamma2", a1)                                             # :378
    H = heads
    attn = F.softmax(logits.view(B, H, hd, Np, k) / np.sqrt(hd), dim=-1)                    # :379-380
    vp = vg.reshape(B, H, hd, Np, k) + pos.view(B, H, hd, Np, k)                            # :386-387
    res = torch.einsum("bhcnk,bhcnk->bhcn", attn, vp).reshape(B, D, Np)                     # :389-391
    res = _conv_bn(sd, p + ".out_proj", res)                                                # :393
    out = _conv_bn(sd, p + ".fc2", res) + pre                                               # :394
    if taps is not None:
        taps[p] = dict(idx=idx, snn1=x, q=q, k=kf, v=v, pos=pos, a1=a1, logits=logits, res_attn=res)
    return out.permute(0, 2, 1).contiguous()


def fn_forward(sd, patches, cfg=None, taps=None):
    """ImprovedSNNNormalEstimation.forward on [B,M,3] (fn/snn_coder.py:670-699 -> :430-476 -> :542-549)."""
    cfg = cfg or dict(k_values=[24, 18, 12], time_steps_enc=6, num_heads=8)
    x = patches.permute(0, 2, 1).contiguous()                                               # :444
    xyz = x.permute(0, 2, 1).contiguous()
    f = lif_chain(_conv_bn(sd, "encoder.conv1", x), neuron_params(sd, "encoder.snn_init"), cfg["time_steps_enc"])
    if taps is not None:
        taps["snn_init"] = f
    f = f.permute(0, 2, 1).contiguous()
    feats = []
    for b in range(3):
        f = fn_block(sd, "encoder.trans%d" % (b + 1), xyz, f, cfg["k_values"][b], cfg["num_heads"], 4, taps)
        feats.append(f)
    ms = torch.cat(feats, dim=2)                                                            # :465
    g = lif_chain(_conv_bn(sd, "encoder.conv_final", ms.permute(0, 2, 1)), neuron_params(sd, "encoder.snn_final"),
                  cfg["time_steps_enc"])                                                    # :467-470
    gmax = F.adaptive_max_pool1d(g, 1).squeeze(-1)                                          # :472
    h = F.linear(gmax, sd["encoder.fc_out.weight"], sd["encoder.fc_out.bias"])              # :475
    if taps is not None:
        taps.update(fcat=ms, snn_final=g, gmax=gmax, enc_out=h)
    for i in (0, 4, 8):                                                                     # decoder.mlp (:523-536)
        h = F.linear(h, sd["decoder.mlp.%d.weight" % i], sd["decoder.mlp.%d.bias" % i])
        h = F.gelu(_bn(sd, "decoder.mlp.%d" % (i + 1), h))
    if taps is not None:
        taps["dec_h3"] = h
    h = F.linear(h, sd["decoder.fc_out.weight"], sd["decoder.fc_out.bias"])
    h = F.layer_norm(h, (3,), sd["decoder.norm_out.weight"], sd["decoder.norm_out.bias"], 1e-5)
    return F.normalize(h, dim=1)                                                            # :545-548


# ----------------------------------------------------------------------------- fd
def fd_encoder(sd, patches, cfg=None, schedule="faithful", taps=None, forced_idx=None):
    """EnhancedTemporalSNN_DGCNN_fd.forward (fd/snn_coder.py:392-492)."""
    cfg = cfg or dict(k=32, time_steps_enc=7, k_scales=[8, 16, 32, 48])
    x = patches.transpose(1, 2).contiguous()                                                # :393-394
    B, _, M = x.shape
    T = cfg["time_steps_enc"]
    step_fns = [eif_step, eif_step, lif_step, lif_step]
    prms = [neuron_params(sd, "encoder.snn_blocks.%d" % i) for i in range(4)]
    states = [None] * 4
    pooled, spikes_t, graph_idx, pre_act = [], [], [None] * 3, [None] * 4
    for t in range(T):                                                                      # :408
        live = (t == 0) or schedule == "faithful"
        feats = []
        if live:
            sf = []
            for ks, i in zip(cfg["k_scales"], range(len(cfg["k_scales"]))):                 # :413-417
                g, _ = graph_feature(x, min(ks, M))
                p = "encoder.multi_scale_first_conv.%d" % i
                sf.append(F.leaky_relu(_conv_bn(sd, p, g), 0.2).max(dim=-1)[0])
            u = F.leaky_relu(_conv_bn(sd, "encoder.scale_fusion", torch.cat(sf, dim=1)), 0.2)   # :420-421
            if t == 0:
                pre_act[0] = u
        else:
            u = torch.zeros(B, 64, M, device=x.device)          # multiplied by the closed gate: value is irrelevant
        s, states[0] = step_fns[0](u, prms[0], states[0])                                   # :432-443
        feats.append(s)
        cur = s
        for b in range(1, 4):                                                               # :447-474
            if live:
                fi = None
                if forced_idx is not None and t == 0:
                    fi = forced_idx[b - 1]
                g, gi = graph_feature(cur, min(cfg["k"], M), fi)
                if t == 0:
                    graph_idx[b - 1] = gi
                u = F.leaky_relu(_conv_bn(sd, "encoder.conv_blocks.%d" % (b - 1), g), 0.2).max(dim=-1)[0]
                if t == 0:
                    pre_act[b] = u
            else:
                u = torch.zeros(B, prms[b]["threshold_base"].numel(), M, device=x.device)
            s, states[b] = step_fns[b](u, prms[b], states[b])
            feats.append(s)
            cur = s
        cat = torch.cat(feats, dim=1)                                                       # :476
        agg = F.leaky_relu(_conv_bn(sd, "encoder.multi_scale_conv", cat), 0.2)              # :477
        pooled.append(F.adaptive_max_pool1d(agg, 1).squeeze(-1))                            # :479-480
        spikes_t.append(cat)
    tf = torch.stack(pooled, dim=0)
    w = F.softmax(sd["encoder.temporal_integration.weights"], dim=0)                        # :326-328
    z = torch.einsum("t,tbf->bf", w, tf)
    s, _ = lif_step(z, neuron_params(sd, "encoder.snn_fc"), None)                           # :485-490 (state is always zero)
    if taps is not None:
        taps.update(spikes=torch.stack(spikes_t, 0), pool=tf, z=s, graph_idx=graph_idx, pre_act=pre_act)
    return s


def fd_decoder(sd, z, heads=8, taps=None):
    """StandardDistanceDecoder.forward (fd/snn_coder.py:711-725, :751-758, :777-798)."""
    d = "distance_decoder."
    lin = lambda p, x: F.linear(x, sd[d + p + ".weight"], sd[d + p + ".bias"])
    x = F.gelu(_bn(sd, d + "fc_in.1", lin("fc_in.0", z)))
    for r in range(2):
        p = "residual_blocks.%d." % r
        out = F.gelu(_bn(sd, d + p + "fc.1", lin(p + "fc.0", x)))
        out = _bn(sd, d + p + "fc.5", lin(p + "fc.4", out))
        res = lin(p + "res_proj", x) if (d + p + "res_proj.weight") in sd else x
        x = F.gelu(out + res)
    if taps is not None:
        taps["dec_d2"] = x
    B, dim = x.shape
    hd = dim // heads
    q, k, v = lin("attention.to_qkv", x).chunk(3, dim=-1)
    q, k, v = q.view(B, heads, hd), k.view(B, heads, hd), v.view(B, heads, hd)
    attn = F.softmax(torch.einsum("bhd,bhd->bh", q, k) * (hd ** -0.5), dim=-1)
    o = torch.einsum("bh,bhd->bhd", attn, v).reshape(B, -1)
    x = F.layer_norm(lin("attention.to_out.0", o) + x, (dim,), sd[d + "attention.norm.weight"],
                     sd[d + "attention.norm.bias"], 1e-5)
    x = F.gelu(_bn(sd, d + "fc_hidden.1", lin("fc_hidden.0", x)))
    if taps is not None:
        taps["dec_hidden"] = x
    return F.softplus(lin("fc_distance", x), beta=5.0).squeeze(-1)


def fd_forward(sd, patches, cfg=None, schedule="faithful", taps=None, forced_idx=None):
    """EnhancedSNNDistanceEstimation.forward on [B,M,3] (fd/snn_coder.py:853-871)."""
    cfg = cfg or dict(k=32, time_steps_enc=7, k_scales=[8, 16, 32, 48], num_heads=8)
    z = fd_encoder(sd, patches, cfg, schedule, taps, forced_idx)
    return fd_decoder(sd, z, cfg.get("num_heads", 8), taps)


# ----------------------------------------------------------------------------- generation.py pipeline
def knn_seed(cloud, seeds, K):
    """KDTree(data).query(chunk, K)[1] (generation.py:110,127,153) restated as an exact fp64 brute force:
    squared distance ((dx*dx)+(dy*dy))+(dz*dz), stable ascending sort (ties -> lowest index)."""
    d = seeds[:, None, :] - cloud[None, :, :]
    d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2]
    return np.argsort(d2, axis=1, kind="stable")[:, :K].astype(np.int32)


def rotation_to_x(n):
    """rotation_matrix_from_vectors(n, [1,0,0]) (generation.py:30-47) with the reference's dtypes: n is float32."""
    a = (n / np.linalg.norm(n)).reshape(3)
    b = (np.array([1, 0, 0]) / np.linalg.norm([1, 0, 0])).reshape(3)
    v = np.cross(a, b)
    if not any(v):
        return np.eye(3)
    c = np.dot(a, b)
    s = np.linalg.norm(v)
    k = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    return np.eye(3) + k + k.dot(k) * ((1 - c) / (s ** 2))


def gather_center(cloud, seeds, idx, normals=None):
    """generation.py:128-129 (fn pass) / :154-160 (fd pass: + per-seed rotation); returns float32 [S,K,3]."""
    patch = cloud[idx] - seeds[:, None, :]
    if normals is not None:
        for j in range(patch.shape[0]):
            patch[j] = np.matmul(rotation_to_x(normals[j]), patch[j].T).T
    return patch.astype(np.float32)


def displace(seeds, normals, dist):
    """generation.py:171-172: seed + n * tile(d)  (fp32 product, fp64 sum)."""
    return seeds + normals * np.tile(np.expand_dims(dist, 1), (1, 3))


def pipeline(sd_fn, sd_fd, cloud, seeds, K=100, batch=256, cfg_fn=None, cfg_fd=None, schedule="faithful", device=None):
    """generation.py:122-172 with injected seeds: returns (points [S,3] f64, idx, normals f32, dist f32).
    device: where the two model forwards run, exactly as in the reference (`.to(device)` per batch, generation.py:137,168;
    kNN, gather and the rotations stay on the host); None = CPU.  On CUDA the caller disables TF32 (SURVEY.md 7-6)."""
    cfg_fd = cfg_fd or dict(k=32, time_steps_enc=7, k_scales=[8, 16, 32, 48], num_heads=8)
    if device is not None:
        sd_fn = {k: v.to(device) for k, v in sd_fn.items()}
        sd_fd = {k: v.to(device) for k, v in sd_fd.items()}
    idx = knn_seed(cloud, seeds, K)
    normals, dists = [], []
    with torch.no_grad():
        for s0 in range(0, seeds.shape[0], batch):
            sl = slice(s0, min(seeds.shape[0], s0 + batch))
            p = torch.from_numpy(gather_center(cloud, seeds[sl], idx[sl])).to(device)
            n = F.normalize(fn_forward(sd_fn, p, cfg_fn), dim=-1).cpu().numpy()             # :138-139
            normals.append(n)
            pr = torch.from_numpy(gather_center(cloud, seeds[sl], idx[sl], n)).to(device)
            dists.append(fd_forward(sd_fd, pr, cfg_fd, schedule).cpu().numpy())
    normals, dists = np.concatenate(normals, 0), np.concatenate(dists, 0)
    return displace(seeds, normals, dists), idx, normals, dists


# ----------------------------------------------------------------------------- "next" rows: outlier filter, FPS
def outlier_filter(xyz, threshold=1.5, k=30):
    """generation.py:176-183: KDTree self-query (k = 30, true distances), keep avg < threshold * global mean."""
    from sklearn.neighbors import KDTree
    dist, _ = KDTree(xyz).query(xyz, k)
    avg = np.mean(dist, axis=1)
    avgtotal = np.mean(dist)
    return np.where(avg < avgtotal * threshold)[0]


def fps(xyz, npoint, start=None):
    """farthest_point_sample (generate.py:56-74) restated in numpy float32: start at N // 2 (or `start`), distances 1e32,
    `dist < distance` update, arg-max (first maximum)."""
    xyz = np.asarray(xyz, dtype=np.float32)
    n = xyz.shape[0]
    out = np.zeros(npoint, dtype=np.int64)
    distance = np.full(n, 1e32, dtype=np.float32)
    far = n // 2 if start is None else int(start)
    for i in range(npoint):
        out[i] = far
        d = xyz - xyz[far]
        dist = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        m = dist < distance
        distance[m] = dist[m]
        far = int(np.argmax(distance))
    return out
