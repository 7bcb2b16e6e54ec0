"""EnhancedSNNDistanceEstimation -- B200-native drop-in for the reference class of the same name
(reference: fd/snn_coder.py:805-892).

As in fn/snn_coder.py the module tree only reproduces the reference's state_dict names
(`encoder.multi_scale_first_conv.2.0.weight`, `encoder.snn_blocks.1.delta_T`,
`distance_decoder.residual_blocks.0.res_proj.weight`, ...); `forward` calls `sapcu_fd_forward`.
"""
import torch
import torch.nn as nn

from .. import _native as N
from .._model_base import NativeModel
from ..neurons import MultiTimeConstantEIFNeuron, MultiTimeConstantLIFNeuron


class TemporalIntegration(nn.Module):
    def __init__(self, time_steps, feature_dim):
        super().__init__()
        self.weights = nn.Parameter(torch.ones(time_steps))


def _edge_conv(cin, cout):
    return nn.Sequential(nn.Conv2d(cin, cout, 1, bias=False), nn.BatchNorm2d(cout), nn.LeakyReLU(0.2))


class EnhancedTemporalSNN_DGCNN_fd(nn.Module):
    """Parameter container of the SNN-DGCNN encoder (reference fd/snn_coder.py:330-390)."""

    def __init__(self, k=20, emb_dims=512, time_steps=5, k_scales=(10, 20, 40)):
        super().__init__()
        self.k, self.emb_dims, self.time_steps, self.k_scales = k, emb_dims, time_steps, list(k_scales)
        self.conv_blocks = nn.ModuleList([_edge_conv(128, 128), _edge_conv(256, 256), _edge_conv(512, 512)])
        self.snn_blocks = nn.ModuleList([
            MultiTimeConstantEIFNeuron(64, delta_T_init=1.0, theta_rh_init=0.8),
            MultiTimeConstantEIFNeuron(128, delta_T_init=1.0, theta_rh_init=0.8),
            MultiTimeConstantLIFNeuron(256),
            MultiTimeConstantLIFNeuron(512),
        ])
        self.multi_scale_first_conv = nn.ModuleList([_edge_conv(6, 64) for _ in k_scales])
        self.scale_fusion = nn.Sequential(nn.Conv1d(64 * len(k_scales), 64, 1, bias=False), nn.BatchNorm1d(64),
                                          nn.LeakyReLU(0.2))
        self.multi_scale_conv = nn.Sequential(nn.Conv1d(64 + 128 + 256 + 512, emb_dims, 1, bias=False),
                                              nn.BatchNorm1d(emb_dims), nn.LeakyReLU(0.2))
        self.snn_fc = MultiTimeConstantLIFNeuron(emb_dims)
        self.temporal_integration = TemporalIntegration(time_steps, emb_dims)


class StandardResidualBlock(nn.Module):
    def __init__(self, in_dim, out_dim, dropout=0.1):
        super().__init__()
        self.fc = nn.Sequential(nn.Linear(in_dim, out_dim), nn.BatchNorm1d(out_dim), nn.GELU(), nn.Dropout(dropout),
                                nn.Linear(out_dim, out_dim), nn.BatchNorm1d(out_dim))
        self.res_proj = nn.Linear(in_dim, out_dim) if in_dim != out_dim else None


class StandardSelfAttention(nn.Module):
    def __init__(self, dim, num_heads=4, dropout=0.1):
        super().__init__()
        self.to_qkv = nn.Linear(dim, dim * 3)
        self.to_out = nn.Sequential(nn.Linear(dim, dim), nn.Dropout(dropout))
        self.norm = nn.LayerNorm(dim)


class StandardDistanceDecoder(nn.Module):
    """Parameter container (reference fd/snn_coder.py:667-709)."""

    def __init__(self, input_dim=512, hidden_dims=(256, 128, 64), dropout=0.1, num_heads=4):
        super().__init__()
        self.fc_in = nn.Sequential(nn.Linear(input_dim, hidden_dims[0]), nn.BatchNorm1d(hidden_dims[0]), nn.GELU())
        self.residual_blocks = nn.ModuleList(
            [StandardResidualBlock(hidden_dims[i], hidden_dims[i + 1], dropout) for i in range(len(hidden_dims) - 1)])
        self.attention = StandardSelfAttention(hidden_dims[-1], num_heads=num_heads, dropout=dropout)
        self.fc_hidden = nn.Sequential(nn.Linear(hidden_dims[-1], 32), nn.BatchNorm1d(32), nn.GELU(), nn.Dropout(dropout))
        self.fc_distance = nn.Linear(32, 1)


class EnhancedSNNDistanceEstimation(NativeModel):
    KIND = N.MODEL_FD

    def __init__(self, k=20, emb_dims=512, time_steps_enc=5, time_steps_dec=8, num_heads=4, dropout=0.1,
                 use_snn_decoder=False, k_scales=(10, 20, 40)):
        super().__init__()
        if use_snn_decoder:
            raise N.SapcuError("use_snn_decoder=True (legacy spiking decoder) is outside the inference hot path")
        self.use_snn_decoder = False
        self.k, self.emb_dims, self.time_steps_enc, self.num_heads = k, emb_dims, time_steps_enc, num_heads
        self.k_scales = list(k_scales)
        self.encoder = EnhancedTemporalSNN_DGCNN_fd(k=k, emb_dims=emb_dims, time_steps=time_steps_enc, k_scales=k_scales)
        self.distance_decoder = StandardDistanceDecoder(emb_dims, (256, 128, 64), dropout=dropout, num_heads=num_heads)
        self.eval()

    def _cfg_ints(self):
        return [int(self.k), int(self.emb_dims), int(self.time_steps_enc), int(self.num_heads), len(self.k_scales)] + \
               [int(k) for k in self.k_scales]

    @torch.no_grad()
    def forward(self, Xc_rotated, forced_idx=None):
        """[B,M,3] -> [B];  [B,Np,M,3] -> [B,Np]  (reference fd/snn_coder.py:853-871).

        forced_idx (tests only): int32 [3,B,M,k] feature-space neighbour lists for blocks 1..3.
        """
        x = self._prep_input(Xc_rotated)
        lead = None
        if x.ndim == 4:
            B, Np, M, _ = x.shape
            lead = (B, Np)
            x = x.reshape(B * Np, M, 3)
        if x.ndim != 3:
            raise N.SapcuError("fd forward expects a 3-D or 4-D tensor, got shape %s" % (tuple(Xc_rotated.shape),))
        if x.shape[1] == 3:
            x = x.transpose(1, 2).contiguous()       # reference fd/snn_coder.py:393-394: shape[1] == 3 IS channel-first [B,3,M] (also for [B,3,3])
        if x.shape[2] != 3:
            raise N.SapcuError("fd forward: last dimension must be 3, got %s" % (tuple(x.shape),))
        S, M = x.shape[0], x.shape[1]
        out = torch.empty(S, dtype=torch.float32, device=x.device)
        if S:
            with torch.cuda.device(x.device):        # weights, workspace, stream and launches all on the input's device
                h = self._ensure_handle(x.device)
                ws, ws_bytes = self._workspace(S, M, x.device)
                if forced_idx is not None:
                    forced_idx = forced_idx.to(device=x.device, dtype=torch.int32).contiguous()
                N.check(N.lib().sapcu_fd_forward(h, N.ptr(x), S, M, N.ptr(out), N.ptr(forced_idx), N.ptr(ws), ws_bytes,
                                                 self.mode, N.stream_ptr(x.device)), "sapcu_fd_forward")
        return out.view(*lead) if lead else out
