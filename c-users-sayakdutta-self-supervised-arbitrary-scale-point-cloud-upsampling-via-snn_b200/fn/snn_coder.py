"""ImprovedSNNNormalEstimation -- B200-native drop-in for the reference class of the same name
(reference: fn/snn_coder.py:627-738).

The module tree below exists only to reproduce the reference's parameter names and shapes
(`encoder.conv1.0.weight`, `encoder.trans2.snn_gamma.threshold_base`, `decoder.mlp.4.bias`, ... --
SURVEY.md section 8b) so that `state_dict()`, `load_state_dict()` and `CheckpointIO` work unchanged.
`forward` hands the whole network to `sapcu_fn_forward` (csrc/forward.cu); nothing is computed in Python.
"""
import torch
import torch.nn as nn

from .. import _native as N
from .._model_base import NativeModel
from ..neurons import MultiTimeConstantLIFNeuron


def _conv_bn(cin, cout, two_d=False):
    conv = nn.Conv2d(cin, cout, 1) if two_d else nn.Conv1d(cin, cout, 1)
    bn = nn.BatchNorm2d(cout) if two_d else nn.BatchNorm1d(cout)
    return nn.Sequential(conv, bn)


class MultiHeadSNNTransformerBlock(nn.Module):
    """Parameter container of one SNN point-transformer block (reference fn/snn_coder.py:212-292)."""

    def __init__(self, d_points, d_model, k, time_steps, num_heads=4, dropout=0.1):
        super().__init__()
        assert d_model % num_heads == 0, "d_model must be divisible by num_heads"
        self.k, self.time_steps, self.num_heads, self.d_model = k, time_steps, num_heads, d_model
        self.fc1 = _conv_bn(d_points, d_model)
        self.snn1 = MultiTimeConstantLIFNeuron(d_model)
        self.fc2 = _conv_bn(d_model, d_points)
        self.fc_delta = _conv_bn(3, d_model, two_d=True)
        self.snn_delta = MultiTimeConstantLIFNeuron(d_model)
        self.fc_delta2 = _conv_bn(d_model, d_model, two_d=True)
        self.snn_delta2 = MultiTimeConstantLIFNeuron(d_model)
        self.fc_gamma = _conv_bn(d_model, d_model, two_d=True)
        self.snn_gamma = MultiTimeConstantLIFNeuron(d_model)
        self.fc_gamma2 = _conv_bn(d_model, d_model, two_d=True)
        self.w_qs = _conv_bn(d_model, d_model)
        self.snn_q = MultiTimeConstantLIFNeuron(d_model)
        self.w_ks = _conv_bn(d_model, d_model)
        self.snn_k = MultiTimeConstantLIFNeuron(d_model)
        self.w_vs = _conv_bn(d_model, d_model)
        self.snn_v = MultiTimeConstantLIFNeuron(d_model)
        self.out_proj = _conv_bn(d_model, d_model)


class ImprovedSNNEncoder(nn.Module):
    """Parameter container (reference fn/snn_coder.py:405-428); block widths 128/256/512 and T=4 are fixed there."""

    def __init__(self, emb_dims=1024, k_values=(20, 20, 16), time_steps=8, num_heads=4):
        super().__init__()
        self.time_steps, self.k_values = time_steps, list(k_values)
        self.conv1 = _conv_bn(3, 64)
        self.snn_init = MultiTimeConstantLIFNeuron(64)
        self.trans1 = MultiHeadSNNTransformerBlock(64, 128, k=k_values[0], time_steps=4, num_heads=num_heads)
        self.trans2 = MultiHeadSNNTransformerBlock(64, 256, k=k_values[1], time_steps=4, num_heads=num_heads)
        self.trans3 = MultiHeadSNNTransformerBlock(64, 512, k=k_values[2], time_steps=4, num_heads=num_heads)
        self.conv_final = _conv_bn(64 * 3, emb_dims)
        self.snn_final = MultiTimeConstantLIFNeuron(emb_dims)
        self.fc_out = nn.Linear(emb_dims, 2048)


class StandardNormalDecoder(nn.Module):
    """Parameter container (reference fn/snn_coder.py:517-540): mlp indices 0,1,4,5,8,9 hold parameters."""

    def __init__(self, input_dim=2048, output_dim=3, hidden_dims=(1024, 512, 256), dropout=0.1):
        super().__init__()
        layers, d = [], input_dim
        for h in hidden_dims:
            layers += [nn.Linear(d, h), nn.BatchNorm1d(h), nn.GELU()]
            if dropout > 0:
                layers.append(nn.Dropout(dropout))
            d = h
        self.mlp = nn.Sequential(*layers)
        self.fc_out = nn.Linear(hidden_dims[-1], output_dim)
        self.norm_out = nn.LayerNorm(output_dim)


class ImprovedSNNNormalEstimation(NativeModel):
    KIND = N.MODEL_FN

    def __init__(self, k_values=(20, 20, 16), emb_dims=1024, time_steps_enc=8, time_steps_dec=12, num_heads=4,
                 use_snn_decoder=False, decoder_dropout=0.1):
        super().__init__()
        if use_snn_decoder:
            raise N.SapcuError("use_snn_decoder=True (legacy spiking decoder) is outside the inference hot path")
        if decoder_dropout <= 0:
            raise N.SapcuError("decoder_dropout must be > 0 to keep the reference's mlp.{0,1,4,5,8,9} parameter names")
        self.use_snn_decoder = False
        self.k_values, self.emb_dims = list(k_values), emb_dims
        self.time_steps_enc, self.num_heads = time_steps_enc, num_heads
        self.encoder = ImprovedSNNEncoder(emb_dims=emb_dims, k_values=k_values, time_steps=time_steps_enc,
                                          num_heads=num_heads)
        self.decoder = StandardNormalDecoder(2048, 3, (1024, 512, 256), dropout=decoder_dropout)
        self.eval()

    def _cfg_ints(self):
        return [int(k) for k in self.k_values] + [int(self.emb_dims), int(self.time_steps_enc), int(self.num_heads)]

    @torch.no_grad()
    def forward(self, point_cloud, _stop_after_block=0):
        """[B,M,3] | [B,3,M] -> [B,3];  [B,Np,M,3] -> [B,Np,3]  (reference fn/snn_coder.py:670-699)."""
        x = self._prep_input(point_cloud)
        lead = None
        if x.ndim == 4:
            B, Np, M, C = x.shape
            lead = (B, Np)
            x = x.reshape(B * Np, M, C)
        if x.ndim != 3:
            raise N.SapcuError("fn forward expects a 3-D or 4-D tensor, got shape %s" % (tuple(point_cloud.shape),))
        if x.shape[1] == 3 and x.shape[2] != 3:
            x = x.permute(0, 2, 1).contiguous()      # [B,3,M] layout (reference fn/snn_coder.py:441-444)
        if x.shape[2] != 3:
            raise N.SapcuError("fn forward: last dimension must be 3, got %s" % (tuple(x.shape),))
        S, M = x.shape[0], x.shape[1]
        out = torch.empty(S, 3, dtype=torch.float32, device=x.device)
        if S:
            with torch.cuda.device(x.device):        # weights, workspace, stream and launches all on the input's device
                h = self._ensure_handle(x.device)
                ws, ws_bytes = self._workspace(S, M, x.device)
                N.check(N.lib().sapcu_fn_forward(h, N.ptr(x), S, M, N.ptr(out), N.ptr(ws), ws_bytes, self.mode | (int(_stop_after_block) << 8),
                                                 N.stream_ptr(x.device)), "sapcu_fn_forward")
        return out.view(*lead, 3) if lead else out

    @torch.no_grad()
    def forward_indexed(self, patches, cloud, gidx):
        """forward() of [S,M,3] patches whose point i of patch s is row gidx[s,i] of `cloud` (f64 [N,3]; the patches are
        cloud[gidx] - seed): the positional encoding is then evaluated once per distinct pair of cloud points
        (sapcu_fn_forward_indexed).  gidx: int32 [S, >= M] on the patches' device, rows may be strided."""
        x = self._prep_input(patches)
        if x.ndim != 3 or x.shape[2] != 3:
            raise N.SapcuError("fn forward_indexed expects [S,M,3] patches, got shape %s" % (tuple(patches.shape),))
        if cloud.dtype != torch.float64 or cloud.ndim != 2 or cloud.shape[1] != 3 or not cloud.is_contiguous():
            raise N.SapcuError("fn forward_indexed: cloud must be a contiguous float64 [N,3] tensor")
        S, M = x.shape[0], x.shape[1]
        if gidx.dtype != torch.int32 or gidx.ndim != 2 or gidx.shape[0] != S or gidx.shape[1] < M or gidx.stride(1) != 1:
            raise N.SapcuError("fn forward_indexed: gidx must be int32 [S, >= M] with unit column stride")
        if cloud.device != x.device or gidx.device != x.device:
            raise N.SapcuError("fn forward_indexed: patches, cloud and gidx must share a device")
        out = torch.empty(S, 3, dtype=torch.float32, device=x.device)
        if S:
            with torch.cuda.device(x.device):
                h = self._ensure_handle(x.device)
                ncl = cloud.shape[0]
                ws, ws_bytes = self._workspace(S, M, x.device, ncloud=ncl)
                N.check(N.lib().sapcu_fn_forward_indexed(h, N.ptr(x), S, M, N.ptr(cloud), ncl, N.ptr(gidx), gidx.stride(0), N.ptr(out),
                                                         N.ptr(ws), ws_bytes, self.mode, N.stream_ptr(x.device)), "sapcu_fn_forward_indexed")
        return out
