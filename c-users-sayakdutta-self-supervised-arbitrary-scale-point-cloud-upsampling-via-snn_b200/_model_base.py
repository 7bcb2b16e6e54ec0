"""Shared machinery of the two model shims: a torch nn.Module that owns the reference-shaped parameters
(so state_dict()/load_state_dict()/CheckpointIO keep working) and forwards through the C ABI.

torch is plumbing here: parameter containers, device memory for inputs/outputs/workspace, the stream.
"""
import ctypes
import threading

import torch
import torch.nn as nn

from . import _native as N


class NativeModel(nn.Module):
    KIND = None            # N.MODEL_FN / N.MODEL_FD
    #: bytes of workspace the shim is willing to allocate per forward (chunks internally below that)
    WORKSPACE_CAP = int(float(__import__('os').environ.get('SAPCU_WS_CAP_GB', '24')) * (1 << 30))

    def __init__(self):
        super().__init__()
        self._owner = None          # DataParallel replicas: the module whose handles and workspaces they use
        self._handles = {}          # device index -> (state version, native handle), built from this module's parameters
        self._workspaces = {}       # (device index, cudaStream_t) -> uint8 workspace tensor
        self._lock = threading.Lock()
        self._ws_last = None
        self.mode = N.MODE_FP32

    # ------------------------------------------------------------------ handle management
    def _cfg_ints(self):
        raise NotImplementedError

    def _state_version(self):
        # parameters/buffers are re-uploaded when any of them was modified in place or replaced
        return tuple((k, v.data_ptr(), v._version) for k, v in self.state_dict(keep_vars=True).items())

    def _root(self):
        return self if self._owner is None else self._owner

    def _ensure_handle(self, device=None):
        """The native handle for the module's current parameters on `device` (default: the current CUDA device).  The weights
        are uploaded to the device that is current at finalize time and the handle only runs there, so callers hold
        torch.cuda.device(device).  One handle per device, built once per parameter version; a DataParallel replica gets
        its owner's handle, built from the owner's parameters."""
        owner = self._root()
        dev_index = torch.device(device).index if device is not None else None
        if dev_index is None:
            dev_index = torch.cuda.current_device() if torch.cuda.is_available() else -1
        ver = owner._state_version()
        with owner._lock:
            cur = owner._handles.get(dev_index)
            if cur is not None and cur[0] == ver:
                return cur[1]
            if cur is not None:
                del owner._handles[dev_index]
                N.lib().sapcu_model_destroy(cur[1])
            h = owner._build_handle()
            owner._handles[dev_index] = (ver, h)
            return h

    def _build_handle(self):
        L = N.lib()
        cfg = (ctypes.c_int32 * len(self._cfg_ints()))(*self._cfg_ints())
        h = L.sapcu_model_create(self.KIND, cfg, len(cfg))
        if not h:
            raise N.SapcuError("sapcu_model_create: " + L.sapcu_last_error().decode())
        try:
            for name, t in self.state_dict().items():
                if not t.dtype.is_floating_point:
                    continue   # num_batches_tracked
                host = t.detach().to("cpu", torch.float32).contiguous()
                N.check(L.sapcu_model_set_tensor(h, name.encode(), N.ptr(host), host.numel()), "set_tensor(%s)" % name)
            N.check(L.sapcu_model_finalize(h), "sapcu_model_finalize")
        except Exception:
            L.sapcu_model_destroy(h)
            raise
        return h

    def __del__(self):
        if self.__dict__.get("_owner") is not None or not self.__dict__.get("_handles"):
            return                  # a replica owns nothing
        try:
            handles, self._handles = self._handles, {}
            L = N.lib()
            for _, h in handles.values():
                L.sapcu_model_destroy(h)
        except Exception:
            pass

    def _replicate_for_data_parallel(self):
        replica = super()._replicate_for_data_parallel()
        replica.__dict__["_owner"] = self._root()       # plain attribute: not a registered submodule
        replica.__dict__["_ws_last"] = None
        return replica

    def __getstate__(self):
        # copies (copy.deepcopy, pickle) start without native state: a handle belongs to exactly one module
        state = self.__dict__.copy()
        state.update(_owner=None, _handles={}, _workspaces={}, _lock=None, _ws_last=None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self._lock = threading.Lock()

    # ------------------------------------------------------------------ reference API surface
    def reset_states(self):
        """No-op: the reference's reset_states() has no effect on eval outputs (SURVEY.md a19)."""
        return None

    def train(self, mode=True):
        if mode:
            raise N.SapcuError("sapcu_b200 implements the inference hot path only (eval mode)")
        return super().train(False)

    def set_mode(self, mode):
        """'fp32' (FFMA, reference-faithful arithmetic), 'tc' (tcgen05 split products, parity-grade), 'tf32' (tcgen05
        single-pass TF32) or 'fast' (single fp16 product per MAC on fp16 spike tensors + cheap LIF chains; the fast mode
        whose deviation is reported separately)."""
        self.mode = {"fp32": N.MODE_FP32, "tc": N.MODE_TC, "tf32": N.MODE_TF32, "fast": N.MODE_FAST}[mode] if isinstance(mode, str) else int(mode)
        return self

    # ------------------------------------------------------------------ helpers for subclasses
    @property
    def _ws(self):
        """The workspace of the most recent forward on this module (what tap() reads).  Setting it to None also releases
        the cached workspaces, so that the next forward allocates under the current WORKSPACE_CAP."""
        return self._ws_last

    @_ws.setter
    def _ws(self, value):
        if value is None:
            self._root()._workspaces.clear()
        self._ws_last = value

    def _workspace(self, S, M, device):
        """(workspace tensor, bytes to pass to the forward).  Workspaces are cached per (device, stream): calls on one stream
        run in order and may share one, calls on two streams never do.  The byte count is max(one patch, min(need,
        WORKSPACE_CAP)) whatever the cached tensor's size, so WORKSPACE_CAP alone decides the chunking."""
        L = N.lib()
        h = self._ensure_handle(device)
        need = L.sapcu_model_workspace_bytes(h, S, M)
        one = L.sapcu_model_workspace_bytes(h, 1, M)
        want = max(one, min(need, self.WORKSPACE_CAP))
        owner = self._root()
        key = (device.index, torch.cuda.current_stream(device).cuda_stream)
        with owner._lock:
            ws = owner._workspaces.get(key)
            if ws is None or ws.numel() < want:
                owner._workspaces.pop(key, None)
                ws = torch.empty(want, dtype=torch.uint8, device=device)
                owner._workspaces[key] = ws
        self._ws_last = ws
        return ws, want

    def _prep_input(self, x):
        if not x.is_cuda:
            raise N.SapcuError("sapcu_b200 models run on CUDA tensors only (no CPU fallback); got a %s tensor" % x.device)
        return x.detach().to(torch.float32).contiguous()

    def tap(self, name, S, M, dtype=torch.float32):
        """Debug view of a named intermediate of the last forward (tests only)."""
        off, rows, cols, ld = (ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64())
        N.check(N.lib().sapcu_model_tap(self._ensure_handle(), name.encode(), S, M, self.mode, ctypes.byref(off), ctypes.byref(rows),
                                        ctypes.byref(cols), ctypes.byref(ld)), "model_tap(%s)" % name)
        fmt = N.lib().sapcu_model_tap_format(self._ensure_handle(), name.encode())
        if fmt == 1:      # fp16 (hi, lo) planes of x * 2^13 (see include/sapcu_b200.h)
            n = rows.value * cols.value
            h = self._ws.view(torch.float16)[2 * off.value: 2 * off.value + 2 * n].view(2, rows.value, cols.value)
            return (h[0].float() + h[1].float()) / 8192.0
        if fmt == 2:      # fast mode: ONE fp16 plane of x * 2^13
            n = rows.value * cols.value
            h = self._ws.view(torch.float16)[2 * off.value: 2 * off.value + n].view(rows.value, cols.value)
            return h.float() / 8192.0
        flat = self._ws.view(torch.float32) if dtype == torch.float32 else self._ws.view(torch.int32)
        return flat[off.value: off.value + rows.value * ld.value].view(rows.value, ld.value)[:, :cols.value]
