"""Device context: one per (GPU, host thread).  Replaces `require 'cunn'` + the implicit cutorch
stream of the reference (VBLinear.lua:2, main.lua:1) and torch.manualSeed (config.lua:40).

PyTorch is used only as plumbing here: it owns the CUDA stream (made current for this thread so
that torch copies and libvbnn kernels are ordered) and the caller-side tensors."""
from __future__ import annotations

import ctypes as C

from . import _lib as L


class Context:
    def __init__(self, device: int = 0, seed: int = 3, stream_mode: int = L.STREAM_GIVEN):
        """stream_mode = L.STREAM_LEGACY_DEFAULT runs the library on stream 0, as a cunn module does
        (vbnn_ctx_create_ex); the default gives it a torch stream made current for this thread."""
        import torch
        if not torch.cuda.is_available():
            raise L.VbnnError(L.E_CUDA, "no CUDA device: vbnn_b200 has no CPU fallback")
        self.device = device
        torch.cuda.set_device(device)
        self.handle = C.c_void_p()
        if stream_mode == L.STREAM_GIVEN:
            self.stream = torch.cuda.Stream(device=device)
            torch.cuda.set_stream(self.stream)
            L.check(L.lib().vbnn_ctx_create_ex(device, C.c_void_p(self.stream.cuda_stream), stream_mode,
                                               C.c_uint64(seed), C.byref(self.handle)))
        else:
            self.stream = torch.cuda.default_stream(device)
            torch.cuda.set_stream(self.stream)
            L.check(L.lib().vbnn_ctx_create_ex(device, None, stream_mode, C.c_uint64(seed), C.byref(self.handle)))
        self.seed = seed
        self.rank, self.nranks = 0, 1

    def synchronize(self):
        L.check(L.lib().vbnn_ctx_synchronize(self.handle))

    def set_step(self, step: int):
        L.check(L.lib().vbnn_ctx_set_step(self.handle, C.c_uint32(step)))

    def get_step(self) -> int:
        v = C.c_uint32()
        L.check(L.lib().vbnn_ctx_get_step(self.handle, C.byref(v)))
        return int(v.value)

    def profile(self, enable: bool):
        L.check(L.lib().vbnn_ctx_profile(self.handle, 1 if enable else 0))

    def profile_read(self):
        """{class: (total_ms, launches, flops)} of the tensor-core GEMM launches, the fused update and the predict
        averaging kernel since profile(True)."""
        names = ["store", "fwd", "fwd_lrt", "dx", "dx_lrt", "dw", "dw_lrt", "update",
                 "predict"]                                   # update, predict: "flops" = bytes
        out = {}
        for cls, name in enumerate(names):
            ms, n, fl = C.c_double(), C.c_longlong(), C.c_double()
            L.check(L.lib().vbnn_ctx_profile_read(self.handle, cls, C.byref(ms), C.byref(n), C.byref(fl)))
            if n.value:
                out[name] = (ms.value, n.value, fl.value)
        return out

    def phase_read(self):
        """{phase: (total_ms, count)} between the step's phase marks since profile(True)."""
        names = {1: "wait_params", 2: "sample", 3: "forward", 4: "loss", 5: "backward", 6: "exchange_update", 7: "finalise"}
        out = {}
        for i, name in names.items():
            ms, n = C.c_double(), C.c_longlong()
            L.check(L.lib().vbnn_ctx_phase_read(self.handle, i, C.byref(ms), C.byref(n)))
            if n.value:
                out[name] = (ms.value, n.value)
        return out

    def close(self):
        if self.handle:
            L.lib().vbnn_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    # ---- data parallel (new: the reference is single-GPU) ----
    def init_comm(self, rank: int, nranks: int, broadcast_bytes):
        """broadcast_bytes(buf: bytes | None) -> bytes : broadcasts rank 0's 128-byte id."""
        buf = (C.c_char * 128)()
        if rank == 0:
            L.check(L.lib().vbnn_comm_unique_id(buf))
        raw = broadcast_bytes(bytes(buf) if rank == 0 else None)
        idbuf = (C.c_char * 128).from_buffer_copy(raw)
        L.check(L.lib().vbnn_comm_init(self.handle, idbuf, rank, nranks))
        self.rank, self.nranks = rank, nranks


_default_ctx = None


def default_context(device: int = 0, seed: int = 3) -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(device, seed)
    return _default_ctx


class DevView:
    """Zero-copy torch view of a device buffer owned by libvbnn (the reference's module fields
    such as `means` / `lvars` are live tensors; so are these)."""

    def __init__(self, ptr: int, shape):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr="<f4", data=(int(ptr), False),
                                             version=2, strides=None)


def as_dev_f32(x, device):
    """Caller tensor -> contiguous fp32 CUDA tensor (host data is copied, as inputs:cuda() did)."""
    import numpy as np
    import torch
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(x)
    return x.to(device=f"cuda:{device}", dtype=torch.float32, non_blocking=True).contiguous()
