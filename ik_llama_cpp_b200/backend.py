"""Host-side mirror of the reference's operator interface for the quantized mat-mul hot path.

The reference is compiled code whose operator boundary for this path is, per op node,
    ggml_cuda_mul_mat(ctx, src0 /*quantized [K, M]*/, src1 /*f32 [K, N]*/, dst /*f32 [M, N]*/)   ggml/src/ggml-cuda.cu:2645
    ggml_cuda_up_gate_unary(ctx, dst)  (GGML_OP_FUSED_UP_GATE)                                   ggml/src/ggml-cuda.cu:3542
and, for weights, ggml_backend_cuda_buffer_set_tensor / get_tensor (:641-672).  This module exposes the
same operations with the same names, argument meaning and error behaviour (raise = GGML_ABORT) on top of the
C ABI of libb200q.so.  PyTorch is used ONLY as the owner of device memory and streams; every FLOP of the
hot path runs in our CUDA kernels.  There is no CPU fallback: importing works anywhere, calling needs a GPU.
"""
from __future__ import annotations

import ctypes
from ctypes import c_int64, c_void_p
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import B200QError, check

# ggml_type ids (reference ggml/include/ggml.h:391-492) of the types the backend implements
GGML_TYPE = {"Q4_0": 2, "Q4_1": 3, "Q5_0": 6, "Q5_1": 7, "Q6_0": 133, "Q8_0": 8, "Q2_K": 10, "Q3_K": 11, "Q4_K": 12, "Q5_K": 13, "Q6_K": 14, "IQ4_NL": 20, "IQ4_XS": 23,
             "IQ2_BN": 135, "IQ2_K": 137, "IQ3_K": 138, "IQ4_K": 139, "IQ5_K": 140, "IQ4_KS": 144, "IQ5_KS": 152, "MXFP4": 39, "IQ2_KS": 145, "IQ3_KS": 156}
UNARY = {"none": 0, "silu": 1, "gelu": 2, "relu": 3, "swiglu_oai": 4}
MMVQ_MAX_BATCH_SIZE = 8          # ggml-cuda/mmvq.cuh:10 — n <= 8 takes the mat-vec path


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda() -> None:
    if not torch.cuda.is_available():
        raise B200QError("ik_llama_cpp_b200: the quantized mat-mul hot path needs a CUDA device (no CPU fallback)")


def type_supported(ggml_type: int) -> bool:
    return bool(_lib.lib().b200q_type_supported(ggml_type))


def row_size(ggml_type: int, k: int) -> int:
    r = _lib.lib().b200q_wire_row_size(ggml_type, k)
    if r < 0:
        raise B200QError(f"row_size: type {ggml_type} / K {k} unsupported")
    return int(r)


def plane_bytes(ggml_type: int, m: int, k: int) -> int:
    r = _lib.lib().b200q_plane_bytes(ggml_type, m, k)
    if r < 0:
        raise B200QError(f"plane_bytes: type {ggml_type} / shape ({m},{k}) unsupported")
    return int(r)


@dataclass
class QuantTensor:
    """A src0 of GGML_OP_MUL_MAT resident in HBM in the B200 plane layout (ne = [K, M] in ggml terms)."""
    ggml_type: int
    m: int            # rows  (ne[1])
    k: int            # cols  (ne[0])
    planes: torch.Tensor  # uint8, plane_bytes(type, m, k)

    @property
    def nbytes_wire(self) -> int:
        return self.m * row_size(self.ggml_type, self.k)

    @property
    def ptr(self) -> int:
        return self.planes.data_ptr()


def set_tensor(ggml_type: int, wire, m: int, k: int, device=None) -> QuantTensor:
    """ggml_backend_cuda_buffer_set_tensor: upload GGUF wire bytes (host numpy/bytes or a CUDA uint8 tensor)."""
    _require_cuda()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    nb = plane_bytes(ggml_type, m, k)
    planes = torch.zeros(nb, dtype=torch.uint8, device=device)   # alignment gaps between planes stay zero
    L = _lib.lib()
    with torch.cuda.device(device):
        if isinstance(wire, torch.Tensor) and wire.is_cuda:
            assert wire.dtype == torch.uint8 and wire.numel() == m * row_size(ggml_type, k)
            check(L.b200q_repack(ggml_type, wire.data_ptr(), planes.data_ptr(), m, k, _stream()), "b200q_repack")
        else:
            host = np.ascontiguousarray(np.frombuffer(wire, dtype=np.uint8) if not isinstance(wire, np.ndarray) else wire.view(np.uint8).ravel())
            assert host.size == m * row_size(ggml_type, k), (host.size, m * row_size(ggml_type, k))
            check(L.b200q_set_tensor(ggml_type, host.ctypes.data, planes.data_ptr(), m, k, _stream()), "b200q_set_tensor")
    return QuantTensor(ggml_type, m, k, planes)


def get_tensor(t: QuantTensor) -> np.ndarray:
    """ggml_backend_cuda_buffer_get_tensor: the original wire bytes, bit-for-bit."""
    _require_cuda()
    out = np.empty(t.nbytes_wire, np.uint8)
    with torch.cuda.device(t.planes.device):
        check(_lib.lib().b200q_get_tensor(t.ggml_type, t.ptr, out.ctypes.data, t.m, t.k, _stream()), "b200q_get_tensor")
    return out


_workspaces: dict[torch.device, torch.Tensor] = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    ws = _workspaces.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _workspaces[device] = ws
    return ws


def convert_activations(x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """f32 [N, K] -> bf16 [N, K] once, for several prefill MUL_MATs that share src1 (Q,K,V / up,gate)."""
    _require_cuda()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    n, k = x.shape
    xb = out if out is not None else torch.empty((n, k), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        check(_lib.lib().b200q_convert_f32_bf16(x.data_ptr(), x.stride(0), xb.data_ptr(), k, n, _stream()), "b200q_convert_f32_bf16")
    return xb


def prefetch_next(ws: "list[QuantTensor]", gate: "QuantTensor | None" = None) -> None:
    """Decode chains: announce the weights of the launch AFTER the next one (b200q_decode_prefetch_next): the next mat-vec warms them in L2."""
    L = _lib.lib()
    if not hasattr(L, "b200q_decode_prefetch_next"):
        return
    nt = len(ws)
    Wp = (c_void_p * nt)(*[w.ptr for w in ws]); Mp = (c_int64 * nt)(*[w.m for w in ws])
    check(L.b200q_decode_prefetch_next(ws[0].ggml_type, nt, Wp, gate.ptr if gate is not None else None, Mp, ws[0].k), "b200q_decode_prefetch_next")


class Q8Scratch:
    """Device scratch of the q8_1 hand-off FUSED_UP_GATE -> MUL_MAT (n = 1): b200q_q8_scratch_bytes(k), zeroed once."""

    def __init__(self, k: int, device=None):
        _require_cuda()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.k = k
        L = _lib.lib()
        self.supported = hasattr(L, "b200q_q8_scratch_bytes")          # (false only for an older library loaded through B200Q_LIB_PATH)
        self.buf = torch.zeros(int(L.b200q_q8_scratch_bytes(k)) if self.supported else 16, dtype=torch.uint8, device=device)
        self.valid = False          # set by fused_up_gate(q8_out=self): the image describes the latest result


def mul_mat(w: QuantTensor, x: torch.Tensor, out: torch.Tensor | None = None, x_bf16: torch.Tensor | None = None,
            q8_in: "Q8Scratch | None" = None) -> torch.Tensor:
    """GGML_OP_MUL_MAT: x f32 [N, K] -> dst f32 [N, M]  (ggml ne: src1 [K, N], dst [M, N]).
    x_bf16: optional result of convert_activations(x) (prefill only) to skip the per-call conversion.
    q8_in: n = 1 only, x was produced by fused_up_gate(q8_out=q8_in): consume its already quantised image."""
    _require_cuda()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.shape[1] == w.k and x.stride(1) == 1
    n = x.shape[0]
    dst = out if out is not None else torch.empty((n, w.m), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        if n == 1 and q8_in is not None and q8_in.valid and q8_in.k == w.k:
            check(L.b200q_mul_mat_vec_q8(w.ggml_type, w.ptr, x.data_ptr(), q8_in.buf.data_ptr(), dst.data_ptr(), w.m, w.k, None, _stream()), "b200q_mul_mat_vec_q8")
        elif n > MMVQ_MAX_BATCH_SIZE and x_bf16 is not None:
            assert x_bf16.dtype == torch.bfloat16 and x_bf16.shape == x.shape and x_bf16.is_contiguous()
            need = w.m * w.k * 2 + 256
            ws = _workspace(need, x.device)
            check(L.b200q_mul_mat_gemm_bf16(w.ggml_type, w.ptr, x_bf16.data_ptr(), dst.data_ptr(), w.m, w.k, n, ws.data_ptr(), ws.numel(), _stream()), "b200q_mul_mat_gemm_bf16")
        elif n <= MMVQ_MAX_BATCH_SIZE:
            check(L.b200q_mul_mat_vec(w.ggml_type, w.ptr, x.data_ptr(), dst.data_ptr(), w.m, w.k, n, x.stride(0), None, _stream()), "b200q_mul_mat_vec")
        else:
            xc = x if x.is_contiguous() else x.contiguous()
            need = L.b200q_mul_mat_workspace(w.ggml_type, w.m, w.k, n)
            ws = _workspace(need, x.device)
            check(L.b200q_mul_mat_gemm(w.ggml_type, w.ptr, xc.data_ptr(), dst.data_ptr(), w.m, w.k, n, ws.data_ptr(), ws.numel(), _stream()), "b200q_mul_mat_gemm")
    return dst


def mul_mat_multi(ws: list[QuantTensor], x: torch.Tensor, outs: list[torch.Tensor] | None = None,
                  x_bf16: torch.Tensor | None = None) -> list[torch.Tensor]:
    """Several MUL_MATs sharing src1 (Q,K,V) in one launch — the reference's look-ahead fusion, ggml-cuda.cu:2573-2601.
    n <= 8: one mat-vec launch over the row segments; n > 8: one GEMM launch over the row tiles of all tensors."""
    _require_cuda()
    n = x.shape[0]
    assert all(w.k == ws[0].k and w.ggml_type == ws[0].ggml_type for w in ws) and x.shape[1] == ws[0].k
    outs = outs or [torch.empty((n, w.m), dtype=torch.float32, device=x.device) for w in ws]
    nt = len(ws)
    Wp = (c_void_p * nt)(*[w.ptr for w in ws])
    Dp = (c_void_p * nt)(*[o.data_ptr() for o in outs])
    Mp = (c_int64 * nt)(*[w.m for w in ws])
    L = _lib.lib()
    with torch.cuda.device(x.device):
        if n <= MMVQ_MAX_BATCH_SIZE:
            check(L.b200q_mul_mat_vec_multi(ws[0].ggml_type, nt, Wp, Dp, Mp, ws[0].k, x.data_ptr(), n, x.stride(0), _stream()), "b200q_mul_mat_vec_multi")
        elif x_bf16 is not None:
            assert x_bf16.dtype == torch.bfloat16 and x_bf16.shape == x.shape and x_bf16.is_contiguous()
            wsb = _workspace(max(w.m for w in ws) * ws[0].k * 2 + 256, x.device)
            check(L.b200q_mul_mat_gemm_multi_bf16(ws[0].ggml_type, nt, Wp, Dp, Mp, ws[0].k, x_bf16.data_ptr(), n, wsb.data_ptr(), wsb.numel(), _stream()),
                  "b200q_mul_mat_gemm_multi_bf16")
        else:
            xc = x if x.is_contiguous() else x.contiguous()
            need = L.b200q_mul_mat_multi_workspace(ws[0].ggml_type, nt, Mp, ws[0].k, n)
            wsb = _workspace(need, x.device)
            check(L.b200q_mul_mat_multi(ws[0].ggml_type, nt, Wp, Dp, Mp, ws[0].k, xc.data_ptr(), n, wsb.data_ptr(), wsb.numel(), _stream()), "b200q_mul_mat_multi")
    return outs


def fused_up_gate(up: QuantTensor, gate: QuantTensor, x: torch.Tensor, unary: str = "silu", limit: float = 0.0,
                  out: torch.Tensor | None = None, x_bf16: torch.Tensor | None = None, out_bf16: torch.Tensor | None = None,
                  q8_out: "Q8Scratch | None" = None) -> torch.Tensor:
    """GGML_OP_FUSED_UP_GATE: dst = unary(gate.x) * (up.x).
    n <= 8: one mat-vec launch; n > 8: two GEMMs with the mul-unary in the gate GEMM's epilogue (the reference runs two MMQs +
    ggml_fused_mul_unary, ggml-cuda.cu:3588-3618).  x_bf16 / out_bf16 (prefill only): reuse an already converted activation /
    also emit the bf16 operand of the following ffn_down MUL_MAT."""
    _require_cuda()
    assert up.m == gate.m and up.k == gate.k and up.ggml_type == gate.ggml_type
    n = x.shape[0]
    dst = out if out is not None else torch.empty((n, up.m), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        if n == 1 and q8_out is not None and q8_out.supported and q8_out.k == up.m and x.is_contiguous():
            produced = ctypes.c_int32(0)
            check(L.b200q_fused_up_gate_vec_q8(up.ggml_type, up.ptr, gate.ptr, x.data_ptr(), dst.data_ptr(), up.m, up.k, UNARY[unary], float(limit),
                                               q8_out.buf.data_ptr(), ctypes.byref(produced), _stream()), "b200q_fused_up_gate_vec_q8")
            q8_out.valid = bool(produced.value)
        elif n <= MMVQ_MAX_BATCH_SIZE:
            if q8_out is not None:
                q8_out.valid = False
            check(L.b200q_fused_up_gate_vec(up.ggml_type, up.ptr, gate.ptr, x.data_ptr(), dst.data_ptr(), up.m, up.k, n,
                                            x.stride(0), UNARY[unary], float(limit), _stream()), "b200q_fused_up_gate_vec")
        elif x_bf16 is not None or out_bf16 is not None:
            xb = x_bf16 if x_bf16 is not None else convert_activations(x)
            assert xb.dtype == torch.bfloat16 and xb.shape == x.shape and xb.is_contiguous()
            if out_bf16 is not None:
                assert out_bf16.dtype == torch.bfloat16 and out_bf16.shape == dst.shape and out_bf16.is_contiguous()
            need = (up.m * n * 4 + 255) // 256 * 256 + up.m * up.k * 2 + 256
            ws = _workspace(need, x.device)
            check(L.b200q_fused_up_gate_gemm_bf16(up.ggml_type, up.ptr, gate.ptr, xb.data_ptr(), dst.data_ptr(),
                                                  out_bf16.data_ptr() if out_bf16 is not None else None, up.m, up.k, n,
                                                  UNARY[unary], float(limit), ws.data_ptr(), ws.numel(), _stream()), "b200q_fused_up_gate_gemm_bf16")
        else:
            xc = x if x.is_contiguous() else x.contiguous()
            need = L.b200q_fused_up_gate_workspace(up.ggml_type, up.m, up.k, n)
            ws = _workspace(need, x.device)
            check(L.b200q_fused_up_gate(up.ggml_type, up.ptr, gate.ptr, xc.data_ptr(), dst.data_ptr(), up.m, up.k, n,
                                        UNARY[unary], float(limit), ws.data_ptr(), ws.numel(), _stream()), "b200q_fused_up_gate")
    return dst


@dataclass
class ExpertTensor:
    """src0 of GGML_OP_MUL_MAT_ID: n_expert matrices [m x k] of one type (ggml ne = [K, M, n_expert]), each in the device layout."""
    ggml_type: int
    n_expert: int
    m: int
    k: int
    planes: torch.Tensor       # uint8 [n_expert * plane_bytes(type, m, k)]

    @property
    def ptr(self) -> int:
        return self.planes.data_ptr()


def set_expert_tensor(ggml_type: int, wire, n_expert: int, m: int, k: int, device=None) -> ExpertTensor:
    """Upload a 3-D expert tensor: every [m x k] matrix is re-laid-out on its own (what the backend plug's set_tensor does for ne[2] > 1)."""
    _require_cuda()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    pb, rs = plane_bytes(ggml_type, m, k), row_size(ggml_type, k)
    host = np.ascontiguousarray(np.frombuffer(wire, dtype=np.uint8) if not isinstance(wire, np.ndarray) else wire.view(np.uint8).ravel())
    assert host.size == n_expert * m * rs
    planes = torch.zeros(n_expert * pb, dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        for e in range(n_expert):
            check(_lib.lib().b200q_set_tensor(ggml_type, host[e * m * rs:].ctypes.data, planes.data_ptr() + e * pb, m, k, _stream()), "b200q_set_tensor")
    return ExpertTensor(ggml_type, n_expert, m, k, planes)


def _check_mul_mat_id(w: ExpertTensor, x: torch.Tensor, ids: torch.Tensor, gate: "ExpertTensor | None"):
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 3 and x.is_contiguous() and x.shape[2] == w.k
    assert ids.is_cuda and ids.dtype == torch.int32 and ids.dim() == 2 and ids.is_contiguous() and ids.shape[0] == x.shape[0]
    assert gate is None or (gate.ggml_type == w.ggml_type and gate.n_expert == w.n_expert and gate.m == w.m and gate.k == w.k)
    n_tokens, nb1, n_used = x.shape[0], x.shape[1], ids.shape[1]
    assert n_used % nb1 == 0
    return n_tokens, nb1, n_used


def mul_mat_id(w: ExpertTensor, x: torch.Tensor, ids: torch.Tensor, gate: "ExpertTensor | None" = None, unary: str = "silu", limit: float = 0.0,
               dispatch: bool = False) -> torch.Tensor:
    """GGML_OP_MUL_MAT_ID (gate is None) / GGML_OP_MOE_FUSED_UP_GATE: x f32 [n_tokens, nb1, K], ids int32 [n_tokens, n_used]
    -> dst f32 [n_tokens, n_used, M] with dst[t, e] = W[ids[t, e]] . x[t, e % nb1]  (gate: unary(gate[id] . x) * (W[id] . x)).
    dispatch=False: the mat-vec kernel at every batch size (b200q_mul_mat_id_vec); dispatch=True: what the graph nodes run (b200q_mul_mat_id:
    the grouped GEMM for large batches of the types it covers, the mat-vec kernel otherwise)."""
    _require_cuda()
    n_tokens, nb1, n_used = _check_mul_mat_id(w, x, ids, gate)
    dst = torch.empty((n_tokens, n_used, w.m), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        if dispatch:
            need = L.b200q_mul_mat_id_workspace(w.ggml_type, w.m, w.k, w.n_expert, n_used, nb1, n_tokens, int(gate is not None))
            ws = _workspace(need, x.device) if need else None
            check(L.b200q_mul_mat_id(w.ggml_type, w.ptr, gate.ptr if gate is not None else None, w.n_expert, ids.data_ptr(), x.data_ptr(), dst.data_ptr(),
                                     w.m, w.k, n_used, nb1, n_tokens, UNARY[unary], float(limit), ws.data_ptr() if ws is not None else None, need, _stream()),
                  "b200q_mul_mat_id")
        else:
            check(L.b200q_mul_mat_id_vec(w.ggml_type, w.ptr, gate.ptr if gate is not None else None, w.n_expert, ids.data_ptr(), x.data_ptr(), dst.data_ptr(),
                                         w.m, w.k, n_used, nb1, n_tokens, UNARY[unary], float(limit), _stream()), "b200q_mul_mat_id_vec")
    return dst


def mul_mat_id_gemm(w: ExpertTensor, x: torch.Tensor, ids: torch.Tensor, gate: "ExpertTensor | None" = None, unary: str = "silu", limit: float = 0.0,
                    out: torch.Tensor | None = None) -> torch.Tensor:
    """The same op as mul_mat_id through the grouped tcgen05 GEMM at any batch size (b200q_mul_mat_id_gemm): routing, gather and GEMM stay on
    the device, so the call can be captured in a CUDA graph.  Raises for types / shapes the grouped path does not cover."""
    _require_cuda()
    n_tokens, nb1, n_used = _check_mul_mat_id(w, x, ids, gate)
    dst = out if out is not None else torch.empty((n_tokens, n_used, w.m), dtype=torch.float32, device=x.device)
    assert dst.dtype == torch.float32 and dst.is_contiguous() and dst.shape == (n_tokens, n_used, w.m)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        need = L.b200q_mul_mat_id_workspace(w.ggml_type, w.m, w.k, w.n_expert, n_used, nb1, n_tokens, int(gate is not None))
        ws = _workspace(max(need, 1), x.device)
        check(L.b200q_mul_mat_id_gemm(w.ggml_type, w.ptr, gate.ptr if gate is not None else None, w.n_expert, ids.data_ptr(), x.data_ptr(), dst.data_ptr(),
                                      w.m, w.k, n_used, nb1, n_tokens, UNARY[unary], float(limit), ws.data_ptr(), ws.numel(), _stream()), "b200q_mul_mat_id_gemm")
    return dst


def dequantize_bf16(w: QuantTensor) -> torch.Tensor:
    _require_cuda()
    out = torch.empty((w.m, w.k), dtype=torch.bfloat16, device=w.planes.device)
    with torch.cuda.device(w.planes.device):
        check(_lib.lib().b200q_dequantize_bf16(w.ggml_type, w.ptr, out.data_ptr(), w.m, w.k, _stream()), "b200q_dequantize_bf16")
    return out


def mul_mat_host(w: QuantTensor, x_host: np.ndarray) -> np.ndarray:
    """End-to-end entry point with HOST activations and results (H2D + kernel + D2H inside the call)."""
    _require_cuda()
    x_host = np.ascontiguousarray(x_host, np.float32)
    n, k = x_host.shape
    assert k == w.k
    out = np.empty((n, w.m), np.float32)
    with torch.cuda.device(w.planes.device):
        check(_lib.lib().b200q_mul_mat_host(w.ggml_type, w.ptr, x_host.ctypes.data, out.ctypes.data, w.m, w.k, n, _stream()), "b200q_mul_mat_host")
    return out


class NvlsComm(ctypes.Structure):
    """struct b200q_nvls_comm of include/b200q.h"""
    _fields_ = [("ll_mc", c_void_p), ("ll_local", c_void_p), ("ll_reduced", c_void_p), ("ll_stride", c_int64),
                ("world_size", ctypes.c_uint32), ("rank", ctypes.c_uint32), ("ll_state", c_void_p), ("ll_peers", ctypes.POINTER(c_void_p))]


class NvlsStage(ctypes.Structure):
    """struct b200q_nvls_stage of include/b200q.h"""
    _fields_ = [("mc_stage", c_void_p), ("local_stage", c_void_p), ("stage_elems", c_int64), ("mc_flag", c_void_p), ("local_flag", c_void_p),
                ("world_size", ctypes.c_uint32), ("rank", ctypes.c_uint32), ("state", c_void_p)]


def mul_mat_vec_tp(ws: list[QuantTensor], x: torch.Tensor | None, outs: list[torch.Tensor] | None, reducer: "NvlsReducer",
                   reduce_in: bool = False, reduce_out: bool = False, gate: QuantTensor | None = None, unary: str = "silu", limit: float = 0.0):
    """Tensor-parallel decode (n = 1) with GGML_OP_REDUCE fused into the mat-vec kernels (b200q_mul_mat_vec_tp).
    reduce_out: the partial rows are summed across ranks inside the NVSwitch into the reducer's buffer (outs may be None);
    reduce_in:  the activations are the result of the previous reduce_out launch (x may be None)."""
    _require_cuda()
    nt = len(ws)
    assert all(w.k == ws[0].k and w.ggml_type == ws[0].ggml_type for w in ws)
    if x is not None:
        assert x.is_cuda and x.dtype == torch.float32 and x.shape == (1, ws[0].k) and x.is_contiguous()
    Wp = (c_void_p * nt)(*[w.ptr for w in ws])
    Dp = (c_void_p * nt)(*[o.data_ptr() for o in outs]) if outs is not None else None
    Mp = (c_int64 * nt)(*[w.m for w in ws])
    dev = ws[0].planes.device
    with torch.cuda.device(dev):
        check(_lib.lib().b200q_mul_mat_vec_tp(ws[0].ggml_type, nt, Wp, gate.ptr if gate is not None else None, Dp, Mp, ws[0].k,
                                              x.data_ptr() if x is not None else None, UNARY[unary], float(limit),
                                              ctypes.byref(reducer.comm()), int(reduce_in), int(reduce_out), _stream()), "b200q_mul_mat_vec_tp")
    return outs


class NvlsReducer:
    """GGML_OP_REDUCE (sum) across the ranks of a torch.distributed group with the in-tree NVLS kernel (b200q_reduce_sum_nvls).
    Symmetric memory + multicast mapping come from torch.distributed._symmetric_memory (plumbing); the reduction itself is
    our kernel: multimem.red into the switch, flag, acquire-spin, copy-out.  Falls back to NCCL all_reduce when the
    platform has no multicast support."""

    LL_STRIDE = 16384        # longest vector of a fused decode reduce (entries)

    def __init__(self, max_elems: int, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.dist = dist
        self.group = group or dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.stride = (max_elems + 3) // 4 * 4
        dev = torch.device("cuda", torch.cuda.current_device())
        self.ok = False
        try:
            # [2 parity buffers of `stride` f32][64 f32: flag words][bf16 staging of `stride` elements (two-shot all-reduce)]
            # [tagged slots of the fused decode reduce: 2 parities x world x LL_STRIDE entries of {f32, u32}]
            self.ll_stride = self.LL_STRIDE
            base_floats = (2 * self.stride + 64 + (self.stride + 1) // 2 + 3) // 4 * 4
            self.buf = symm.empty(base_floats + 2 * self.world * self.ll_stride * 2, dtype=torch.float32, device=dev)
            self.hdl = symm.rendezvous(self.buf, self.group)
            self.mc = int(self.hdl.multicast_ptr) if self.hdl.has_multicast_support else 0
            if self.mc:
                self.buf.zero_()
                self.local = self.buf.data_ptr()
                self.flag_off = 2 * self.stride * 4
                self.state = torch.zeros(16, dtype=torch.int32, device=dev)     # [0] seq counter, [4] cta counter, [8..11] two-shot state
                self.rank = dist.get_rank(self.group)
                self.flag2_off = self.flag_off + 128                          # second flag word (own 128-byte line): two-shot bf16 all-reduce
                self.stage_off = (2 * self.stride + 64) * 4
                self.ll_off = base_floats * 4
                self.ll_reduced = torch.zeros(2 * self.ll_stride * 2, dtype=torch.float32, device=dev)    # rank-local: published sums {f32, tag}
                torch.cuda.synchronize()
                self.hdl.barrier()
                self.ok = True
        except Exception as e:  # no symmetric memory / multicast on this platform
            self.err = repr(e)
        if not self.ok:
            self.mc = 0

    def comm(self):
        """ctypes b200q_nvls_comm for the fused tensor-parallel mat-vec (b200q_mul_mat_vec_tp)."""
        assert self.ok
        if not hasattr(self, "_comm"):
            peers = None
            try:        # every rank's mapping of the symmetric buffer (peer memory): unicast variant of the tagged-slot exchange
                ptrs = [int(p) for p in self.hdl.buffer_ptrs]
                if len(ptrs) == self.world and self.world <= 8 and all(ptrs):
                    self._peer_arr = (c_void_p * self.world)(*[p + self.ll_off for p in ptrs])
                    peers = ctypes.cast(self._peer_arr, ctypes.POINTER(c_void_p))
            except Exception:
                peers = None
            self._comm = NvlsComm(self.mc + self.ll_off, self.local + self.ll_off, self.ll_reduced.data_ptr(), self.ll_stride, self.world, self.rank,
                                  self.state.data_ptr() + 48, peers)
        return self._comm

    def reduced_view(self, n: int) -> torch.Tensor:
        """The summed vector of the latest fused reduce, rebuilt from this rank's copy of the tagged slots exactly as the consumer kernels do
        (f32, rank order): debugging / tests only (synchronises)."""
        torch.cuda.synchronize()
        seq = int(self.state[12].item())
        par = (seq - 1) & 1
        o = self.ll_off // 4
        ent = self.buf[o: o + 2 * self.world * self.ll_stride * 2].view(2, self.world, self.ll_stride, 2)[par, :, :n]
        assert bool((ent[:, :, 1].contiguous().view(torch.int32) == seq).all()), "not every rank's rows of the latest reduce have arrived"
        acc = ent[0, :, 0].clone()
        for r in range(1, self.world):
            acc = acc + ent[r, :, 0]
        return acc

    def stage(self):
        """ctypes b200q_nvls_stage for b200q_reduce_sum_nvls_bf16."""
        assert self.ok
        if not hasattr(self, "_stage"):
            self._stage = NvlsStage(self.mc + self.stage_off, self.local + self.stage_off, self.stride, self.mc + self.flag2_off, self.local + self.flag2_off,
                                    self.world, self.rank, self.state.data_ptr() + 32)
        return self._stage

    def all_reduce_bf16(self, t: torch.Tensor, out_bf16: torch.Tensor | None = None, out_f32: torch.Tensor | None = None):
        """Sum over ranks of a contiguous f32 tensor with a bf16 payload (two-shot, in the switch): the reference's reduce for ne[1] > 32.
        out_bf16: bf16 result (activation operand of the next GEMM); out_f32: f32 result (may alias t).  At least one."""
        assert self.ok and t.dtype == torch.float32 and t.is_contiguous() and t.numel() % 8 == 0 and t.numel() <= self.stride
        assert out_bf16 is not None or out_f32 is not None
        if out_bf16 is not None:
            assert out_bf16.dtype == torch.bfloat16 and out_bf16.is_contiguous() and out_bf16.numel() == t.numel()
        if out_f32 is not None:
            assert out_f32.dtype == torch.float32 and out_f32.is_contiguous() and out_f32.numel() == t.numel()
        check(_lib.lib().b200q_reduce_sum_nvls_bf16(t.data_ptr(), out_f32.data_ptr() if out_f32 is not None else None,
                                                    out_bf16.data_ptr() if out_bf16 is not None else None, t.numel(), ctypes.byref(self.stage()), _stream()),
              "b200q_reduce_sum_nvls_bf16")
        return out_bf16 if out_bf16 is not None else out_f32

    def all_reduce(self, t: torch.Tensor) -> torch.Tensor:
        """In-place sum over ranks of a contiguous f32 tensor."""
        if not self.ok or t.numel() > self.stride:
            self.dist.all_reduce(t, group=self.group)
            return t
        assert t.dtype == torch.float32 and t.is_contiguous()
        L = _lib.lib()
        check(L.b200q_reduce_sum_nvls(t.data_ptr(), t.data_ptr(), t.numel(), self.mc, self.local, self.stride,
                                      self.mc + self.flag_off, self.local + self.flag_off, self.world,
                                      self.state.data_ptr(), self.state.data_ptr() + 16, _stream()), "b200q_reduce_sum_nvls")
        return t
