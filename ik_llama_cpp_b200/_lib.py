"""ctypes binding of libb200q.so (the product).  Fails loudly if the CUDA library is missing: no CPU fallback."""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p, POINTER

HERE = os.path.dirname(os.path.abspath(__file__))
# B200Q_LIB_PATH: tuning experiments only (a variant of the same library built with other -D knobs, scripts/build_variant.sh)
LIB_PATH = os.environ.get("B200Q_LIB_PATH") or os.path.join(HERE, "libb200q.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "b200q.h")


class B200QError(RuntimeError):
    pass


_lib = None


def header_symbols() -> list[str]:
    """Every function include/b200q.h declares (used by the ABI-completeness test)."""
    with open(HEADER) as f:
        src = f.read()
    return sorted(set(re.findall(r"B200Q_API\s+[\w\s\*]+?\b(b200q_\w+)\s*\(", src)))


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200QError(f"{LIB_PATH} is missing: build it with `python -m ik_llama_cpp_b200.build` "
                         "(there is no CPU / PyTorch fallback for the hot path)")
    L = ctypes.CDLL(LIB_PATH)
    vp, i64, i32 = c_void_p, c_int64, c_int
    L.b200q_abi_version.restype = i32
    L.b200q_last_error.restype = c_char_p
    L.b200q_device_count.restype = i32
    L.b200q_set_option.argtypes = [c_char_p, i32]
    L.b200q_type_supported.argtypes = [i32]
    L.b200q_wire_row_size.restype = i64
    L.b200q_wire_row_size.argtypes = [i32, i64]
    L.b200q_plane_bytes.restype = i64
    L.b200q_plane_bytes.argtypes = [i32, i64, i64]
    for name in ("b200q_repack", "b200q_unrepack", "b200q_set_tensor", "b200q_get_tensor"):
        getattr(L, name).argtypes = [i32, vp, vp, i64, i64, vp]
    L.b200q_mul_mat_vec.argtypes = [i32, vp, vp, vp, i64, i64, i32, i64, vp, vp]
    L.b200q_mul_mat_vec_multi.argtypes = [i32, i32, POINTER(vp), POINTER(vp), POINTER(i64), i64, vp, i32, i64, vp]
    L.b200q_fused_up_gate_vec.argtypes = [i32, vp, vp, vp, vp, i64, i64, i32, i64, i32, c_float, vp]
    L.b200q_mul_mat_workspace.restype = c_size_t
    L.b200q_mul_mat_workspace.argtypes = [i32, i64, i64, i64]
    L.b200q_mul_mat_gemm.argtypes = [i32, vp, vp, vp, i64, i64, i64, vp, c_size_t, vp]
    L.b200q_dequantize_bf16.argtypes = [i32, vp, vp, i64, i64, vp]
    L.b200q_convert_f32_bf16.argtypes = [vp, i64, vp, i64, i64, vp]
    L.b200q_mul_mat_gemm_bf16.argtypes = [i32, vp, vp, vp, i64, i64, i64, vp, c_size_t, vp]
    L.b200q_mul_mat_gemm_multi_bf16.argtypes = [i32, i32, vp, vp, vp, i64, vp, i64, vp, c_size_t, vp]
    L.b200q_fused_up_gate_gemm_bf16.argtypes = [i32, vp, vp, vp, vp, vp, i64, i64, i64, i32, c_float, vp, c_size_t, vp]
    L.b200q_mul_mat_multi_workspace.restype = c_size_t
    L.b200q_mul_mat_multi_workspace.argtypes = [i32, i32, vp, i64, i64]
    L.b200q_mul_mat_multi.argtypes = [i32, i32, vp, vp, vp, i64, vp, i64, vp, c_size_t, vp]
    L.b200q_fused_up_gate_workspace.restype = c_size_t
    L.b200q_fused_up_gate_workspace.argtypes = [i32, i64, i64, i64]
    L.b200q_fused_up_gate.argtypes = [i32, vp, vp, vp, vp, i64, i64, i64, i32, c_float, vp, c_size_t, vp]
    L.b200q_mul_mat_vec_tp.argtypes = [i32, i32, vp, vp, vp, vp, i64, vp, i32, c_float, vp, i32, i32, vp]
    L.b200q_reduce_sum_nvls.argtypes = [vp, vp, i64, vp, vp, i64, vp, vp, ctypes.c_uint32, vp, vp, vp]
    L.b200q_mul_mat.argtypes = [i32, vp, vp, vp, i64, i64, i64, vp, c_size_t, vp]
    L.b200q_mul_mat_host.argtypes = [i32, vp, vp, vp, i64, i64, i64, vp]
    if os.environ.get("B200Q_LIB_PATH") and not hasattr(L, "b200q_reduce_sum_nvls_bf16"):
        _lib = L                    # an older build loaded for an A/B experiment (scripts/sweep_decode.py): only the round-1 entry points
        return L
    L.b200q_q8_scratch_bytes.restype = c_size_t
    L.b200q_q8_scratch_bytes.argtypes = [i64]
    L.b200q_q8_scratch_init.argtypes = [vp, i64, vp]
    L.b200q_fused_up_gate_vec_q8.argtypes = [i32, vp, vp, vp, vp, i64, i64, i32, c_float, vp, POINTER(i32), vp]
    L.b200q_mul_mat_vec_q8.argtypes = [i32, vp, vp, vp, vp, i64, i64, vp, vp]
    L.b200q_reduce_sum_nvls_bf16.argtypes = [vp, vp, vp, i64, vp, vp]
    if hasattr(L, "b200q_mul_mat_id_vec"):
        L.b200q_mul_mat_id_vec.argtypes = [i32, vp, vp, i32, vp, vp, vp, i64, i64, i32, i32, i32, i32, c_float, vp]
        L.b200q_add_rows.argtypes = [vp, vp, vp, i64, i64, i64, vp]
    if hasattr(L, "b200q_mul_mat_id_gemm"):
        L.b200q_mul_mat_id_workspace.restype = c_size_t
        L.b200q_mul_mat_id_workspace.argtypes = [i32, i64, i64, i32, i32, i32, i32, i32]
        L.b200q_mul_mat_id_gemm.argtypes = [i32, vp, vp, i32, vp, vp, vp, i64, i64, i32, i32, i32, i32, c_float, vp, c_size_t, vp]
        L.b200q_mul_mat_id.argtypes = [i32, vp, vp, i32, vp, vp, vp, i64, i64, i32, i32, i32, i32, c_float, vp, c_size_t, vp]
    if hasattr(L, "b200q_decode_prefetch_next"):
        L.b200q_decode_prefetch_next.argtypes = [i32, i32, vp, vp, vp, i64]
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise B200QError(f"{what}: rc={rc}: {lib().b200q_last_error().decode(errors='replace')}")
