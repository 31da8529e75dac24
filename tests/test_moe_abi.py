"""CPU tests of the MoE prefill entry points of the C ABI: declared and exported, workspace arithmetic, argument checks, no CPU fallback."""
import ctypes

import numpy as np
import pytest

import ik_llama_cpp_b200 as pkg
from oracle.oracle import GGML_TYPE

GROUPED_TYPES = ["IQ4_NL", "Q4_0", "Q4_1", "Q5_0", "Q5_1", "Q4_K", "Q5_K", "IQ4_K", "IQ5_K"]
NEW = ["b200q_mul_mat_id_workspace", "b200q_mul_mat_id_gemm", "b200q_mul_mat_id"]


def test_new_symbols_declared_and_exported():
    L = pkg.lib()
    syms = pkg.header_symbols()
    for s in NEW:
        assert s in syms and hasattr(L, s), s
    assert L.b200q_abi_version() == 1


@pytest.mark.parametrize("name", GROUPED_TYPES)
@pytest.mark.parametrize("m,k,n_expert,n_used,nb1", [(768, 2048, 128, 8, 1), (2048, 768, 128, 8, 8), (14336, 4096, 8, 2, 1), (4096, 14336, 8, 2, 2), (200, 512, 5, 3, 3)])
@pytest.mark.parametrize("up_gate", [0, 1])
def test_workspace_positive_and_monotone(name, m, k, n_expert, n_used, nb1, up_gate):
    L = pkg.lib()
    t = GGML_TYPE[name]
    prev = 0
    for n in list(range(1, 70)) + [127, 128, 129, 255, 256, 257, 511, 512, 513, 1024, 2048, 4096]:
        ws = L.b200q_mul_mat_id_workspace(t, m, k, n_expert, n_used, nb1, n, up_gate)
        assert ws > 0 and ws >= prev, (n, ws, prev)
        assert ws >= n * n_used * k * 2 + (n * n_used * m * 4 if up_gate else 0)      # bf16 gather (+ f32 up scratch)
        prev = ws


def test_workspace_zero_where_not_covered():
    L = pkg.lib()
    for name in ("Q6_K", "IQ2_XXS", "Q8_0", "MXFP4"):
        assert L.b200q_mul_mat_id_workspace(GGML_TYPE[name], 256, 1024, 8, 2, 1, 512, 0) == 0, name
    t = GGML_TYPE["IQ4_NL"]
    assert L.b200q_mul_mat_id_workspace(t, 2048, 1408, 64, 6, 6, 512, 0) == 0        # K % 256 != 0 (DeepSeek-Lite down)
    assert L.b200q_mul_mat_id_workspace(t, 256, 1024, 1024, 2, 1, 512, 0) == 0        # more experts than the routing kernel holds
    assert L.b200q_mul_mat_id_workspace(t, 256, 1024, 8, 3, 2, 512, 0) == 0           # n_used % nb1 != 0


def _aligned(nbytes, align=256):
    buf = np.zeros(nbytes + align, np.uint8)
    off = (-buf.ctypes.data) % align
    return buf, buf.ctypes.data + off


def test_bad_arguments_are_errors():
    L = pkg.lib()
    t = GGML_TYPE["IQ4_NL"]
    for fn in (L.b200q_mul_mat_id_gemm, L.b200q_mul_mat_id):
        rc = fn(t, None, None, 8, None, None, None, 256, 1024, 2, 1, 512, 1, 0.0, None, 0, None)
        assert rc == -4, (fn, rc)
    w, wp = _aligned(1 << 16); x, xp = _aligned(1 << 16); ids = np.zeros(8, np.int32); y, yp = _aligned(1 << 16)
    ws, wsp = _aligned(1 << 20)
    rc = L.b200q_mul_mat_id_gemm(t, wp, None, 8, ids.ctypes.data, xp, yp, 256, 1024, 3, 2, 4, 1, 0.0, wsp, 1 << 20, None)
    assert rc == -4 and b"slot" in L.b200q_last_error()                                  # n_used % nb1 != 0
    rc = L.b200q_mul_mat_id_gemm(t, wp, None, 8, ids.ctypes.data, xp, yp, 256, 1024, 2, 1, 4, 1, 0.0, wsp, 16, None)
    assert rc == -4 and b"workspace" in L.b200q_last_error()
    rc = L.b200q_mul_mat_id_gemm(GGML_TYPE["Q6_K"], wp, None, 8, ids.ctypes.data, xp, yp, 256, 1024, 2, 1, 4, 1, 0.0, wsp, 1 << 20, None)
    assert rc == -1
    rc = L.b200q_mul_mat_id_gemm(t, wp, None, 8, ids.ctypes.data, xp, yp, 256, 1000, 2, 1, 4, 1, 0.0, wsp, 1 << 20, None)
    assert rc == -2


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = pkg.lib()
    t = GGML_TYPE["IQ4_NL"]
    w, wp = _aligned(1 << 16); x, xp = _aligned(1 << 16); y, yp = _aligned(1 << 16); ids = np.zeros(8, np.int32)
    need = L.b200q_mul_mat_id_workspace(t, 64, 256, 4, 2, 1, 4, 0)
    ws, wsp = _aligned(need)
    for fn in (L.b200q_mul_mat_id_gemm, L.b200q_mul_mat_id):
        rc = fn(t, wp, None, 4, ids.ctypes.data, xp, yp, 64, 256, 2, 1, 4, 1, 0.0, wsp, need, None)
        assert rc == -3, "compute entry points must fail with B200Q_E_CUDA when there is no device"
