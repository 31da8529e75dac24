"""GPU tests of the grouped MoE prefill GEMM (b200q_mul_mat_id_gemm / b200q_mul_mat_id): GGML_OP_MUL_MAT_ID and GGML_OP_MOE_FUSED_UP_GATE
over expert-sorted tokens on tcgen05.

Tolerances:
  * versus the dense GEMM entry point (b200q_mul_mat_gemm) on the same expert with the columns routed to it: NMSE <= 1e-9.  Same bf16
    operands, same MMA order; only the dense path's split-K (f32 atomics) may reorder the sums.
  * versus the exact f64 product of the oracle: NMSE <= 2e-5 (the bar of test_gemm_vs_oracle: bf16 operands, f32 accumulation).
  * MOE_FUSED_UP_GATE versus act(gate) * up on the exact products: NMSE <= 2e-4, 1e-3 with a limit (the bars of test_fused_up_gate_gemm).
"""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import make_wire
from oracle.oracle import GGML_TYPE, nmse

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUPED_TYPES = ["IQ4_NL", "Q4_0", "Q4_1", "Q5_0", "Q5_1", "Q4_K", "Q5_K", "IQ4_K", "IQ5_K"]


@pytest.fixture(scope="module")
def be():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from ik_llama_cpp_b200 import backend
    return backend


def glu_ref(unary, g, u, limit=0.0):
    """act(gate) * up with the reference's order of operations: the clamp follows silu and exists for silu only; swiglu_oai: alpha 1.702, limit 7."""
    g = np.asarray(g, np.float64); u = np.asarray(u, np.float64)
    if unary == "silu":
        a = g / (1 + np.exp(-g))
        if limit > 1e-6:
            a = np.minimum(a, limit); u = np.clip(u, -limit, limit)
        return a * u
    if unary == "gelu":
        return 0.5 * g * (1 + np.tanh(0.79788456080286535588 * g * (1 + 0.044715 * g * g))) * u
    if unary == "relu":
        return np.maximum(g, 0) * u
    if unary == "swiglu_oai":
        g = np.minimum(g, 7.0); u = np.clip(u, -7.0, 7.0)
        return g / (1 + np.exp(-1.702 * g)) * (1 + u)
    raise ValueError(unary)


def experts(be, name, n_expert, m, k, seed):
    t = GGML_TYPE[name]
    wires = [make_wire(name, m, k, seed=seed + e, quantised=True) for e in range(n_expert)]
    return be.set_expert_tensor(t, np.concatenate(wires), n_expert, m, k), wires


def expert_view(be, W, e):
    pb = be.plane_bytes(W.ggml_type, W.m, W.k)
    return be.QuantTensor(W.ggml_type, W.m, W.k, W.planes[e * pb:(e + 1) * pb])


def dense_gemm(be, w, cols):
    """b200q_mul_mat_gemm at any n (the tcgen05 GEMM, also below the mat-vec threshold of the dispatcher)."""
    import ik_llama_cpp_b200 as pkg
    n = cols.shape[0]
    x = cols.contiguous()
    dst = torch.empty((n, w.m), dtype=torch.float32, device="cuda")
    ws = torch.empty(n * w.k * 2 + w.m * w.k * 2 + 1024, dtype=torch.uint8, device="cuda")
    pkg._lib.check(pkg.lib().b200q_mul_mat_gemm(w.ggml_type, w.ptr, x.data_ptr(), dst.data_ptr(), w.m, w.k, n, ws.data_ptr(), ws.numel(),
                                                torch.cuda.current_stream().cuda_stream), "b200q_mul_mat_gemm")
    return dst


def check_against_dense(be, oracle, W, wires, x, ids, y, exact_bar=2e-5):
    """Every slot of y against the dense GEMM of its (clamped) expert on the same columns, and against the exact product."""
    n_tokens, nb1, _ = x.shape
    idc = np.clip(ids.cpu().numpy(), 0, W.n_expert - 1)
    xn = x.cpu().numpy(); yn = y.cpu().numpy()
    n_used = idc.shape[1]
    for e in range(W.n_expert):
        sl = [(t, s) for t in range(n_tokens) for s in range(n_used) if idc[t, s] == e]
        if not sl:
            continue
        cols = torch.stack([x[t, s % nb1] for t, s in sl])
        ref = dense_gemm(be, expert_view(be, W, e), cols).cpu().numpy()
        got = np.stack([yn[t, s] for t, s in sl])
        assert nmse(got, ref) <= 1e-9, (e, nmse(got, ref))
        ex = oracle.mul_mat_exact(W.ggml_type, wires[e], np.stack([xn[t, s % nb1] for t, s in sl]), W.m)
        assert nmse(got, ex) <= exact_bar, (e, nmse(got, ex))


def rand_ids(rng, n_tokens, n_expert, n_used):
    return np.stack([rng.permutation(n_expert)[:n_used] for _ in range(n_tokens)]).astype(np.int32)


@pytest.mark.parametrize("name", GROUPED_TYPES)
@pytest.mark.parametrize("nb1", [1, 3])
def test_grouped_matches_dense_gemm(be, oracle, name, nb1):
    n_expert, n_used, m, k, n_tokens = 5, 3, 200, 512, 70           # ragged M, counts not multiples of the tile
    W, wires = experts(be, name, n_expert, m, k, seed=1000)
    rng = np.random.default_rng(5 + nb1)
    x = torch.from_numpy(rng.standard_normal((n_tokens, nb1, k)).astype(np.float32)).cuda()
    ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
    y = be.mul_mat_id_gemm(W, x, ids)
    assert y.shape == (n_tokens, n_used, m)
    check_against_dense(be, oracle, W, wires, x, ids, y)


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K"])
@pytest.mark.parametrize("case", ["empty_experts", "one_expert_many_tiles", "same_expert_twice", "one_token", "out_of_range_ids"])
def test_routing_edge_cases(be, oracle, name, case):
    m, k = 136, 512
    rng = np.random.default_rng(11)
    if case == "empty_experts":                       # only experts 1 and 6 of 8 receive rows
        n_expert, n_used, n_tokens, nb1 = 8, 2, 40, 2
        ids = np.tile(np.array([1, 6], np.int32), (n_tokens, 1)); ids[::3] = [6, 1]
    elif case == "one_expert_many_tiles":             # expert 0 gets 300 rows (> 2 * 128, not a multiple), 16 experts in all
        n_expert, n_used, n_tokens, nb1 = 16, 2, 300, 1
        ids = np.stack([[0, 1 + rng.integers(0, n_expert - 1)] for _ in range(n_tokens)]).astype(np.int32)
    elif case == "same_expert_twice":                 # a token that selects one expert in two slots
        n_expert, n_used, n_tokens, nb1 = 4, 2, 33, 2
        ids = rand_ids(rng, n_tokens, n_expert, n_used); ids[::2, 1] = ids[::2, 0]
    elif case == "one_token":
        n_expert, n_used, n_tokens, nb1 = 6, 3, 1, 1
        ids = rand_ids(rng, n_tokens, n_expert, n_used)
    else:                                             # corrupt ids are clamped into [0, n_expert), like the mat-vec kernel
        n_expert, n_used, n_tokens, nb1 = 5, 2, 24, 1
        ids = rng.integers(-3, n_expert + 3, (n_tokens, n_used)).astype(np.int32)
    W, wires = experts(be, name, n_expert, m, k, seed=2000)
    x = torch.from_numpy(rng.standard_normal((n_tokens, nb1, k)).astype(np.float32)).cuda()
    idg = torch.from_numpy(ids).cuda()
    y = be.mul_mat_id_gemm(W, x, idg)
    check_against_dense(be, oracle, W, wires, x, idg, y)
    if case == "out_of_range_ids":                    # both paths resolve a corrupt id to the same expert
        yv = be.mul_mat_id(W, x, idg)
        assert nmse(y.cpu().numpy(), yv.cpu().numpy()) <= 5e-4


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K"])
@pytest.mark.parametrize("unary,limit", [("silu", 0.0), ("gelu", 0.0), ("relu", 0.0), ("swiglu_oai", 0.0), ("silu", 1.5)])
def test_moe_fused_up_gate(be, oracle, name, unary, limit):
    n_expert, n_used, m, k, n_tokens = 6, 2, 260, 512, 50
    t = GGML_TYPE[name]
    U, uw = experts(be, name, n_expert, m, k, seed=3000)
    G, gw = experts(be, name, n_expert, m, k, seed=3100)
    rng = np.random.default_rng(21)
    xn = (rng.standard_normal((n_tokens, 1, k)) * 2).astype(np.float32)
    ids = rand_ids(rng, n_tokens, n_expert, n_used)
    y = be.mul_mat_id_gemm(U, torch.from_numpy(xn).cuda(), torch.from_numpy(ids).cuda(), gate=G, unary=unary, limit=limit).cpu().numpy()
    ref = np.empty_like(y, dtype=np.float64)
    for e in range(n_expert):
        sl = [(tk, s) for tk in range(n_tokens) for s in range(n_used) if ids[tk, s] == e]
        if not sl:
            continue
        cols = np.stack([xn[tk, 0] for tk, s in sl])
        u, g = oracle.mul_mat_exact(t, uw[e], cols, m).astype(np.float64), oracle.mul_mat_exact(t, gw[e], cols, m).astype(np.float64)
        r = glu_ref(unary, g, u, limit)
        for i, (tk, s) in enumerate(sl):
            ref[tk, s] = r[i]
    assert nmse(y, ref) <= (2e-4 if limit == 0 else 1e-3), nmse(y, ref)


def test_deterministic(be):
    n_expert, n_used, m, k, n_tokens = 8, 2, 384, 1024, 200
    W, _ = experts(be, "IQ4_NL", n_expert, m, k, seed=4000)
    rng = np.random.default_rng(31)
    x = torch.from_numpy(rng.standard_normal((n_tokens, 1, k)).astype(np.float32)).cuda()
    ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
    a = be.mul_mat_id_gemm(W, x, ids)
    b = be.mul_mat_id_gemm(W, x, ids)
    assert torch.equal(a, b)


def test_cuda_graph_capture_with_new_ids(be):
    """Routing, gather and GEMM never touch the host: a captured call replays correctly with ids written after capture."""
    n_expert, n_used, m, k, n_tokens = 8, 2, 256, 512, 96
    W, _ = experts(be, "Q4_K", n_expert, m, k, seed=5000)
    G, _ = experts(be, "Q4_K", n_expert, m, k, seed=5100)
    rng = np.random.default_rng(41)
    x = torch.from_numpy(rng.standard_normal((n_tokens, 1, k)).astype(np.float32)).cuda()
    ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
    out = torch.empty((n_tokens, n_used, m), dtype=torch.float32, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                         # warm-up outside the capture: workspace, kernel attributes
        be.mul_mat_id_gemm(W, x, ids, gate=G, out=out)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        be.mul_mat_id_gemm(W, x, ids, gate=G, out=out)
    for seed in (1, 2):
        new = rand_ids(np.random.default_rng(seed), n_tokens, n_expert, n_used)
        new[: n_tokens // 2, 0] = 3                    # a different routing (expert 3 crowded)
        ids.copy_(torch.from_numpy(new))
        graph.replay()
        torch.cuda.synchronize()
        ref = be.mul_mat_id_gemm(W, x, ids, gate=G)
        assert torch.equal(out, ref), seed


def test_dispatcher(be):
    n_expert, n_used, m, k = 8, 2, 256, 1024
    W, _ = experts(be, "IQ4_NL", n_expert, m, k, seed=6000)
    rng = np.random.default_rng(51)
    for n_tokens in (1, 2):                            # decode-sized: exactly the mat-vec kernel
        x = torch.from_numpy(rng.standard_normal((n_tokens, 1, k)).astype(np.float32)).cuda()
        ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
        assert torch.equal(be.mul_mat_id(W, x, ids, dispatch=True), be.mul_mat_id(W, x, ids))
    n_tokens = 512                                     # prefill-sized: exactly the grouped GEMM
    x = torch.from_numpy(rng.standard_normal((n_tokens, 1, k)).astype(np.float32)).cuda()
    ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
    assert torch.equal(be.mul_mat_id(W, x, ids, dispatch=True), be.mul_mat_id_gemm(W, x, ids))


@pytest.mark.parametrize("name", ["Q6_K", "IQ2_XXS"])
def test_dispatcher_keeps_mat_vec_for_uncovered_types(be, name):
    n_expert, n_used, m, k, n_tokens = 4, 2, 128, 1024, 512
    W, _ = experts(be, name, n_expert, m, k, seed=7000)
    rng = np.random.default_rng(61)
    x = torch.from_numpy(rng.standard_normal((n_tokens, 1, k)).astype(np.float32)).cuda()
    ids = torch.from_numpy(rand_ids(rng, n_tokens, n_expert, n_used)).cuda()
    assert torch.equal(be.mul_mat_id(W, x, ids, dispatch=True), be.mul_mat_id(W, x, ids))
    import ik_llama_cpp_b200 as pkg
    with pytest.raises(pkg.B200QError):
        be.mul_mat_id_gemm(W, x, ids)


def test_backend_ops_moe_prefill_through_ggml_backend_api():
    """MUL_MAT_ID / MOE_FUSED_UP_GATE at 64 to 512 tokens through the plug (b200q_mul_mat_id), against the reference CPU backend."""
    exe = os.path.join(ROOT, "tests", "backend_ops", "test_moe_prefill_backend")
    if not os.path.exists(exe):
        pytest.skip("harness not built (needs the reference headers at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    print(r.stdout[-6000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "PASSED: 0 failures" in r.stdout
