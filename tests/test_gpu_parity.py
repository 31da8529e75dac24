"""GPU parity tests (run on the B200 with -m gpu).  Everything goes through the C ABI of libb200q.so
(ik_llama_cpp_b200.backend is a thin ctypes mirror); the oracle is only the checker.

Tolerances (written here, justified in DESIGN.md §Parity):
  * wire<->planes: bit-exact.
  * decode mat-vec (n <= 8): the kernel evaluates the same quantity as the reference's MMVQ kernels —
    dequant(W) . dequant_q8_1(x) with integer partial sums.  Versus the oracle restatement of the product's
    quantiser (variant="b200": one division per block, round-half-even) only the f32 summation order differs:
    max |diff| <= 2e-5 * rms(y); versus the reference's quantiser (roundf(x/d), variant="reference") a 1-LSB
    difference at rounding ties is possible: max |diff| <= 1e-3 * rms(y) (north_star tolerance; measured ~1e-4 worst).  Versus the exact f64 result the reference's own test bar applies:
    NMSE <= 5e-4 (tests/test-backend-ops.cpp:979-981); we measure ~2e-5.
  * prefill GEMM (n > 8): bf16 x bf16 -> f32 on tcgen05: NMSE vs exact <= 5e-4 (bar), and we also require
    NMSE <= 2e-5, i.e. at least as accurate as the reference's own int8 (q8_1) path (~2e-5).
"""
import numpy as np
import pytest
import torch

from conftest import ALL_TYPES, load_golden, make_wire
from oracle.oracle import GGML_TYPE, nmse

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from ik_llama_cpp_b200 import backend
    return backend


def rms(a):
    return float(np.sqrt((a.astype(np.float64) ** 2).mean()))


def glu_ref(unary, g, u, limit=0.0):
    """act(gate) * up with the reference's order of operations (fused_mul_mat_vec_q, mmvq-templates.cuh:240-275; fused_mul_silu_f32 with
    limit, unary.cu:63-72; CPU ggml.c:16939-16945): the clamp FOLLOWS silu and exists for silu only; swiglu_oai: alpha 1.702, limit 7."""
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


@pytest.mark.parametrize("name", ALL_TYPES)
def test_set_get_tensor_roundtrip(be, name):
    g = load_golden(name)
    t, m, k = int(g["ggml_type"]), int(g["m"]), int(g["k"])
    w = be.set_tensor(t, g["wire"], m, k)
    assert np.array_equal(be.get_tensor(w), g["wire"])
    # device-side repack entry point gives the same planes
    w2 = be.set_tensor(t, torch.from_numpy(g["wire"]).cuda(), m, k)
    assert torch.equal(w.planes, w2.planes)


@pytest.mark.parametrize("name", ALL_TYPES)
def test_golden_mat_vec(be, oracle, name):
    g = load_golden(name)
    t, m, k = int(g["ggml_type"]), int(g["m"]), int(g["k"])
    w = be.set_tensor(t, g["wire"], m, k)
    x = torch.from_numpy(g["x"]).cuda()
    y = be.mul_mat(w, x).cpu().numpy()
    yq = oracle.mul_mat_q8_1(t, g["wire"], g["x"], m, variant="b200")
    assert np.abs(y - yq).max() <= 2e-5 * rms(yq)
    yr = oracle.mul_mat_q8_1(t, g["wire"], g["x"], m, variant="reference")
    # north-star tolerance vs the reference's own arithmetic.  Our activation quantiser differs from roundf(x/d) only at rounding
    # ties (1 LSB of one int8, DESIGN.md §3); when this x contains such a tie (the two oracle quantisers disagree: Q2_K's vector does)
    # the affected outputs move by ~w*d8, which can exceed 1e-3 of the rms -> bound by the tie's own size instead
    q_ref, q_b2 = oracle.quantize_q8_1(g["x"])[0], oracle.quantize_q8_1_b200(g["x"])[0]
    tie = not np.array_equal(q_ref, q_b2)
    assert np.abs(y - yr).max() <= (1e-3 if not tie else 5e-3) * rms(yr)
    assert nmse(y, oracle.mul_mat_exact(t, g["wire"], g["x"], m)) <= 5e-4
    # dequantise-to-bf16 kernel == bf16(reference to_float)
    d = be.dequantize_bf16(w).float().cpu().numpy()
    ref = torch.from_numpy(g["dequant_ref"]).to(torch.bfloat16).float().numpy()
    np.testing.assert_allclose(d, ref, rtol=8e-3, atol=1e-9)      # IQ4_KS/IQ2_BN: 1-ulp f32 association before bf16 rounding
    if name not in ("IQ4_KS", "IQ5_KS", "IQ2_BN", "IQ6_K"):      # (IQ6_K: the reference build contracts its float cubic into FMAs)
        assert np.array_equal(d, ref)


@pytest.mark.parametrize("name", ALL_TYPES)
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
def test_mat_vec_vs_oracle(be, oracle, name, n):
    t = GGML_TYPE[name]
    m, k = (260 if name.endswith("_R4") else 257), 2048      # ragged M (not a multiple of the CTA tile; the _R4 repacks come in groups of 4 rows)
    wire = make_wire(name, m, k, seed=11 + t + n, quantised=True)
    rng = np.random.default_rng(5 + n)
    x = rng.standard_normal((n, k)).astype(np.float32)
    x[0, 64:96] = 0.0                      # amax == 0 block
    w = be.set_tensor(t, wire, m, k)
    y = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
    yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200")
    assert np.abs(y - yq).max() <= 2e-5 * rms(yq), f"{name} n={n}"
    yr = oracle.mul_mat_q8_1(t, wire, x, m, variant="reference")
    assert np.abs(y - yr).max() <= 1e-3 * rms(yr), f"{name} n={n}"
    assert nmse(y, oracle.mul_mat_exact(t, wire, x, m)) <= 5e-4


@pytest.mark.parametrize("name,k", [("IQ2_BN", 3200), ("IQ2_BN", 8640), ("Q4_0", 160), ("IQ4_NL", 96), ("Q8_0", 224), ("Q5_1", 1056)])
@pytest.mark.parametrize("n", [1, 3, 32])
def test_k_not_multiple_of_256(be, oracle, name, k, n):
    """bitnet-b1.58 rows (K = 3200 / 8640 = 50 / 135 IQ2_BN blocks, SURVEY Appendix A config 4) and short 32-weight-block rows:
    the TMA ring needs K % 256 == 0, these shapes take the LDG mat-vec / the zero-filled last GEMM k-block."""
    t = GGML_TYPE[name]
    m = 130
    wire = make_wire(name, m, k, seed=300 + n)
    x = np.random.default_rng(50 + n).standard_normal((n, k)).astype(np.float32)
    w = be.set_tensor(t, wire, m, k)
    assert np.array_equal(be.get_tensor(w), np.frombuffer(wire, np.uint8))
    y = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
    exact = oracle.mul_mat_exact(t, wire, x, m)
    if n <= 8:
        yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200")
        assert np.abs(y - yq).max() <= 2e-5 * rms(yq)
        assert nmse(y, exact) <= 5e-4
    else:
        assert nmse(y, exact) <= (3e-4 if name == "IQ2_BN" else 2e-5)        # IQ2_BN: int8 tensor pipe, per-token 8-bit activations


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K", "IQ5_K"])
def test_mat_vec_llama_shapes(be, oracle, name):
    """BASELINE config 1: MUL_MAT 4096x4096 n=1 (and the 14336-wide FFN shape) at full size."""
    t = GGML_TYPE[name]
    for (m, k) in ((4096, 4096), (512, 14336)):
        wire = make_wire(name, m, k, seed=3)
        x = np.random.default_rng(1).standard_normal((1, k)).astype(np.float32)
        w = be.set_tensor(t, wire, m, k)
        y = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
        yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200")
        assert np.abs(y - yq).max() <= 2e-5 * rms(yq)


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K"])
def test_mat_vec_full_size_ffn_and_head_shapes(be, oracle, name):
    """Full-size shapes (FFN up/gate 14336 x 4096, a quarter of the output head, ffn_down with its 14336-long rows): every CTA works through many
    units per warp (in-CTA claiming, ring wrap-around, long-row segments); three launches in a row, all equal to the oracle."""
    t = GGML_TYPE[name]
    x_rng = np.random.default_rng(21)
    for (m, k, glu) in ((14336, 4096, True), (32064, 4096, False), (4096, 14336, False)):
        wire = make_wire(name, m, k, seed=5)
        w = be.set_tensor(t, wire, m, k)
        if glu:
            wire2 = make_wire(name, m, k, seed=6); w2 = be.set_tensor(t, wire2, m, k)
        for it in range(3):
            x = x_rng.standard_normal((1, k)).astype(np.float32)
            xg = torch.from_numpy(x).cuda()
            if glu:
                y = be.fused_up_gate(w, w2, xg, unary="silu").cpu().numpy()
                u, g = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200").astype(np.float64), oracle.mul_mat_q8_1(t, wire2, x, m, variant="b200").astype(np.float64)
                ref = glu_ref("silu", g, u)
                assert np.abs(y - ref).max() <= 5e-5 * rms(ref), (m, k, it)
            else:
                y = be.mul_mat(w, xg).cpu().numpy()
                yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200")
                assert np.abs(y - yq).max() <= 2e-5 * rms(yq), (m, k, it)


def test_multi_tensor_launch_qkv(be, oracle):
    t = GGML_TYPE["IQ4_NL"]
    k = 1024
    ms = [512, 128, 128]
    wires = [make_wire("IQ4_NL", m, k, seed=20 + i) for i, m in enumerate(ms)]
    ws = [be.set_tensor(t, wire, m, k) for wire, m in zip(wires, ms)]
    x = np.random.default_rng(2).standard_normal((2, k)).astype(np.float32)
    outs = be.mul_mat_multi(ws, torch.from_numpy(x).cuda())
    for wire, m, o in zip(wires, ms, outs):
        yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200")
        assert np.abs(o.cpu().numpy() - yq).max() <= 2e-5 * rms(yq)


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "IQ2_BN"])
@pytest.mark.parametrize("unary,limit", [("silu", 0.0), ("gelu", 0.0), ("relu", 0.0), ("silu", 1.5), ("gelu", 1.5), ("swiglu_oai", 0.0)])
@pytest.mark.parametrize("n", [1, 2, 5])
def test_fused_up_gate(be, oracle, name, unary, limit, n):
    """n = 1, 2: the TMA-ring kernel; n = 5: the LDG kernel.  limit: after the activation, silu only (gelu ignores it)."""
    t = GGML_TYPE[name]
    m, k = 384, 1024
    wu, wg = make_wire(name, m, k, seed=31), make_wire(name, m, k, seed=32)
    x = np.random.default_rng(3).standard_normal((n, k)).astype(np.float32) * 4
    up, gate = be.set_tensor(t, wu, m, k), be.set_tensor(t, wg, m, k)
    y = be.fused_up_gate(up, gate, torch.from_numpy(x).cuda(), unary=unary, limit=limit).cpu().numpy()
    u, g = oracle.mul_mat_q8_1(t, wu, x, m, variant="b200").astype(np.float64), oracle.mul_mat_q8_1(t, wg, x, m, variant="b200").astype(np.float64)
    ref = glu_ref(unary, g, u, limit)
    assert np.abs(y - ref).max() <= 5e-5 * max(rms(ref), 1e-30)


def test_fused_up_gate_limit_matches_reference_cpu_op(be, oracle):
    """The clamp semantics pinned on the reference itself: GGML_OP_FUSED_UP_GATE with op_params limit through the unmodified CPU backend,
    recorded in reference_xcheck.npz (tests/golden/gen_golden.py --xcheck)."""
    g = load_golden("reference_xcheck")
    t = GGML_TYPE["Q4_0"]
    m, k = 256, 512
    wu, wg = make_wire("Q4_0", m, k, seed=61), make_wire("Q4_0", m, k, seed=62)
    x = np.random.default_rng(9).standard_normal((1, k)).astype(np.float32) * 6
    up, gate = be.set_tensor(t, wu, m, k), be.set_tensor(t, wg, m, k)
    for limit in (0.0, 1.5):
        y = be.fused_up_gate(up, gate, torch.from_numpy(x).cuda(), unary="silu", limit=limit).cpu().numpy()
        r = g[f"fused_up_gate.Q4_0.silu.limit{limit}"]
        assert nmse(y, r) <= 5e-4, (limit, nmse(y, r))


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K"])
def test_q8_handoff_up_gate_to_down(be, oracle, name):
    """FUSED_UP_GATE (n = 1) emits its result quantised to q8_1 in its epilogue; the following MUL_MAT consumes that image.
    Bit-identical to the path that re-quantises per CTA (same arithmetic on the same f32 values), and equal to the oracle."""
    t = GGML_TYPE[name]
    k, ff, m2 = (1024, 1536, 512) if name != "Q6_K" else (2048, 2048, 256)     # Q6_K's 2-byte d plane is bulk-copyable only for K % 2048 == 0
    wu, wg, wd = make_wire(name, ff, k, seed=71), make_wire(name, ff, k, seed=72), make_wire(name, m2, ff, seed=73)
    up, gate, down = be.set_tensor(t, wu, ff, k), be.set_tensor(t, wg, ff, k), be.set_tensor(t, wd, m2, ff)
    x = torch.from_numpy(np.random.default_rng(4).standard_normal((1, k)).astype(np.float32) * 3).cuda()
    q8 = be.Q8Scratch(ff)
    for it in range(3):                                     # the arrival counters must re-arm themselves
        a = be.fused_up_gate(up, gate, x, unary="silu", q8_out=q8)
        assert q8.valid, "eligible shape: the hand-off must be taken"
        y = be.mul_mat(down, a, q8_in=q8)
        y_plain = be.mul_mat(down, a)
        assert torch.equal(y, y_plain), f"iteration {it}"
        x = x * 0.5 + 0.25
    an = a.cpu().numpy()
    yq = oracle.mul_mat_q8_1(t, wd, an, m2, variant="b200")
    assert np.abs(y.cpu().numpy() - yq).max() <= 2e-5 * rms(yq)
    # the image itself: q / d / sums of the oracle's quantiser
    q_ref, d_ref = oracle.quantize_q8_1_b200(an)[:2]
    img = q8.buf.cpu().numpy()
    assert np.array_equal(img[:ff].view(np.int8), np.asarray(q_ref, np.int8).reshape(-1))
    assert np.array_equal(img[ff:ff + 4 * (ff // 32)].view(np.float32), np.asarray(d_ref, np.float32).reshape(-1))
    assert not img[ff + 8 * (ff // 32): ff + 12 * (ff // 32)].any(), "arrival counters must be back at zero"


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K"])
@pytest.mark.parametrize("n", [1, 2, 5])
def test_mat_vec_bias(be, oracle, name, n):
    """bias operand of the mat-vec kernels (fused trailing ADD of ggml_cuda_mul_mat_q, ggml-cuda.cu:2590-2600)."""
    import ctypes
    import ik_llama_cpp_b200 as pkg
    t = GGML_TYPE[name]
    m, k = 322, 1024
    wire = make_wire(name, m, k, seed=81)
    w = be.set_tensor(t, wire, m, k)
    x = np.random.default_rng(12).standard_normal((n, k)).astype(np.float32)
    bias = np.random.default_rng(13).standard_normal(m).astype(np.float32)
    xg, bg = torch.from_numpy(x).cuda(), torch.from_numpy(bias).cuda()
    y = torch.empty((n, m), dtype=torch.float32, device="cuda")
    pkg._lib.check(pkg.lib().b200q_mul_mat_vec(t, w.ptr, xg.data_ptr(), y.data_ptr(), m, k, n, k, bg.data_ptr(), torch.cuda.current_stream().cuda_stream), "bias")
    yq = oracle.mul_mat_q8_1(t, wire, x, m, variant="b200") + bias[None, :]
    assert np.abs(y.cpu().numpy() - yq).max() <= 2e-5 * rms(yq)


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K", "IQ2_K", "IQ4_KS", "IQ2_XXS", "IQ3_S", "IQ4_K_R4", "IQ2_KT"])
@pytest.mark.parametrize("n_tokens,nb1", [(1, 1), (1, 3), (4, 1), (3, 3)])
@pytest.mark.parametrize("glu", [False, True])
def test_mul_mat_id(be, oracle, name, n_tokens, nb1, glu):
    """GGML_OP_MUL_MAT_ID / MOE_FUSED_UP_GATE for decode-sized batches: expert ids are resolved on the device, one launch.
    Oracle: the plain mat-vec oracle on the selected expert's wire bytes."""
    t = GGML_TYPE[name]
    n_expert, n_used, m, k = 6, 3, 260, 1024
    rs = len(make_wire(name, 4, k, seed=1)) // 4
    wires = [make_wire(name, m, k, seed=400 + e) for e in range(n_expert)]
    gwires = [make_wire(name, m, k, seed=500 + e) for e in range(n_expert)]
    assert all(len(w) == m * rs for w in wires)
    W = be.set_expert_tensor(t, np.concatenate(wires), n_expert, m, k)
    G = be.set_expert_tensor(t, np.concatenate(gwires), n_expert, m, k) if glu else None
    rng = np.random.default_rng(77 + n_tokens + nb1)
    x = rng.standard_normal((n_tokens, nb1, k)).astype(np.float32)
    ids = np.stack([rng.permutation(n_expert)[:n_used] for _ in range(n_tokens)]).astype(np.int32)
    y = be.mul_mat_id(W, torch.from_numpy(x).cuda(), torch.from_numpy(ids).cuda(), gate=G, unary="silu").cpu().numpy()
    assert y.shape == (n_tokens, n_used, m)
    for tk in range(n_tokens):
        for e in range(n_used):
            col = x[tk, e % nb1][None, :]
            ref = oracle.mul_mat_q8_1(t, wires[ids[tk, e]], col, m, variant="b200")[0].astype(np.float64)
            if glu:
                ref = glu_ref("silu", oracle.mul_mat_q8_1(t, gwires[ids[tk, e]], col, m, variant="b200")[0].astype(np.float64), ref)
            assert np.abs(y[tk, e] - ref).max() <= 5e-5 * max(rms(ref), 1e-30), (tk, e)


def test_mul_mat_id_token_chunks(be):
    """Batches beyond one launch's shared-memory capacity are walked in token chunks: 20 tokens, both column modes, in one launch and forced to
    3 tokens per launch.  The chunk size is read once per process, so the check (scripts/moe_chunk_check.py) runs in child processes."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for forced in (None, "3"):
        env = dict(os.environ)
        if forced:
            env["B200Q_MOE_CHUNK_TOKENS"] = forced
        r = subprocess.run([sys.executable, os.path.join(root, "scripts", "moe_chunk_check.py")], capture_output=True, text=True, env=env, cwd=root, timeout=300)
        assert "CHUNKS-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_add_rows(be):
    import ik_llama_cpp_b200 as pkg
    a, b = torch.randn(5, 322, device="cuda"), torch.randn(322, device="cuda")
    d = torch.empty_like(a)
    pkg._lib.check(pkg._lib.lib().b200q_add_rows(a.data_ptr(), b.data_ptr(), d.data_ptr(), 322, 5, 1, torch.cuda.current_stream().cuda_stream), "add")
    assert torch.equal(d, a + b)
    pkg._lib.check(pkg._lib.lib().b200q_add_rows(a.data_ptr(), a.data_ptr(), d.data_ptr(), 322, 5, 5, torch.cuda.current_stream().cuda_stream), "add")
    assert torch.equal(d, a + a)


@pytest.mark.parametrize("name", ALL_TYPES)
@pytest.mark.parametrize("n", [16, 33, 512])
def test_gemm_vs_oracle(be, oracle, name, n):
    t = GGML_TYPE[name]
    m, k = (384, 1024) if n == 512 else (200, 512)        # ragged M and N
    wire = make_wire(name, m, k, seed=41 + t, quantised=True)
    x = np.random.default_rng(6 + n).standard_normal((n, k)).astype(np.float32)
    w = be.set_tensor(t, wire, m, k)
    y = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
    exact = oracle.mul_mat_exact(t, wire, x, m)
    e = nmse(y, exact)
    assert e <= 5e-4, f"{name} n={n}: NMSE {e}"          # the reference's own bar
    if name == "IQ2_BN":                                  # int8 tensor pipe: activations rounded to 8 bits per token (test_bitnet_int8_gemm_is_exact_integer_arithmetic)
        assert e <= 3e-4, f"{name} n={n}: NMSE {e}"
    else:
        assert e <= 2e-5, f"{name} n={n}: NMSE {e}"      # ours: bf16 inputs, f32 accumulate


@pytest.mark.parametrize("m,k,n", [(384, 1024, 512), (130, 3200, 40), (256, 8640, 70), (128, 64, 16)])
def test_bitnet_int8_gemm_is_exact_integer_arithmetic(be, oracle, m, k, n):
    """IQ2_BN prefill = tcgen05.mma kind::i8 on per-token int8 activations: dst = rs[m] * ts[n] * (sum_k q*xq - sum_k xq) with exact integer sums.
    Emulated in numpy (same quantiser: ts = amax/127, xq = rint(x / ts)): only the two f32 multiplies of the epilogue may round.  K = 3200 / 8640 are the
    bitnet-b1.58 row lengths (not multiples of the 128-wide k-block: zero-filled TMA tails), K = 64 a single wire block."""
    import ik_llama_cpp_b200 as pkg
    t = GGML_TYPE["IQ2_BN"]
    wire = make_wire("IQ2_BN", m, k, seed=400 + n)
    x = (np.random.default_rng(60 + n).standard_normal((n, k)) * 1.7).astype(np.float32)
    x[0, :] = 0.0                                           # an all-zero token (amax == 0)
    w = be.set_tensor(t, wire, m, k)
    y = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
    wd = oracle.dequantize(t, wire, m, k).astype(np.float64)
    amax = np.abs(x).max(1, keepdims=True)
    ts = (amax / np.float32(127)).astype(np.float32)
    inv = np.where(ts > 0, np.float32(1) / np.where(ts > 0, ts, 1), 0).astype(np.float32)
    xq = np.clip(np.rint(x * inv), -127, 127)
    emul = (xq.astype(np.float64) * ts.astype(np.float64)) @ wd.T
    assert np.abs(y - emul).max() <= 4e-7 * np.abs(emul).max() + 1e-30, float(np.abs(y - emul).max() / np.abs(emul).max())
    assert nmse(y, oracle.mul_mat_exact(t, wire, x, m)) <= 3e-4
    # the bf16 tensor-pipe path (B200Q_BN_INT8=0 equivalent: fused_gemm off) still agrees with exact math to bf16 accuracy
    pkg.lib().b200q_set_option(b"fused_gemm", 0)
    try:
        y0 = be.mul_mat(w, torch.from_numpy(x).cuda()).cpu().numpy()
    finally:
        pkg.lib().b200q_set_option(b"fused_gemm", 1)
    assert nmse(y0, oracle.mul_mat_exact(t, wire, x, m)) <= 2e-5


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K"])
def test_gemm_shared_activation_and_unfused_path(be, oracle, name):
    """convert_activations once + _bf16 entry point; fused (in-kernel dequant) and unfused (bf16 scratch) kernels agree."""
    import ik_llama_cpp_b200 as pkg
    t = GGML_TYPE[name]
    m, k, n = 256, 768, 40
    wire = make_wire(name, m, k, seed=91 + t)
    x = np.random.default_rng(17).standard_normal((n, k)).astype(np.float32)
    w = be.set_tensor(t, wire, m, k)
    xg = torch.from_numpy(x).cuda()
    xb = be.convert_activations(xg)
    assert torch.equal(xb, xg.to(torch.bfloat16))
    exact = oracle.mul_mat_exact(t, wire, x, m)
    y1 = be.mul_mat(w, xg, x_bf16=xb).cpu().numpy()
    pkg.lib().b200q_set_option(b"fused_gemm", 0)
    try:
        y0 = be.mul_mat(w, xg, x_bf16=xb).cpu().numpy()
    finally:
        pkg.lib().b200q_set_option(b"fused_gemm", 1)
    assert nmse(y1, exact) <= 2e-5 and nmse(y0, exact) <= 2e-5
    assert nmse(y1, y0) <= 1e-9          # same bf16 operands, same MMA order


@pytest.mark.parametrize("name", ["IQ4_NL", "Q4_K", "Q6_K"])
@pytest.mark.parametrize("n", [40, 512])
def test_gemm_multi_tensor_launch_qkv(be, oracle, name, n):
    """n > 8 look-ahead fusion: Q,K,V in ONE GEMM launch (row tiles of three tensors, ragged M) == three single launches."""
    t = GGML_TYPE[name]
    k = 1024
    ms = [512, 128, 200]
    wires = [make_wire(name, m, k, seed=120 + i) for i, m in enumerate(ms)]
    ws = [be.set_tensor(t, wire, m, k) for wire, m in zip(wires, ms)]
    x = np.random.default_rng(21).standard_normal((n, k)).astype(np.float32)
    xg = torch.from_numpy(x).cuda()
    xb = be.convert_activations(xg)
    outs_b = be.mul_mat_multi(ws, xg, x_bf16=xb)
    outs_f = be.mul_mat_multi(ws, xg)                        # f32 activations: conversion inside the call
    for w, wire, m, ob, of in zip(ws, wires, ms, outs_b, outs_f):
        single = be.mul_mat(w, xg, x_bf16=xb).cpu().numpy()
        assert nmse(ob.cpu().numpy(), single) <= 1e-9       # same operands; only the split-K summation order may differ
        assert nmse(of.cpu().numpy(), single) <= 1e-9
        cols = [0, n // 2, n - 1]
        assert nmse(ob.cpu().numpy()[cols], oracle.mul_mat_exact(t, wire, x[cols], m)) <= 2e-5


@pytest.mark.parametrize("name,m,k", [("IQ4_NL", 1000, 256), ("IQ4_NL", 384, 1024), ("Q4_K", 1000, 256), ("Q6_K", 384, 1024), ("IQ2_BN", 256, 512)])
@pytest.mark.parametrize("unary,limit", [("silu", 0.0), ("gelu", 0.0), ("relu", 0.0), ("silu", 1.5), ("swiglu_oai", 0.0)])
@pytest.mark.parametrize("fuse", [0, 1])
def test_fused_up_gate_gemm(be, oracle, name, m, k, unary, limit, fuse):
    """GGML_OP_FUSED_UP_GATE for n > 8.  fuse=1 with k=256 (split-K 1): unary-mul inside the gate GEMM's epilogue; everything else:
    gate GEMM + k_mul_unary.  Checked against act(gate.x)*(up.x) from the plain GEMM entry point and the oracle."""
    t = GGML_TYPE[name]
    n = 70
    wu, wg = make_wire(name, m, k, seed=131), make_wire(name, m, k, seed=132)
    up, gate = be.set_tensor(t, wu, m, k), be.set_tensor(t, wg, m, k)
    x = np.random.default_rng(23).standard_normal((n, k)).astype(np.float32) * 2
    xg = torch.from_numpy(x).cuda()
    xb = be.convert_activations(xg)
    ybf = torch.empty((n, m), dtype=torch.bfloat16, device="cuda")
    import ik_llama_cpp_b200 as pkg
    pkg.lib().b200q_set_option(b"fuse_epilogue", fuse)       # 1: unary-mul inside the gate GEMM's epilogue (opt-in), 0: k_mul_unary tail
    try:
        y = be.fused_up_gate(up, gate, xg, unary=unary, limit=limit, x_bf16=xb, out_bf16=ybf)
        y2 = be.fused_up_gate(up, gate, xg, unary=unary, limit=limit)           # f32 activations, no bf16 copy
    finally:
        pkg.lib().b200q_set_option(b"fuse_epilogue", 0)
    u, g = be.mul_mat(up, xg, x_bf16=xb).double(), be.mul_mat(gate, xg, x_bf16=xb).double()
    ref = torch.from_numpy(glu_ref(unary, g.cpu().numpy(), u.cpu().numpy(), limit)).cuda()
    scale = float(ref.pow(2).mean().sqrt())
    assert float((y.double() - ref).abs().max()) <= 2e-5 * scale
    if name == "IQ2_BN":        # f32 activations take the int8 tensor pipe for ternary weights (8-bit activations): compare at that accuracy
        assert float(((y2.double() - ref) ** 2).sum() / (ref ** 2).sum()) <= 1e-3
    else:
        assert float((y2.double() - ref).abs().max()) <= 2e-5 * scale
    assert torch.equal(ybf, y.to(torch.bfloat16))
    # and against exact math on a few tokens (bf16-operand noise only)
    cols = [0, 33, 69]
    ue, ge = oracle.mul_mat_exact(t, wu, x[cols], m).astype(np.float64), oracle.mul_mat_exact(t, wg, x[cols], m).astype(np.float64)
    assert nmse(y[cols].cpu().numpy(), glu_ref(unary, ge, ue, limit)) <= (2e-4 if limit == 0 else 1e-3)


def test_gemm_llama_shape_properties(be, oracle):
    """pp512 shape 4096x4096x512: GEMM path must agree with the mat-vec path column by column (two independent kernels)
    within their documented noise, and with the oracle on a sample of columns."""
    t = GGML_TYPE["IQ4_NL"]
    m = k = 4096
    n = 512
    wire = make_wire("IQ4_NL", m, k, seed=77)
    x = np.random.default_rng(8).standard_normal((n, k)).astype(np.float32)
    w = be.set_tensor(t, wire, m, k)
    xg = torch.from_numpy(x).cuda()
    y = be.mul_mat(w, xg)
    cols = [0, 1, 255, 256, 511]
    yv = torch.cat([be.mul_mat(w, xg[c:c + 1]) for c in cols]).cpu().numpy()
    yg = y[cols].cpu().numpy()
    assert nmse(yg, yv) <= 1e-4
    exact = oracle.mul_mat_exact(t, wire, x[cols], m)
    assert nmse(yg, exact) <= 2e-5
    assert torch.isfinite(y).all()


def test_host_buffer_entry_point(be, oracle):
    t = GGML_TYPE["Q4_K"]
    m, k = 320, 1024
    wire = make_wire("Q4_K", m, k, seed=51)
    w = be.set_tensor(t, wire, m, k)
    for n in (1, 24):
        x = np.random.default_rng(n).standard_normal((n, k)).astype(np.float32)
        y = be.mul_mat_host(w, x)
        assert nmse(y, oracle.mul_mat_exact(t, wire, x, m)) <= 5e-4


def test_extension_is_the_code_that_runs(be):
    """The .so must be in-tree and loaded; a silent fallback would leave it unloaded."""
    import ik_llama_cpp_b200 as pkg
    with open("/proc/self/maps") as f:
        assert pkg.LIB_PATH in f.read()
