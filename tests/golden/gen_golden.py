"""Generate tests/golden/*.npz FROM THE UNMODIFIED REFERENCE (oracle/_ref, built by oracle/Makefile.ref).

Run in the container that has /root/reference:   python tests/golden/gen_golden.py
For every supported wire type: seeded f32 weights -> ggml_quantize_chunk (reference) -> wire bytes;
reference to_float(wire) -> dequantised f32; reference CPU backend MUL_MAT (IQK path) -> y_ref_cpu.
The fixtures pin the oracle restatement (tests/test_oracle.py) and are replayed against the CUDA
kernels on the GPU box (tests/test_gpu_parity.py), where /root/reference does not exist.

python tests/golden/gen_golden.py --xcheck  writes reference_xcheck.npz instead: what the reference computes for the cross-check tests
(tests/test_oracle.py::test_oracle_vs_live_reference, tests/test_gpu_parity.py::test_fused_up_gate_limit_matches_reference_cpu_op),
so that they run without the reference library.
"""
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from conftest import make_wire  # noqa: E402
from oracle.oracle import GGML_TYPE, RefLib  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
TYPES = ["Q4_0", "Q4_1", "Q5_0", "Q5_1", "Q6_0", "Q8_0", "Q2_K", "Q3_K", "Q4_K", "Q5_K", "Q6_K", "IQ4_NL", "IQ4_XS", "IQ2_K", "IQ3_K", "IQ4_K", "IQ5_K", "IQ4_KS", "IQ5_KS", "IQ2_KS", "IQ3_KS", "MXFP4", "IQ2_BN"]
# types whose ORACLE is pinned already while the device kernel is still to come (DESIGN.md §7b): fixtures for tests/test_oracle.py only
ORACLE_ONLY = []
# types that are consumed verbatim on the device (wire layout, generic decode; b200q_wire.cuh): codebook / trellis / row-interleaved types
WIRE_TYPES = ["IQ2_XXS", "IQ2_XS", "IQ3_XXS", "IQ2_S", "IQ3_S", "IQ6_K", "IQ1_BN", "IQ4_KSS", "IQ1_S", "IQ1_M", "IQ2_KL", "IQ1_KT", "IQ2_KT", "IQ3_KT", "IQ4_KT",
              "IQ1_S_R4", "IQ1_M_R4", "IQ2_K_R4", "IQ3_K_R4", "IQ4_K_R4", "IQ5_K_R4", "IQ4_KS_R4", "IQ5_KS_R4"]
M, K, N = 16, 512, 3


# to_float is stored in full only for IQ6_K, whose reference build contracts a float cubic into FMAs, so the oracle matches it within a
# tolerance only (tests/test_oracle.py FMA_DEPENDENT).  Every other type must match bit for bit on this data: the SHA-256 of the f32
# bytes is enough for that and keeps the file small.  That includes IQ4_KS / IQ5_KS: _assert_dequant_equal allows them one ulp because
# the oracle evaluates dl*(v+4) where the reference evaluates dl*v + 4*dl, which can round differently for some scale values; for the
# scales in this data the two agree on every element, so the exact check holds here and is the stricter one.  Should a change of the
# oracle's arithmetic move them by that ulp, add them here and regenerate
DEQUANT_STORED = ("IQ6_K",)


def xcheck(R):
    out = {}
    for name in TYPES + WIRE_TYPES:
        t = GGML_TYPE[name]
        rng = np.random.default_rng(99 + t)
        m, k, n = 8, 1024, 2
        w = (rng.standard_normal((m, k)) * 0.05).astype(np.float32)
        if name in ("IQ2_BN", "IQ1_BN"):
            w = (rng.integers(-1, 2, (m, k)) * 0.37).astype(np.float32)
        wire = R.quantize(t, w)
        deq = R.to_float(t, wire, m, k)
        x = rng.uniform(-1, 1, (n, k)).astype(np.float32)
        out[f"{name}.wire"] = wire
        if name in DEQUANT_STORED:
            out[f"{name}.dequant"] = deq
        else:
            out[f"{name}.dequant_sha256"] = np.array(hashlib.sha256(deq.tobytes()).hexdigest())
        out[f"{name}.y"] = R.mul_mat(t, wire, x, m, n_threads=2)[0]
    # GGML_OP_FUSED_UP_GATE (silu, op_params limit) through the reference CPU backend on Q4_0 weights
    t, m, k = GGML_TYPE["Q4_0"], 256, 512
    wu, wg = make_wire("Q4_0", m, k, seed=61), make_wire("Q4_0", m, k, seed=62)
    x = np.random.default_rng(9).standard_normal((1, k)).astype(np.float32) * 6
    for limit in (0.0, 1.5):
        out[f"fused_up_gate.Q4_0.silu.limit{limit}"] = R.fused_up_gate(t, wu, wg, x, m, "silu", limit)
    np.savez_compressed(os.path.join(HERE, "reference_xcheck.npz"), **out)


def main():
    R = RefLib()
    if sys.argv[1:] == ["--xcheck"]:
        return xcheck(R)
    only = sys.argv[1:]
    for name in TYPES + ORACLE_ONLY + WIRE_TYPES:
        if only and name not in only:
            continue
        t = GGML_TYPE[name]
        rng = np.random.default_rng(1234 + t)
        w = (rng.standard_normal((M, K)) * 0.02).astype(np.float32)
        w[0, :32] = 0.0                       # an all-zero block (d == 0 edge case)
        w[1, 5] = 1.5                         # an outlier
        if name in ("IQ2_BN", "IQ1_BN"):     # ternary weights so the quantiser is lossless (SURVEY.md §8d)
            w = (rng.integers(-1, 2, (M, K)) * 0.043).astype(np.float32)
        x = rng.uniform(-1, 1, (N, K)).astype(np.float32)
        x[0, :32] = 0.0                       # an all-zero activation block (amax == 0 edge case of quantize_q8_1)
        wire = R.quantize(t, w)
        deq = R.to_float(t, wire, M, K)
        y_cpu, _ = R.mul_mat(t, wire, x, M, n_threads=1)
        np.savez_compressed(os.path.join(HERE, f"{name}.npz"), ggml_type=t, m=M, k=K, n=N, wire=wire, x=x,
                            dequant_ref=deq, y_ref_cpu=y_cpu, row_size=R.row_size(t, K))
        print(name, "wire", wire.size, "row_size", R.row_size(t, K))


if __name__ == "__main__":
    main()
