"""CPU tests: pin the oracle restatement to the reference (golden vectors recorded from the reference library)."""
import hashlib

import numpy as np
import pytest

from conftest import ALL_TYPES, ORACLE_ONLY_TYPES, load_golden
from oracle.oracle import GGML_TYPE, nmse

REF_CPU_DEVIATES = {"IQ4_XS", "IQ5_KS", "IQ4_KSS", "IQ2_KT"}      # reference CPU kernels that deviate from their own to_float (SURVEY §8c pitfall 2; IQ2_KT: NMSE 2.6e-3)
# IQ6_K: the reference's to_float evaluates a float cubic (iqk_quantize.cpp:3442-3486) that its build contracts into FMAs: not bit-reproducible without them
FMA_DEPENDENT = {"IQ6_K"}


def _assert_dequant_equal(name, a, b):
    if name in ("IQ4_KS", "IQ5_KS"):       # dl*(v+4) vs dl*v + 4*dl association: <= 1 ulp
        np.testing.assert_allclose(a, b, rtol=2e-7, atol=0)
    elif name in FMA_DEPENDENT:            # cancellation near the cubic's zero
        np.testing.assert_allclose(a, b, rtol=3e-6, atol=1e-5 * float(np.abs(b).max()))
    else:
        assert np.array_equal(a, b), f"{name}: dequantize != reference to_float (bit-exact expected)"


@pytest.mark.parametrize("name", ALL_TYPES)
def test_oracle_dequant_matches_reference_golden(oracle, name):
    g = load_golden(name)
    t, m, k = int(g["ggml_type"]), int(g["m"]), int(g["k"])
    assert oracle.row_size(t, k) == int(g["row_size"])
    deq = oracle.dequantize(t, g["wire"], m, k)
    _assert_dequant_equal(name, deq, g["dequant_ref"])


@pytest.mark.parametrize("name", ALL_TYPES)
def test_oracle_mul_mat_vs_reference_cpu_backend_golden(oracle, name):
    """test-backend-ops semantics (tests/test-backend-ops.cpp:979-981): NMSE(reference CPU backend, exact) <= 5e-4."""
    g = load_golden(name)
    t, m = int(g["ggml_type"]), int(g["m"])
    exact = oracle.mul_mat_exact(t, g["wire"], g["x"], m)
    if name in REF_CPU_DEVIATES:
        # SURVEY.md §8c pitfall 2: the reference's direct CPU kernel for this type is off by NMSE ~1e-2 from its own
        # to_float (reproduced here with the unmodified reference build) -> ground truth is the f64 dot, not the CPU backend.
        assert nmse(g["y_ref_cpu"], exact) <= 1e-1
    else:
        assert nmse(g["y_ref_cpu"], exact) <= 5e-4
    q8 = oracle.mul_mat_q8_1(t, g["wire"], g["x"], m)
    assert nmse(q8, exact) <= 5e-4


def test_quantize_q8_1_restatement(oracle):
    rng = np.random.default_rng(7)
    x = rng.standard_normal((3, 256)).astype(np.float32)
    x[1, 32:64] = 0.0
    q, d, s = oracle.quantize_q8_1(x)
    xb = x.reshape(3, 8, 32)
    amax = np.abs(xb).max(-1)
    np.testing.assert_array_equal(d, (amax / np.float32(127)).astype(np.float16))
    assert np.all(q.reshape(3, 8, 32)[1, 1] == 0) and d[1, 1] == 0
    assert np.abs(q).max() <= 127
    # |x - d*q| <= d/2 (+ rounding of d to half is applied only to the stored scale)
    dq = (amax / np.float32(127))[..., None]
    assert np.all(np.abs(xb - dq * q.reshape(3, 8, 32)) <= dq * 0.5 + 1e-7)
    np.testing.assert_allclose(s.astype(np.float32), xb.sum(-1), rtol=2e-3, atol=1e-3)


def test_b200_quantizer_variant_vs_reference_variant(oracle):
    """The product's quantiser (one division per block, rint) must agree with the reference's (roundf(x/d)) except at ties."""
    rng = np.random.default_rng(11)
    x = rng.standard_normal((8, 4096)).astype(np.float32)
    q0, d0, _ = oracle.quantize_q8_1(x)
    q1, d1 = oracle.quantize_q8_1_b200(x)
    assert np.array_equal(d0, d1)
    diff = np.abs(q0.astype(np.int32) - q1.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).mean() <= 1e-3


def test_half_conversions(oracle):
    hs = np.arange(0, 65536, 7, dtype=np.uint16)
    f = np.array([oracle.lib.oracle_h2f(int(h)) for h in hs], np.float32)
    ref = hs.view(np.float16).astype(np.float32)
    ok = np.isfinite(ref)
    np.testing.assert_array_equal(f[ok], ref[ok])
    back = np.array([oracle.lib.oracle_f2h(float(v)) for v in ref[ok]], np.uint16)
    np.testing.assert_array_equal(back, hs[ok])


@pytest.mark.parametrize("name", ALL_TYPES)
def test_oracle_vs_live_reference(oracle, name):
    """Cross-check against the unmodified reference library on a second data set: what it computed is recorded in
    reference_xcheck.npz (tests/golden/gen_golden.py --xcheck): the wire bytes of its quantiser for the weights drawn below, its
    to_float (as a SHA-256 of the f32 bytes where the match must be bit-exact) and its CPU MUL_MAT."""
    g = load_golden("reference_xcheck")
    t = GGML_TYPE[name]
    rng = np.random.default_rng(99 + t)
    m, k, n = 8, 1024, 2
    rng.standard_normal((m, k))            # the weights the reference quantised into `wire`, drawn so that x below is the recorded one
    if name in ("IQ2_BN", "IQ1_BN"):
        rng.integers(-1, 2, (m, k))
    wire = g[f"{name}.wire"]
    assert wire.size == m * oracle.row_size(t, k)
    a = oracle.dequantize(t, wire, m, k)
    if f"{name}.dequant" in g:
        _assert_dequant_equal(name, a, g[f"{name}.dequant"])
    else:       # bit-exact, IQ4_KS / IQ5_KS included: on these weights their one-ulp association difference does not occur (gen_golden.py)
        assert hashlib.sha256(a.tobytes()).hexdigest() == str(g[f"{name}.dequant_sha256"]), f"{name}: dequantize != reference to_float (bit-exact expected)"
    x = rng.uniform(-1, 1, (n, k)).astype(np.float32)
    assert nmse(g[f"{name}.y"], oracle.mul_mat_exact(t, wire, x, m)) <= (1e-1 if name in REF_CPU_DEVIATES else 5e-4)


@pytest.mark.parametrize("name", ORACLE_ONLY_TYPES)
def test_oracle_only_types_are_pinned_to_the_reference(oracle, name):
    """Types staged for the next round: the oracle (with the codebook extracted from the running reference, tests/golden/gen_codebooks.py)
    must already equal the reference to_float bit-for-bit on reference-quantised data, and reproduce the MMVQ / exact relation."""
    g = load_golden(name)
    t, m, k = int(g["ggml_type"]), int(g["m"]), int(g["k"])
    assert oracle.supported(t) and oracle.row_size(t, k) == int(g["row_size"])
    deq = oracle.dequantize(t, g["wire"], m, k)
    if name == "IQ6_K":     # the reference to_float evaluates a float cubic (iqk_quantize.cpp:3442-3486); its build contracts it into FMAs
        np.testing.assert_allclose(deq, g["dequant_ref"], rtol=3e-6, atol=1e-5 * float(np.abs(g["dequant_ref"]).max()))   # cancellation near the cubic's zero
    else:
        assert np.array_equal(deq, g["dequant_ref"])
    exact = oracle.mul_mat_exact(t, g["wire"], g["x"], m)
    # the reference CPU backend agrees with the f64 dot on its own to_float (IQ4_KSS: same small-n deviation as IQ4_KS/IQ5_KS, SURVEY §8c pitfall 2)
    assert nmse(g["y_ref_cpu"], exact) <= (1e-1 if name == "IQ4_KSS" else 5e-4)
    assert nmse(oracle.mul_mat_q8_1(t, g["wire"], g["x"], m), exact) <= 5e-4
