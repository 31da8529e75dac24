import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
ORACLE_ONLY_TYPES = []
# plane layout (b200q_types.cuh: 16-byte low-bit plane per 32 weights, TMA-ring mat-vec, fused tcgen05 prefill for the 2-plane types)
PLANE_TYPES = ["Q4_0", "Q4_1", "Q5_0", "Q5_1", "Q6_0", "Q8_0", "Q2_K", "Q3_K", "Q4_K", "Q5_K", "Q6_K", "IQ4_NL", "IQ4_XS", "IQ2_K", "IQ3_K", "IQ4_K", "IQ5_K", "IQ4_KS", "IQ5_KS", "IQ2_KS", "IQ3_KS", "MXFP4", "IQ2_BN"]
# wire layout (b200q_wire.cuh: GGUF bytes verbatim, generic decode): grid-codebook, trellis and row-interleaved types
WIRE_TYPES = ["IQ2_XXS", "IQ2_XS", "IQ3_XXS", "IQ2_S", "IQ3_S", "IQ6_K", "IQ1_BN", "IQ4_KSS", "IQ1_S", "IQ1_M", "IQ2_KL", "IQ1_KT", "IQ2_KT", "IQ3_KT", "IQ4_KT",
              "IQ1_S_R4", "IQ1_M_R4", "IQ2_K_R4", "IQ3_K_R4", "IQ4_K_R4", "IQ5_K_R4", "IQ4_KS_R4", "IQ5_KS_R4"]
ALL_TYPES = PLANE_TYPES + WIRE_TYPES      # every quantized type the reference's CUDA back-end accepts for MUL_MAT (ggml-cuda.cu:4862-4917)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle import Oracle
    return Oracle()


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"))
    return {k: z[k] for k in z.files}


def make_wire(name, m, k, seed, quantised=False):
    """Wire bytes for a random tensor: random but VALID wire blocks (every bit pattern of the payload is a valid encoding; scales are
    drawn as sane fp16/f32 values).  quantised=True, and always for the codebook / trellis / row-interleaved types: blocks and row
    headers resampled from the golden tensor the reference's own quantiser produced, i.e. data with the statistics of real quantiser output."""
    rng = np.random.default_rng(seed)
    if quantised:
        return _resample_golden_wire(name, m, k, rng)
    return random_wire(name, m, k, rng)


# byte offsets of fp16 scale fields inside one wire block, per type: (block_bytes, [offsets of half fields], row_meta)
_GEOM = {
    "Q4_0": (18, [0], 0), "Q4_1": (20, [0, 2], 0), "Q5_0": (22, [0], 0), "Q5_1": (24, [0, 2], 0), "Q6_0": (26, [0], 0), "Q8_0": (34, [0], 0), "IQ4_NL": (18, [0], 0), "Q4_K": (144, [0, 2], 0), "Q5_K": (176, [0, 2], 0),
    "IQ2_K": (76, [0], 0), "IQ3_K": (110, [0], 0), "Q2_K": (84, [80, 82], 0), "Q3_K": (110, [108], 0), "Q6_K": (210, [208], 0), "IQ4_XS": (136, [0], 0), "IQ4_K": (144, [0], 0), "IQ5_K": (176, [0], 0), "IQ4_KS": (136, [], 4), "IQ5_KS": (168, [], 4), "IQ2_KS": (70, [], 2), "IQ3_KS": (102, [], 2), "MXFP4": (17, [], 0), "IQ2_BN": (16, [], 4),
}
_QK = {"Q4_0": 32, "Q4_1": 32, "Q5_0": 32, "Q5_1": 32, "Q6_0": 32, "Q8_0": 32, "IQ4_NL": 32, "MXFP4": 32, "IQ2_BN": 64}


# per-ROW wire geometry of the wire-layout types: (weights per block, block bytes, row header bytes, rows interleaved)
_WIRE_GEOM = {"IQ2_XXS": (256, 66, 0, 1), "IQ2_XS": (256, 74, 0, 1), "IQ3_XXS": (256, 98, 0, 1), "IQ2_S": (256, 82, 0, 1), "IQ3_S": (256, 110, 0, 1), "IQ1_S": (256, 50, 0, 1),
              "IQ1_M": (256, 56, 0, 1), "IQ6_K": (256, 212, 0, 1), "IQ4_KSS": (256, 128, 4, 1), "IQ2_KL": (256, 86, 2, 1), "IQ1_BN": (64, 13, 2, 1), "IQ1_KT": (256, 56, 4, 1),
              "IQ2_KT": (256, 68, 4, 1), "IQ3_KT": (256, 100, 4, 1), "IQ4_KT": (256, 128, 4, 1), "IQ1_S_R4": (32, 6, 2, 4), "IQ1_M_R4": (32, 7, 2, 4), "IQ2_K_R4": (256, 76, 0, 4),
              "IQ3_K_R4": (256, 110, 0, 4), "IQ4_K_R4": (256, 144, 0, 4), "IQ5_K_R4": (256, 176, 0, 4), "IQ4_KS_R4": (256, 136, 4, 4), "IQ5_KS_R4": (256, 168, 4, 4)}


def _resample_golden_wire(name, m, k, rng):
    """Valid wire bytes of a wire-layout type without the reference library (GPU box): row groups assembled from randomly drawn blocks and
    row headers of the committed golden tensor (which the reference's own quantiser produced)."""
    qk, bs, meta, il = _WIRE_GEOM[name] if name in _WIRE_GEOM else (_QK.get(name, 256), _GEOM[name][0], _GEOM[name][2], 1)
    g = load_golden(name)
    gm, gk = int(g["m"]), int(g["k"])
    assert m % il == 0 and k % qk == 0
    gw = g["wire"].reshape(gm // il, il * (meta + (gk // qk) * bs))
    heads = gw[:, :il * meta]
    blocks = gw[:, il * meta:].reshape(gm // il, gk // qk, il * bs)
    ng, nb = m // il, k // qk
    out = np.empty((ng, il * meta + nb * il * bs), np.uint8)
    out[:, :il * meta] = heads[rng.integers(0, gm // il, ng)]
    out[:, il * meta:] = blocks[rng.integers(0, gm // il, (ng, nb)), rng.integers(0, gk // qk, (ng, nb))].reshape(ng, nb * il * bs)
    return out.reshape(-1)


def random_wire(name, m, k, rng):
    if name in _WIRE_GEOM:
        return _resample_golden_wire(name, m, k, rng)
    bs, halfs, meta = _GEOM[name]
    qk = _QK.get(name, 256)
    nb = k // qk
    rows = np.empty((m, meta + nb * bs), np.uint8)
    blocks = rng.integers(0, 256, (m, nb, bs), dtype=np.uint8)
    for off in halfs:
        sc = (rng.uniform(0.5, 2.0, (m, nb)) * 1e-3).astype(np.float16)
        if off in (2, 82):   # dmin of Q4_K/Q5_K/Q2_K: keep it small
            sc = (rng.uniform(0.0, 1.0, (m, nb)) * 1e-4).astype(np.float16)
        blocks[:, :, off:off + 2] = sc.view(np.uint8).reshape(m, nb, 2)
    if name == "MXFP4":   # E8M0 block exponent: keep the scale in a sane range (2^-18 .. 2^-4), every other bit pattern is payload
        blocks[:, :, 0] = rng.integers(110, 125, (m, nb), dtype=np.uint8)
    rows[:, meta:] = blocks.reshape(m, nb * bs)
    if meta == 2:       # IQ2_KS / IQ3_KS: ggml_half row scale
        rs = (rng.uniform(0.5, 2.0, m) * 1e-3).astype(np.float16)
        rows[:, :2] = rs.view(np.uint8).reshape(m, 2)
    if meta == 4:
        rs = (rng.uniform(0.5, 2.0, m) * 1e-3).astype(np.float32)
        rows[:, :4] = rs.view(np.uint8).reshape(m, 4)
    return rows.reshape(-1)
