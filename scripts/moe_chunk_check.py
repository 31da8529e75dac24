"""MoE token-chunk check (run by tests/test_gpu_parity.py::test_mul_mat_id_token_chunks in child processes, with and without B200Q_MOE_CHUNK_TOKENS):
20 tokens through b200q_mul_mat_id_vec, both activation-column modes, against the mat-vec oracle on the selected expert."""
import os, sys, numpy as np, torch
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
from conftest import make_wire
from ik_llama_cpp_b200 import backend as be
from oracle.oracle import GGML_TYPE, Oracle
orc = Oracle(); t = GGML_TYPE["IQ4_NL"]; n_expert, n_used, m, k, n_tokens = 5, 2, 132, 1024, 20
wires = [make_wire("IQ4_NL", m, k, seed=900 + e) for e in range(n_expert)]
W = be.set_expert_tensor(t, np.concatenate(wires), n_expert, m, k)
rng = np.random.default_rng(3)
for nb1 in (1, 2):
    x = rng.standard_normal((n_tokens, nb1, k)).astype(np.float32)
    ids = np.stack([rng.permutation(n_expert)[:n_used] for _ in range(n_tokens)]).astype(np.int32)
    y = be.mul_mat_id(W, torch.from_numpy(x).cuda(), torch.from_numpy(ids).cuda()).cpu().numpy()
    for tk in range(n_tokens):
        for e in range(n_used):
            ref = orc.mul_mat_q8_1(t, wires[ids[tk, e]], x[tk, e % nb1][None, :], m, variant="b200")[0]
            assert np.abs(y[tk, e] - ref).max() <= 5e-5 * float(np.sqrt((ref.astype(np.float64) ** 2).mean())), (nb1, tk, e)
print("CHUNKS-OK", os.environ.get("B200Q_MOE_CHUNK_TOKENS"))
