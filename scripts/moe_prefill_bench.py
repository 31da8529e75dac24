"""MoE prefill: the grouped tcgen05 GEMM (b200q_mul_mat_id_gemm) against the mat-vec kernel walked in token chunks (b200q_mul_mat_id_vec).

One MoE FFN layer per point: MOE_FUSED_UP_GATE (silu) on the token's column, then MUL_MAT_ID of the down experts on the per-slot columns
(nb1 = n_used), for Qwen3-30B-A3B-shaped experts (2048 -> 768, 128 experts, 8 used) and Mixtral-8x7B-shaped experts (4096 -> 14336, 8
experts, 2 used), in IQ4_NL and Q4_K, at several batch sizes.  Expert ids are seeded and uniform (each token picks n_used distinct experts);
the "skew" variant sends half of the tokens to expert 0.  Both paths run in this process, alternating, timed with CUDA events after warm-up.
The expert weights (340 MB / 793 MB per layer) exceed the 126 MB L2, so every layer streams them from HBM.

    python scripts/moe_prefill_bench.py --out DIR [--tokens 8,16,...] [--shapes qwen3,mixtral] [--types IQ4_NL,Q4_K]

Per point: us per layer and tokens/s of both paths, algorithmic TFLOP/s (2 * n_tokens * n_used * M * K per matrix, three matrices),
active-expert weight bytes over time, NMSE between the two results.  DIR/moe_prefill_bench.json also records the GPU name, power limit and
max SM clock, read with nvidia-smi in the same run (query only)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import random_wire                          # noqa: E402  (valid random wire blocks with sane scales)
from ik_llama_cpp_b200 import backend as be               # noqa: E402
from oracle.oracle import GGML_TYPE                       # noqa: E402

SHAPES = {   # d_model, expert ffn, n_expert, n_used
    "qwen3": (2048, 768, 128, 8),
    "mixtral": (4096, 14336, 8, 2),
}


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [s.strip() for s in out.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clk}
    except Exception as e:      # noqa: BLE001
        return {"error": repr(e), "torch_name": torch.cuda.get_device_name()}


def expert_tensor(name, n_expert, m, k, seed):
    t = GGML_TYPE[name]
    rng = np.random.default_rng(seed)
    wire = np.concatenate([random_wire(name, m, k, rng) for _ in range(n_expert)])
    return be.set_expert_tensor(t, wire, n_expert, m, k)


def make_ids(n_tokens, n_expert, n_used, skew, rng):
    ids = np.stack([rng.permutation(n_expert)[:n_used] for _ in range(n_tokens)]).astype(np.int32)
    if skew:        # half of the tokens pick expert 0 (in their first slot, the other slots stay distinct)
        for t in range(0, n_tokens, 2):
            row = [0] + [e for e in ids[t] if e != 0][: n_used - 1]
            ids[t] = row
    return ids


def time_paths(fns, iters, reps):
    """fns: {name: callable}.  Alternates the paths `reps` times, `iters` calls per window; returns the median us per call of each."""
    ev = {n: [] for n in fns}
    for _ in range(reps):
        for n, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                f()
            b.record()
            b.synchronize()
            ev[n].append(a.elapsed_time(b) * 1e3 / iters)
    return {n: float(np.median(v)) for n, v in ev.items()}


def nmse(a, b):
    a = a.double(); b = b.double()
    return float(((a - b) ** 2).sum() / max(float((b ** 2).sum()), 1e-300))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--tokens", default="8,16,32,64,128,512,2048")
    ap.add_argument("--shapes", default="qwen3,mixtral")
    ap.add_argument("--types", default="IQ4_NL,Q4_K")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--min-window-ms", type=float, default=30.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("moe_prefill_bench: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    print("GPU:", info, flush=True)
    tokens = [int(s) for s in args.tokens.split(",")]
    points = []
    t_start = time.time()
    for shape in args.shapes.split(","):
        d, ff, n_expert, n_used = SHAPES[shape]
        for tname in args.types.split(","):
            up, gate = expert_tensor(tname, n_expert, ff, d, 1), expert_tensor(tname, n_expert, ff, d, 2)
            down = expert_tensor(tname, n_expert, d, ff, 3)
            pb_ug = be.plane_bytes(GGML_TYPE[tname], ff, d)
            pb_dn = be.plane_bytes(GGML_TYPE[tname], d, ff)
            for n in tokens:
                for skew in (False, True):
                    rng = np.random.default_rng(1000 * n + skew)
                    ids = torch.from_numpy(make_ids(n, n_expert, n_used, skew, rng)).cuda()
                    x = torch.from_numpy(rng.standard_normal((n, 1, d)).astype(np.float32)).cuda()
                    h_v = torch.empty((n, n_used, ff), device="cuda"); h_g = torch.empty_like(h_v)

                    def layer_vec():
                        h = be.mul_mat_id(up, x, ids, gate=gate, unary="silu")
                        return be.mul_mat_id(down, h, ids)

                    def layer_gemm():
                        be.mul_mat_id_gemm(up, x, ids, gate=gate, unary="silu", out=h_g)
                        return be.mul_mat_id_gemm(down, h_g, ids)

                    y_v, y_g = layer_vec(), layer_gemm()           # warm-up (module load, workspace, tensor-map encoders)
                    torch.cuda.synchronize()
                    err = nmse(y_g, y_v)
                    # calls per timing window: enough for min_window_ms of the slower path
                    t0 = time.time(); layer_vec(); torch.cuda.synchronize(); tv = time.time() - t0
                    iters = max(1, min(200, int(args.min_window_ms / 1e3 / max(tv, 1e-6))))
                    us = time_paths({"vec": layer_vec, "gemm": layer_gemm}, iters, args.reps)
                    flops = 2.0 * n * n_used * (2 * ff * d + d * ff)
                    active = int(torch.unique(ids).numel())
                    wbytes = active * (2 * pb_ug + pb_dn)
                    p = {"shape": shape, "type": tname, "n_tokens": n, "skew": skew, "d_model": d, "ffn": ff, "n_expert": n_expert, "n_used": n_used,
                         "active_experts": active, "iters": iters, "reps": args.reps, "nmse_gemm_vs_vec": err}
                    for path in ("vec", "gemm"):
                        p[f"{path}_us"] = us[path]
                        p[f"{path}_tok_s"] = n / (us[path] * 1e-6)
                        p[f"{path}_tflops"] = flops / (us[path] * 1e-6) / 1e12
                        p[f"{path}_weight_GBs"] = wbytes / (us[path] * 1e-6) / 1e9
                    p["speedup_gemm"] = us["vec"] / us["gemm"]
                    points.append(p)
                    print(f"{shape:8s} {tname:7s} n={n:5d} {'skew' if skew else 'unif'}  vec {us['vec']:10.1f} us  gemm {us['gemm']:10.1f} us  "
                          f"x{p['speedup_gemm']:6.2f}  gemm {p['gemm_tflops']:6.1f} TFLOP/s {p['gemm_weight_GBs']:7.0f} GB/s  nmse {err:.2e}", flush=True)
            del up, gate, down
            torch.cuda.empty_cache()
    res = {"gpu": info, "torch": torch.__version__, "seconds": time.time() - t_start, "points": points,
           "note": "one MoE FFN layer (MOE_FUSED_UP_GATE silu + MUL_MAT_ID down); vec = b200q_mul_mat_id_vec, gemm = b200q_mul_mat_id_gemm"}
    with open(os.path.join(args.out, "moe_prefill_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", os.path.join(args.out, "moe_prefill_bench.json"))


if __name__ == "__main__":
    main()
