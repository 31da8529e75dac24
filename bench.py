#!/usr/bin/env python
"""bench.py — llama-bench-shaped measurement of the quantized mat-mul hot path on B200.

Workload (BASELINE.json configs[1]): Llama-3-8B, pure IQ4_NL (`llama-quantize --pure`), synthetic random-init weights.
One "step" = one pass of the hot path over one batch:
  * tg128: ONE token (n_batch = 1) through every MUL_MAT of the model, in graph order:
           32 x [ QKV (one multi-tensor mat-vec launch) -> wo -> fused up/gate/SiLU -> ffn_down ] -> output head.
           129 launches of our k_mmvq kernel and nothing else (attention/norm/rope are NOT the hot path and are not run;
           the q projection is fed straight to wo so the chain keeps the dependency structure).  On one GPU every layer's
           Q,K,V read the same unit-rms activation in place of the RMS norm of the residual stream (see Model), so that
           the logits are not zero.
  * pp512: the same matrices with n_batch = 512 through the tcgen05 GEMM path (head on the last token only,
           as llama-bench does); the SiLU*mul glue between up/gate and down is a torch elementwise op.
Weights live in HBM in the plane layout (uploaded through the C-ABI repack); 4.2 GB of weights per pass >> 126 MB L2,
so every timed iteration streams from HBM ("inputs larger than L2").

value  = tok/s with inputs already resident in HBM (CUDA-graph replay of the step, CUDA-event timed, max over ranks)
e2e    = tok/s through host buffers: pinned-host activations H2D + the same launches + logits D2H, every step
N > 1  = the fork's "split mode graph" tensor parallelism: QKV/up/gate row-sharded, wo/down K-sharded + all-reduce (NCCL).

--impl reference times the reference's own CPU IQK path (oracle/_ref, the unmodified ggml CPU backend) on a bounded
sample of the same workload (one transformer layer's mat-muls), scaled to the whole token.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Llama-3-8B (SURVEY.md §8): per-layer matmul shapes (M x K)
N_EMBD, N_FF, N_LAYER, N_VOCAB, N_KV_DIM = 4096, 14336, 32, 128256, 1024
IQ4_NL = 20


def model_bytes_per_token(n_layer=N_LAYER, tp=1):
    per_layer_w = N_EMBD * N_EMBD * 2 + 2 * N_KV_DIM * N_EMBD + 3 * N_FF * N_EMBD
    return (per_layer_w * n_layer + N_VOCAB * N_EMBD) * 18 // 32


def model_flops_pp(n_tokens, n_layer=N_LAYER):
    per_layer_w = N_EMBD * N_EMBD * 2 + 2 * N_KV_DIM * N_EMBD + 3 * N_FF * N_EMBD
    return 2.0 * per_layer_w * n_layer * n_tokens + 2.0 * N_VOCAB * N_EMBD


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(s[0]) for s in self.samples if len(s) >= 7 and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 7 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            if len(s) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def random_planes_iq4nl(be, torch, m, k, gen, scale):
    """Random valid IQ4_NL wire blocks made on the GPU, then re-laid-out by the product's repack kernel."""
    nb = m * (k // 32)
    blocks = torch.randint(0, 256, (nb, 18), dtype=torch.uint8, device="cuda", generator=gen)
    d = (torch.rand(nb, device="cuda", generator=gen) * 0.6 + 0.7) * scale
    # random sign per block: the IQ4_NL codebook has a non-zero mean (-5.9), with all-positive d every matrix would amplify the mean of its input
    d = d * (torch.randint(0, 2, (nb,), device="cuda", generator=gen).float() * 2 - 1)
    blocks[:, 0:2] = d.to(torch.float16).view(torch.uint8).view(nb, 2)
    return be.set_tensor(IQ4_NL, blocks.view(-1), m, k)


# wire geometry of the types of the default `llama-quantize ... IQ4_NL` mix (SURVEY.md §8 a-note): (ggml type id, block bytes, weights per block,
# byte offsets of ggml_half scale fields that get a sane value, of ggml_half min fields that get a small one)
MIX_TYPES = {"IQ4_NL": (20, 18, 32, [0], []), "Q5_K": (13, 176, 256, [0], [2]), "Q6_K": (14, 210, 256, [208], []), "IQ5_K": (140, 176, 256, [0], [])}


def random_planes(be, torch, name, m, k, gen, scale):
    """Random valid wire blocks of a mix type made on the GPU (every payload bit pattern is a valid encoding), re-laid-out by the product."""
    if name == "IQ4_NL":
        return random_planes_iq4nl(be, torch, m, k, gen, scale)
    t, bs, qk, d_off, m_off = MIX_TYPES[name]
    nb = m * (k // qk)
    blocks = torch.randint(0, 256, (nb, bs), dtype=torch.uint8, device="cuda", generator=gen)
    # sub-block scales of these types are ~6-bit integers: scale the super-block d down accordingly
    d = (torch.rand(nb, device="cuda", generator=gen) * 0.6 + 0.7) * scale / 32.0
    for o in d_off:
        blocks[:, o:o + 2] = d.to(torch.float16).view(torch.uint8).view(nb, 2)
    for o in m_off:
        blocks[:, o:o + 2] = (d * 0.01).to(torch.float16).view(torch.uint8).view(nb, 2)
    return be.set_tensor(t, blocks.view(-1), m, k)


class Model:
    """Llama-3-8B matmul skeleton, optionally one tensor-parallel shard (rank r of tp)."""

    def __init__(self, be, torch, n_layer, tp=1, rank=0, seed=1234, collective=True, mix="pure"):
        """collective=False: only the weights of rank `rank`'s shard (no reducer, no head): used by rank 0 to rebuild the other ranks'
        shards for the tensor-parallel correctness gate."""
        self.be, self.torch, self.tp, self.n_layer = be, torch, tp, n_layer
        gen = torch.Generator(device="cuda")
        gen.manual_seed(seed + rank)
        # unit-gain weights (IQ4_NL codebook rms ~ 70).  There is no norm between the layers of this MUL_MAT-only skeleton and silu(g)*u makes the
        # magnitude map quadratic: chained from layer to layer the values would vanish within ~8 layers (all 32 then compute zeros) or
        # overflow.  On one GPU the Q,K,V of every layer therefore read self.x, a unit-rms activation standing in for the normed residual
        # stream; wo, up/gate and ffn_down still consume their predecessor's output, and the launches are the same.  The tensor-parallel
        # paths keep the layer-to-layer chain: the fused kernels take the reduced output of the previous layer as their input
        s_e, s_f = 1.0 / (70.0 * N_EMBD ** 0.5), 1.0 / (70.0 * N_FF ** 0.5)
        # mix = "default": what `llama-quantize model IQ4_NL` produces WITHOUT --pure on this GQA model (src/llama-quantize.cpp:617-621, 739-745, 385-388):
        # attn_v -> IQ5_K, ffn_down of the first n_layer/8 layers -> Q5_K, output.weight -> Q6_K, everything else IQ4_NL
        self.mix = mix
        mk = lambda m, k, s, name="IQ4_NL": random_planes(be, torch, name, m, k, gen, s)
        dflt = mix == "default"
        self.layers = []
        for li in range(n_layer):
            self.layers.append(dict(
                wq=mk(N_EMBD // tp, N_EMBD, s_e), wk=mk(N_KV_DIM // tp, N_EMBD, s_e), wv=mk(N_KV_DIM // tp, N_EMBD, s_e, "IQ5_K" if dflt else "IQ4_NL"),
                wo=mk(N_EMBD, N_EMBD // tp, s_e), up=mk(N_FF // tp, N_EMBD, s_e), gate=mk(N_FF // tp, N_EMBD, s_e),
                down=mk(N_EMBD, N_FF // tp, s_f, "Q5_K" if dflt and li < N_LAYER // 8 else "IQ4_NL")))
        self.head = mk(N_VOCAB // tp, N_EMBD, s_e, "Q6_K" if dflt else "IQ4_NL") if collective else None
        self.launches_tg = n_layer * (5 if dflt else 4) + 1      # (attn_v has its own type in the default mix: it cannot ride in the Q,K launch)
        self.reducer = None
        self.fused_tp = False
        self.bf16_reduce = False
        if tp > 1 and collective and os.environ.get("B200Q_NCCL_REDUCE", "0") != "1":
            self.reducer = be.NvlsReducer(512 * N_EMBD)
            # decode: the reduce fused into the mat-vecs (tagged-slot exchange) wins at 2 ranks (595-631 vs 574 tok/s) but its cost grows with the number
            # of ranks (+4.5 us per exchange at N = 2, +9.5 us at N = 4: 511-532 tok/s), while the one-shot reduce kernel's rendezvous did not grow with N
            # in round 1 -> more than 2 ranks use the separate reduce kernel unless B200Q_TP_FUSED says otherwise (profiles/r2_tp_timeline.md)
            self.fused_tp = self.reducer.ok and os.environ.get("B200Q_TP_FUSED", "1" if tp <= 2 else "0") == "1"
            self.bf16_reduce = self.reducer.ok and os.environ.get("B200Q_TP_BF16_REDUCE", "1") == "1"
            self.launches_tg += 2 * n_layer if (self.reducer.ok and not self.fused_tp) else 0
        self.weight_bytes = sum(t.nbytes_wire for L in self.layers for t in L.values()) + (self.head.nbytes_wire if self.head is not None else 0)

    def alloc(self, n):
        t, tp = self.torch, self.tp
        f = lambda *s: t.empty(s, dtype=t.float32, device="cuda")
        self.x = f(n, N_EMBD); self.q = f(n, N_EMBD // tp); self.kk = f(n, N_KV_DIM // tp); self.v = f(n, N_KV_DIM // tp)
        self.h = f(n, N_EMBD); self.a = f(n, N_FF // tp); self.x2 = f(n, N_EMBD); self.logits = f(1, N_VOCAB // tp)
        self.q8a = self.be.Q8Scratch(N_FF // tp) if n == 1 else None
        self.u = f(n, N_FF // tp) if n > 8 else None
        self.g = f(n, N_FF // tp) if n > 8 else None
        b = lambda *s: t.empty(s, dtype=t.bfloat16, device="cuda")
        self.xb, self.qb, self.hb, self.ab = (b(n, N_EMBD), b(n, N_EMBD // tp), b(n, N_EMBD), b(n, N_FF // tp)) if n > 8 else (None,) * 4

    def allreduce(self, t):
        if self.tp > 1:
            if self.reducer is not None:
                self.reducer.all_reduce(t)          # our NVLS kernel (falls back to NCCL without multicast support)
            else:
                import torch.distributed as dist
                dist.all_reduce(t)

    def step_tg_fused_tp(self, with_head=True):
        """tp > 1: the two GGML_OP_REDUCE per layer are fused into the mat-vec kernels (multimem.red from the wo / ffn_down epilogue,
        flag wait in the prologue of the next mat-vec): 4 launches per layer like the single-GPU graph, no reduce kernel."""
        be, r = self.be, self.reducer
        first = True
        for L in self.layers:
            be.mul_mat_vec_tp([L["wq"], L["wk"], L["wv"]], self.x if first else None, [self.q, self.kk, self.v], r, reduce_in=not first)
            be.mul_mat_vec_tp([L["wo"]], self.q, None, r, reduce_out=True)
            be.mul_mat_vec_tp([L["up"]], None, [self.a], r, reduce_in=True, gate=L["gate"], unary="silu")
            be.mul_mat_vec_tp([L["down"]], self.a, None, r, reduce_out=True)
            first = False
        if with_head:
            be.mul_mat_vec_tp([self.head], None, [self.logits], r, reduce_in=True)
        else:               # (correctness gate) a consumer that only materialises the reduced vector
            be.mul_mat_vec_tp([self.layers[0]["wq"]], None, [self.q], r, reduce_in=True)

    def step_tg(self, with_head=True):
        be = self.be
        if self.tp > 1 and self.fused_tp:
            return self.step_tg_fused_tp(with_head)
        x = self.x
        pf = getattr(be, "prefetch_next", lambda *a, **k: None)       # every launch warms the first stages of the NEXT launch's weights in L2
        nl = len(self.layers)
        for li, L in enumerate(self.layers):
            xq = x if self.tp > 1 else self.x
            pf([L["wo"]])
            if L["wv"].ggml_type == L["wq"].ggml_type:
                be.mul_mat_multi([L["wq"], L["wk"], L["wv"]], xq, [self.q, self.kk, self.v])
            else:
                be.mul_mat_multi([L["wq"], L["wk"]], xq, [self.q, self.kk]); be.mul_mat(L["wv"], xq, out=self.v)
            pf([L["up"]], gate=L["gate"])
            be.mul_mat(L["wo"], self.q, out=self.h); self.allreduce(self.h)
            pf([L["down"]])
            # the up/gate launch also emits its result quantised to q8_1 (once, in its tail) for ffn_down
            be.fused_up_gate(L["up"], L["gate"], self.h, "silu", out=self.a, q8_out=self.q8a)
            if li + 1 < nl:
                N = self.layers[li + 1]; pf([N["wq"], N["wk"], N["wv"]])
            elif with_head:
                pf([self.head])
            be.mul_mat(L["down"], self.a, out=self.x2, q8_in=self.q8a); self.allreduce(self.x2)
            x = self.x2
        if with_head:
            be.mul_mat(self.head, x, out=self.logits)

    def step_pp(self, with_head=True):
        be, t = self.be, self.torch
        x = self.x
        have_xb = False
        for li, L in enumerate(self.layers):
            xq = x if self.tp > 1 else self.x
            if not have_xb:
                be.convert_activations(xq, self.xb)     # f32 -> bf16 once per distinct activation (shared by Q,K,V)
            if L["wv"].ggml_type == L["wq"].ggml_type:
                be.mul_mat_multi([L["wq"], L["wk"], L["wv"]], xq, [self.q, self.kk, self.v], x_bf16=self.xb)      # one launch
            else:
                be.mul_mat_multi([L["wq"], L["wk"]], xq, [self.q, self.kk], x_bf16=self.xb); be.mul_mat(L["wv"], xq, out=self.v, x_bf16=self.xb)
            be.convert_activations(self.q, self.qb)
            be.mul_mat(L["wo"], self.q, out=self.h, x_bf16=self.qb)
            if self.bf16_reduce:
                # GGML_OP_REDUCE with a bf16 payload (the reference casts the partial when ne[1] > 32): two-shot in the switch, the result
                # is the bf16 activation operand of the next GEMM (no f32 -> bf16 pass)
                self.reducer.all_reduce_bf16(self.h, out_bf16=self.hb)
            else:
                self.allreduce(self.h)
                be.convert_activations(self.h, self.hb)
            # FUSED_UP_GATE (n > 8): up GEMM, gate GEMM with silu(gate)*up in its epilogue; it also emits the bf16 operand of ffn_down
            be.fused_up_gate(L["up"], L["gate"], self.h, "silu", out=self.a, x_bf16=self.hb, out_bf16=self.ab)
            be.mul_mat(L["down"], self.a, out=self.x2, x_bf16=self.ab)
            if self.bf16_reduce:
                last = li == len(self.layers) - 1
                self.reducer.all_reduce_bf16(self.x2, out_bf16=self.xb, out_f32=self.x2 if last else None)    # f32 copy only where a mat-vec (head) reads it
                have_xb = True
            else:
                self.allreduce(self.x2)
            x = self.x2
        if with_head:
            be.mul_mat(self.head, x[-1:], out=self.logits)


def bitnet_line(be, torch, steps, warmup, hbm_peak, outputs):
    """BASELINE.json configs[3] / SURVEY App. A config 4: bitnet-b1.58-3B (n_embd 3200, n_ff 8640, 26 layers), IQ2_BN (2.0 bpw + f32 row scale), the
    per-layer MUL_MAT nodes only (the output matrix of that model is not IQ2_BN).  K = 3200 / 8640 are not multiples of 256: decode takes the TMA ring
    through the byte-granular geometry, prefill the int8 tensor-core path (ternary x int8 activations, tcgen05 kind::i8)."""
    E, FF, NL, T = 3200, 8640, 26, 135
    gen = torch.Generator(device="cuda"); gen.manual_seed(4321)
    def mk(m, k):
        rows = torch.randint(0, 256, (m, 4 + (k // 64) * 16), dtype=torch.uint8, device="cuda", generator=gen)
        rs = (torch.rand(m, device="cuda", generator=gen) * 0.6 + 0.7) / k ** 0.5 * (torch.randint(0, 2, (m,), device="cuda", generator=gen).float() * 2 - 1)
        rows[:, 0:4] = rs.view(torch.uint8).view(m, 4)
        return be.set_tensor(T, rows.view(-1), m, k)
    layers = [dict(wq=mk(E, E), wk=mk(E, E), wv=mk(E, E), wo=mk(E, E), up=mk(FF, E), gate=mk(FF, E), down=mk(E, FF)) for _ in range(NL)]
    wbytes = sum(t.nbytes_wire for L in layers for t in L.values())
    f = lambda *sh: torch.empty(sh, dtype=torch.float32, device="cuda")
    out = {"workload": "bitnet-b1.58-3B IQ2_BN (BASELINE.json configs[3]): the 26 layers' MUL_MAT / FUSED_UP_GATE nodes in graph order, no output matrix",
           "algorithmic_bytes_per_step": wbytes}
    for n in (1, 512):
        x, q, k_, v, h, a, x2 = f(n, E), f(n, E), f(n, E), f(n, E), f(n, E), f(n, FF), f(n, E)
        x.normal_()
        def step():
            for L in layers:
                be.mul_mat_multi([L["wq"], L["wk"], L["wv"]], x, [q, k_, v])      # every layer reads the unit-rms x, as in Model
                be.mul_mat(L["wo"], q, out=h)
                be.fused_up_gate(L["up"], L["gate"], h, "silu", out=a)
                be.mul_mat(L["down"], a, out=x2)
        ms = time_graph(torch, step, steps, warmup)
        outputs[f"bitnet_{'tg' if n == 1 else 'pp512'}_hidden"] = x2
        if n == 1:
            ach = wbytes / (ms * 1e-3) / 1e9
            out["tg"] = {"value": 1000.0 / ms, "unit": "tok/s", "ms_per_step": ms, "launches_per_step": 4 * NL,
                         "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak}}
        else:
            ops = 2.0 * sum(t.m * t.k for L in layers for t in L.values()) * n
            out["pp512"] = {"value": n * 1000.0 / ms, "unit": "tok/s", "ms_per_step": ms, "dtype": "u8 (ternary) x s8 activations -> s32 (tcgen05 kind::i8), f32 rescale",
                            "achieved_int8_TOP/s": ops / (ms * 1e-3) / 1e12}
    return out


def tp_correctness_gate(be, torch, dist, model, rank, world, n, n_check_layers=2, tol=5e-4):
    """N > 1 only, before anything is timed: the reduced hidden state of a 2-layer slice of THIS model, computed by the tensor-parallel
    path (all ranks, the collectives under test), must match what rank 0 gets by rebuilding every rank's shard locally (same seeds),
    running each shard through the single-GPU kernels and summing the row-parallel partials in f64.  NMSE > tol -> every rank exits non-zero."""
    saved = model.layers
    model.layers = saved[:n_check_layers]
    model.alloc(n)
    gen = torch.Generator(device="cuda"); gen.manual_seed(777)
    x0 = torch.randn(n, N_EMBD, device="cuda", generator=gen)          # identical on every rank
    model.x.copy_(x0)
    if n == 1:
        model.step_tg(with_head=False)
        torch.cuda.synchronize()
        got = model.reducer.reduced_view(N_EMBD)[None, :].double() if model.fused_tp else model.x2.double()
    else:
        model.step_pp(with_head=False)
        torch.cuda.synchronize()
        got = model.x2.double()
    verdict = torch.zeros(1, device="cuda")
    err = float("nan")
    if rank == 0:
        shards = [model if r == 0 else Model(be, torch, n_check_layers, tp=world, rank=r, collective=False) for r in range(world)]
        x = x0.clone()
        for li in range(n_check_layers):
            part = torch.zeros(n, N_EMBD, dtype=torch.float64, device="cuda")
            for sh in shards:
                L = sh.layers[li]
                q = be.mul_mat(L["wq"], x)                               # (wk / wv feed attention, which is not on this path)
                part += be.mul_mat(L["wo"], q).double()
            h = part.float()
            part = torch.zeros(n, N_EMBD, dtype=torch.float64, device="cuda")
            for sh in shards:
                L = sh.layers[li]
                a = be.fused_up_gate(L["up"], L["gate"], h, "silu")
                part += be.mul_mat(L["down"], a).double()
            x = part.float()
        ref = x.double()
        err = float(((got - ref) ** 2).sum() / (ref ** 2).sum())
        verdict[0] = 0.0 if err <= tol else 1.0
        del shards
    dist.all_reduce(verdict)
    model.layers = saved
    torch.cuda.empty_cache()
    return err, float(verdict.item()) == 0.0


def time_graph(torch, fn, steps, warmup, dist=None, pre=None, post=None):
    """Capture fn into a CUDA graph, W warm-up replays, then K replays bracketed by barrier+sync, CUDA-event timed."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()                                   # eager warm-up (sets func attributes, allocates workspaces)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()

    def one():
        if pre: pre()
        g.replay()
        if post: post()

    for _ in range(max(warmup, 3)):
        one()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms = e0.elapsed_time(e1) / steps
    if dist is not None:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def cpu_baseline(n_threads=None, budget_s=12.0, n=1):
    """Reference CPU IQK path (oracle/_ref) on ONE transformer layer's mat-muls, scaled to the whole model."""
    from oracle.oracle import RefLib
    path = RefLib.find(prefer_native=True)
    if path is None:
        return None
    R = RefLib(path)
    n_threads = n_threads or max(1, (os.cpu_count() or 2) // 2)
    shapes = [(N_EMBD, N_EMBD), (N_KV_DIM, N_EMBD), (N_KV_DIM, N_EMBD), (N_EMBD, N_EMBD), (N_FF, N_EMBD), (N_FF, N_EMBD), (N_EMBD, N_FF)]
    import ctypes
    nm = len(shapes)
    types = (ctypes.c_int * nm)(*[IQ4_NL] * nm)
    ms_ = (ctypes.c_int64 * nm)(*[s[0] for s in shapes]); ks_ = (ctypes.c_int64 * nm)(*[s[1] for s in shapes])
    ch = R.lib.refshim_chain_new(nm, types, ms_, ks_, n, n_threads)
    rng = np.random.default_rng(0)
    for i, (m, k) in enumerate(shapes):
        nb = m * (k // 32)
        blocks = rng.integers(0, 256, (nb, 18), dtype=np.uint8)
        blocks[:, 0:2] = (rng.uniform(0.7, 1.3, nb) / (70.0 * k ** 0.5)).astype(np.float16).view(np.uint8).reshape(nb, 2)
        x = rng.standard_normal((n, k)).astype(np.float32)
        R.lib.refshim_chain_set(ch, i, blocks.ctypes.data, x.ctypes.data)
    R.lib.refshim_chain_run(ch)                    # warm-up
    t0, times = time.time(), []
    while time.time() - t0 < budget_s and len(times) < 200:
        times.append(R.lib.refshim_chain_run(ch))
    R.lib.refshim_chain_free(ch)
    layer_s = float(np.median(times))
    layer_w = sum(m * k for m, k in shapes)
    total_w = layer_w * N_LAYER + N_VOCAB * N_EMBD * (1 if n == 1 else 1.0 / n)
    step_s = layer_s * total_w / layer_w
    return {"value": n / step_s, "unit": "tok/s", "cores": n_threads, "kind": "reference",
            "sample": f"{len(times)} runs of one layer's 7 MUL_MATs (218 M weights, IQ4_NL, n={n}) through the unmodified reference CPU backend "
                      f"({os.path.basename(path)}), median {layer_s*1e3:.2f} ms/layer, scaled x{total_w/layer_w:.2f} to the full model"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=N_LAYER, help="debug only: a run with fewer layers is not a bench value")
    ap.add_argument("--no-pp", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-mix", action="store_true", help="skip the default-quantisation-mix line (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what each timed path computed in its last step "
                    "(logits, final hidden states) as DIR/<name>.npy, float32; the inputs are seeded, so runs of two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    config = {"reduce": "b200q NVLS kernel" if world > 1 and os.environ.get("B200Q_NCCL_REDUCE", "0") != "1" else ("nccl" if world > 1 else "none"), "workload": "Llama-3-8B pure IQ4_NL, llama-bench tg128 (n_batch=1) / pp512 (n_ubatch=512): all MUL_MAT nodes in graph order",
              "n_layer": args.layers, "l2_policy": "inputs larger than L2 (4.2 GB of weights streamed per step)",
              "parallelism": f"tp{world}" if world > 1 else "none"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # "all the host threads it can use": the reference's spin-barrier thread pool collapses when oversubscribed
        # (SURVEY.md §8c pitfall 4), so calibrate the thread count on a short sample and keep the fastest
        ncpu = os.cpu_count() or 8
        cands = sorted({max(1, ncpu), max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 16), min(ncpu, 8)}, reverse=True)
        best = None
        for nt in cands:
            c = cpu_baseline(n_threads=nt, budget_s=2.5)
            if c and (best is None or c["value"] > best[1]["value"]):
                best = (nt, c)
        cb = cpu_baseline(n_threads=best[0], budget_s=12.0) if best else None
        if cb:
            cb["sample"] += f"; thread count calibrated over {cands} (logical CPUs: {ncpu})"
        if cb is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (reference CPU build) not present"}))
            return 0
        line = {"metric": "llama-bench tg128 tok/s (MUL_MAT hot path)", "value": cb["value"], "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "int8 (IQ4_NL weights x Q8 activations, f32 accumulate)", "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    from ik_llama_cpp_b200 import backend as be
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device — the hot path has no CPU fallback", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.manual_seed(0)
    # name -> host copy of what a timed path computed in its last step, taken right after that path's timing, before its buffers are reused
    outputs = {}

    def keep(**ts):
        if args.dump_outputs:
            outputs.update({k: t.float().cpu() for k, t in ts.items()})

    model = Model(be, torch, args.layers, tp=world, rank=rank)
    if model.fused_tp:
        config["reduce"] = "tg: fused into the mat-vec kernels (wo/ffn_down epilogue broadcasts tagged partial rows with multimem.st, the next mat-vec's prologue sums them); pp512: " + \
            ("two-shot bf16 NVLS kernel (multimem.ld_reduce + multimem.st)" if model.bf16_reduce else "one-shot f32 NVLS kernel")
    elif model.reducer is not None and model.reducer.ok:
        config["reduce"] = "tg: one-shot f32 NVLS reduce kernel after wo / ffn_down (multimem.red + multicast flag; default for more than 2 ranks, see Model); pp512: " + \
            ("two-shot bf16 NVLS kernel (multimem.ld_reduce + multimem.st)" if model.bf16_reduce else "one-shot f32 NVLS kernel")
    # ---------------- N > 1: correctness gate on the collectives, before anything is timed ----------------
    if world > 1:
        gate = {}
        ok_all = True
        for n_chk, nm in ((1, "tg"), (512, "pp512")):
            if nm == "pp512" and args.no_pp:
                continue
            err, ok = tp_correctness_gate(be, torch, dist, model, rank, world, n_chk)
            gate[nm] = err
            ok_all = ok_all and ok
        config["tp_gate"] = {"nmse_vs_unsharded": gate, "tol": 5e-4, "layers_checked": 2}
        if not ok_all:
            if rank == 0:
                print(f"bench.py: tensor-parallel correctness gate FAILED: NMSE of the reduced hidden state vs the unsharded result = {gate}", file=sys.stderr)
            dist.destroy_process_group()
            return 3
    # ---------------- tg128 ----------------
    model.alloc(1)
    x_host = torch.randn(1, N_EMBD).pin_memory()
    logits_host = torch.empty(1, N_VOCAB // world).pin_memory()
    model.x.copy_(x_host)
    with ClockSampler(local_rank) as cs:
        ms_tg = time_graph(torch, model.step_tg, args.steps, args.warmup, dist)
    clocks = cs.summary()
    keep(tg_logits=model.logits)
    ms_tg_e2e = time_graph(torch, model.step_tg, args.steps, args.warmup, dist,
                           pre=lambda: model.x.copy_(x_host, non_blocking=True),
                           post=lambda: (logits_host.copy_(model.logits, non_blocking=True), torch.cuda.current_stream().synchronize()))
    tok_s = 1000.0 / ms_tg
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # the pp512 timed region is ~0.1 s at full SM clock: that is the BURST regime of MEASURED_PEAKS (its sustained figure was taken after 4 s at
    # a 1410 MHz median); report against the burst peak and give the sustained fraction next to it
    tf_peak = float(peaks.get("bf16_tflops", 1722.0))
    tf_peak_sustained = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    bytes_tok = model.weight_bytes
    traffic, traffic_src = {}, None
    try:   # DRAM bytes per step measured by ncu --set full (scripts/make_traffic.py, committed under profiles/), N = 1 only
        tf = [f for f in ("r2_traffic.json", "r1_traffic.json") if os.path.exists(os.path.join(ROOT, "profiles", f))]
        traffic = json.load(open(os.path.join(ROOT, "profiles", tf[0]))) if tf and world == 1 and args.layers == N_LAYER else {}
        traffic_src = f"static: profiles/{tf[0]} (ncu --set full capture of the same kernels, not measured in this run)" if traffic else None
    except Exception:
        pass
    ach = bytes_tok / (ms_tg * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": "k_mmvq<IQ4_NL>", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic.get("tg", {}).get("dram_bytes_per_step"),
            "traffic_source": traffic_src, "algorithmic_bytes_per_step": bytes_tok, "launches_per_step": model.launches_tg, "peak_source": peak_src,
            "note": "the step consists only of k_mmvq launches; achieved = weight bytes per token / step time (per rank)"}
    line = {"metric": "llama-bench tg128 tok/s (MUL_MAT hot path)", "value": tok_s, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_tg, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int8 (IQ4_NL weights x q8_1 activations, dp4a, f32 accumulate)", "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": 1000.0 / ms_tg_e2e, "unit": "tok/s", "h2d_bytes_per_step": N_EMBD * 4, "d2h_bytes_per_step": (N_VOCAB // world) * 4},
            "gpu_launches": model.launches_tg * args.steps, "roofline": roof}
    # ---------------- pp512 ----------------
    if not args.no_pp:
        n = 512
        model.alloc(n)
        xh = torch.randn(n, N_EMBD).pin_memory()
        model.x.copy_(xh)
        ms_pp = time_graph(torch, model.step_pp, args.steps, args.warmup, dist)
        keep(pp512_logits=model.logits, pp512_hidden=model.x2)
        ms_pp_e2e = time_graph(torch, model.step_pp, args.steps, args.warmup, dist,
                               pre=lambda: model.x.copy_(xh, non_blocking=True),
                               post=lambda: (logits_host.copy_(model.logits, non_blocking=True), torch.cuda.current_stream().synchronize()))
        fl = model_flops_pp(n, args.layers) / world
        tfs = fl / (ms_pp * 1e-3) / 1e12
        line["pp512"] = {"metric": "llama-bench pp512 tok/s (MUL_MAT hot path)", "value": n * 1000.0 / ms_pp, "unit": "tok/s", "ms_per_step": ms_pp, "steps": args.steps,
                         "dtype": "bf16 x bf16 -> f32 (tcgen05 kind::f16)", "e2e": {"value": n * 1000.0 / ms_pp_e2e, "unit": "tok/s", "h2d_bytes_per_step": n * N_EMBD * 4, "d2h_bytes_per_step": (N_VOCAB // world) * 4},
                         "roofline": {"bound": "tensor", "kernel": "k_gemm_q<IQ4_NL> (fused dequant + tcgen05; + k_f32_to_bf16)", "achieved": tfs, "peak": tf_peak, "unit": "TFLOP/s", "frac": tfs / tf_peak,
                                      "traffic": traffic.get("pp", {}).get("dram_bytes_per_step_gemm_only"), "traffic_source": traffic_src, "algorithmic_flops_per_step": fl,
                                      "peak_source": peak_src + " burst (timed region << 1 s at max SM clock)", "frac_of_sustained_peak": tfs / tf_peak_sustained}}
    # ---------------- the default quantisation mix next to --pure (N = 1): IQ5_K attn_v, Q5_K ffn_down x4, Q6_K output ----------------
    if world == 1 and not args.no_mix and args.layers == N_LAYER:
        del model
        torch.cuda.empty_cache()
        mm = Model(be, torch, args.layers, mix="default")
        mm.alloc(1); mm.x.copy_(x_host)
        ms_m = time_graph(torch, mm.step_tg, args.steps, args.warmup)
        keep(mix_tg_logits=mm.logits)
        ach_m = mm.weight_bytes / (ms_m * 1e-3) / 1e9
        mix = {"workload": "same model, default `llama-quantize ... IQ4_NL` mix (no --pure): attn_v IQ5_K, ffn_down of layers 0-3 Q5_K, output.weight Q6_K",
               "tg": {"value": 1000.0 / ms_m, "unit": "tok/s", "ms_per_step": ms_m, "launches_per_step": mm.launches_tg,
                      "roofline": {"bound": "hbm", "achieved": ach_m, "peak": hbm_peak, "unit": "GB/s", "frac": ach_m / hbm_peak, "algorithmic_bytes_per_step": mm.weight_bytes}}}
        if not args.no_pp:
            mm.alloc(512); mm.x.copy_(xh)
            ms_mp = time_graph(torch, mm.step_pp, args.steps, args.warmup)
            keep(mix_pp512_logits=mm.logits, mix_pp512_hidden=mm.x2)
            tfm = model_flops_pp(512, args.layers) / (ms_mp * 1e-3) / 1e12
            mix["pp512"] = {"value": 512 * 1000.0 / ms_mp, "unit": "tok/s", "ms_per_step": ms_mp,
                            "roofline": {"bound": "tensor", "achieved": tfm, "peak": tf_peak, "unit": "TFLOP/s", "frac": tfm / tf_peak}}
        line["default_mix"] = mix
        del mm
        torch.cuda.empty_cache()
        try:
            bitnet_out = {}
            line["bitnet"] = bitnet_line(be, torch, args.steps, args.warmup, hbm_peak, bitnet_out)
            keep(**bitnet_out)
        except Exception as e:      # a side line must never cost the headline
            line["bitnet"] = {"error": repr(e)}
    # ---------------- cpu baseline (rank 0, N=1 only) ----------------
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            # the reference's spin-barrier pool collapses when oversubscribed: pick the better of two thread counts on a short sample
            ncpu = os.cpu_count() or 8
            trial = [(nt, cpu_baseline(n_threads=nt, budget_s=1.5)) for nt in sorted({max(1, ncpu // 2), min(ncpu, 16)})]
            trial = [(nt, c) for nt, c in trial if c]
            cb = cpu_baseline(n_threads=max(trial, key=lambda t: t[1]["value"])[0], budget_s=8.0) if trial else None
            if cb:
                line["cpu_baseline"] = cb
        except Exception as e:  # the baseline is a reported number, never a reason to lose the bench line
            line["cpu_baseline"] = {"error": repr(e)}
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in outputs.items():      # tensor parallel: each rank writes its own shard
            np.save(os.path.join(args.dump_outputs, f"{name}.npy" if world == 1 else f"{name}.rank{rank}.npy"), t.numpy())
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
