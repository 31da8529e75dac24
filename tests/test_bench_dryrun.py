"""bench.py's model skeleton walked on the CPU with a stub backend: catches plumbing errors (names, argument lists, buffer shapes)
before GPU time is spent on them.  No kernels run here."""
import os
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench


class _T:
    def __init__(self, m, k, ggml_type=20):
        self.m, self.k, self.nbytes_wire, self.ggml_type = m, k, m * k * 18 // 32, ggml_type


class _BE:
    class Q8Scratch:
        def __init__(self, k):
            self.k, self.valid = k, False

    calls = []

    def prefetch_next(self, ws, gate=None):
        assert all(hasattr(w, "m") for w in ws)

    def mul_mat(self, w, x, out=None, x_bf16=None, q8_in=None):
        assert x.shape[1] == w.k and (out is None or out.shape[1] == w.m)
        self.calls.append("mul_mat"); return out

    def mul_mat_multi(self, ws, x, outs=None, x_bf16=None):
        assert all(x.shape[1] == w.k and o.shape[1] == w.m for w, o in zip(ws, outs))
        self.calls.append("multi"); return outs

    def fused_up_gate(self, up, gate, x, unary="silu", limit=0.0, out=None, x_bf16=None, out_bf16=None, q8_out=None):
        assert x.shape[1] == up.k and out.shape[1] == up.m
        self.calls.append("upgate"); return out

    def convert_activations(self, x, out=None):
        assert out.shape == x.shape
        self.calls.append("cvt"); return out


def test_model_skeleton_walks_tg_and_pp(monkeypatch):
    monkeypatch.setattr(bench, "random_planes", lambda be, torch_, name, m, k, gen, scale: _T(m, k))
    gen = types.SimpleNamespace(manual_seed=lambda s: None)
    tt = types.SimpleNamespace(Generator=lambda device=None: gen, empty=lambda s, dtype=None, device=None: torch.empty(s, dtype=dtype),
                               float32=torch.float32, bfloat16=torch.bfloat16)
    be = _BE()
    m = bench.Model(be, tt, 2)
    m.alloc(1); m.step_tg()
    assert be.calls.count("multi") == 2 and be.calls.count("upgate") == 2 and be.calls.count("mul_mat") == 5
    assert m.launches_tg == 9
    be.calls.clear()
    m.alloc(512); m.step_pp()
    assert be.calls.count("cvt") == 6 and be.calls.count("mul_mat") == 5
    assert bench.model_bytes_per_token(32) == 4221370368
    # the default quantisation mix: attn_v has its own type, so it gets its own launch
    monkeypatch.setattr(bench, "random_planes", lambda be, torch_, name, m, k, gen, scale: _T(m, k, bench.MIX_TYPES[name][0]))
    be.calls.clear()
    mm = bench.Model(be, tt, 2, mix="default")
    mm.alloc(1); mm.step_tg()
    assert be.calls.count("multi") == 2 and be.calls.count("mul_mat") == 7 and mm.launches_tg == 11
    assert mm.head.ggml_type == 14 and mm.layers[0]["down"].ggml_type == 13 and mm.layers[1]["wv"].ggml_type == 140
    mm.alloc(512); mm.step_pp()


def test_time_graph_times_exactly_steps_replays():
    """--steps is the timed loop count: time_graph brackets exactly `steps` graph replays with its two timing events and divides by steps."""
    log = []

    class _Ctx:
        def __enter__(self): return self
        def __exit__(self, *a): return False

    class _Event:
        def __init__(self, enable_timing=False): pass
        def record(self): log.append("record")
        def elapsed_time(self, other): return 14.0

    class _Graph:
        def replay(self): log.append("replay")

    stream = types.SimpleNamespace(wait_stream=lambda s: None)
    cuda = types.SimpleNamespace(Stream=lambda: stream, current_stream=lambda: stream, stream=lambda s: _Ctx(), synchronize=lambda: None,
                                 CUDAGraph=_Graph, graph=lambda g: _Ctx(), Event=_Event)
    for steps in (1, 7, 40):
        log.clear()
        ms = bench.time_graph(types.SimpleNamespace(cuda=cuda), lambda: log.append("eager"), steps, warmup=2)
        i0, i1 = log.index("record"), len(log) - 1 - log[::-1].index("record")
        assert log[i0 + 1:i1] == ["replay"] * steps and ms == 14.0 / steps
