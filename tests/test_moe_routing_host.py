"""CPU tests of the MoE routing arithmetic (ik_llama_cpp_b200/csrc/b200q_moe.cuh).  The same __host__ __device__ functions build the
expert-sorted rows and the tile table on the GPU (k_moe_route); here they are compiled with g++ and compared with numpy."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "host_emul", "moe_route.cpp")
HDR = os.path.join(ROOT, "ik_llama_cpp_b200", "csrc", "b200q_moe.cuh")


@pytest.fixture(scope="module")
def moe(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("moe_route") / "libmoe_route.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    L = ctypes.CDLL(so)
    p = ctypes.c_void_p
    L.emul_moe_route.argtypes = [p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, p, p, p, p, p, p]
    L.emul_moe_tiles_bound.argtypes = [ctypes.c_int] * 3
    L.emul_moe_clamp.argtypes = [ctypes.c_int] * 2
    return L


def route(L, ids, nb1, n_expert, bn):
    n_tokens, n_used = ids.shape
    n_rows = n_tokens * n_used
    bound = L.emul_moe_tiles_bound(n_rows, n_expert, bn)
    ids = np.ascontiguousarray(ids, np.int32)
    counts, bounds, toff = np.zeros(n_expert, np.int32), np.zeros(n_expert + 1, np.int32), np.zeros(n_expert + 1, np.int32)
    src, dst = np.full(n_rows, -1, np.int32), np.full(n_rows, -1, np.int32)
    tiles = np.full((bound + 1, 4), -7, np.int32)                # one spare entry: must stay untouched
    c = lambda a: a.ctypes.data
    nt = L.emul_moe_route(c(ids), n_tokens, n_used, nb1, n_expert, bn, c(counts), c(bounds), c(toff), c(src), c(dst), c(tiles))
    return nt, bound, bounds, src, dst, tiles


def reference(ids, nb1, n_expert, bn):
    n_tokens, n_used = ids.shape
    e = np.clip(ids.reshape(-1), 0, n_expert - 1)
    counts = np.bincount(e, minlength=n_expert)
    bounds = np.concatenate([[0], np.cumsum(counts)])
    order = np.argsort(e, kind="stable")                         # sorted by expert, slot order inside an expert
    t, slot = order // n_used, order % n_used
    tiles = [(x, c0, bounds[x + 1]) for x in range(n_expert) for c0 in range(bounds[x], bounds[x + 1], bn)]
    return bounds, t * nb1 + slot % nb1, order, tiles


def check(L, ids, nb1, n_expert, bn):
    nt, bound, bounds, src, dst, tiles = route(L, ids, nb1, n_expert, bn)
    rb, rsrc, rdst, rtiles = reference(ids, nb1, n_expert, bn)
    n_rows = ids.size
    assert np.array_equal(bounds, rb)
    assert np.array_equal(src, rsrc) and np.array_equal(dst, rdst)
    assert nt == len(rtiles) <= bound
    assert [tuple(r[:3]) for r in tiles[:nt]] == [tuple(map(int, r)) for r in rtiles]
    assert (tiles[bound:] == -7).all()
    cover = np.zeros(n_rows, np.int32)                           # every sorted row lies in exactly one tile, of its own expert
    for x, c0, c1, _ in tiles[:nt]:
        cover[c0:min(c0 + bn, c1)] += 1
        assert bounds[x] <= c0 < c1 == bounds[x + 1]
    assert (cover == 1).all()
    assert sorted(dst.tolist()) == list(range(n_rows))           # every output row written once


@pytest.mark.parametrize("bn", [128, 256, 512])
@pytest.mark.parametrize("n_tokens,n_used,n_expert,nb1", [(1, 1, 1, 1), (1, 8, 128, 1), (7, 2, 8, 2), (512, 8, 128, 1), (333, 2, 8, 2), (2048, 6, 64, 3)])
def test_random_ids(moe, bn, n_tokens, n_used, n_expert, nb1):
    rng = np.random.default_rng(n_tokens * 7 + n_expert)
    ids = np.stack([rng.permutation(n_expert)[:n_used] for _ in range(n_tokens)]) if n_used <= n_expert else rng.integers(0, n_expert, (n_tokens, n_used))
    check(moe, ids.astype(np.int32), nb1, n_expert, bn)


@pytest.mark.parametrize("bn", [128, 256])
def test_adversarial_ids(moe, bn):
    rng = np.random.default_rng(3)
    # every slot on one expert (many tiles, last one partial)
    check(moe, np.full((700, 2), 5, np.int32), 2, 8, bn)
    # out-of-range ids: clamped into [0, n_expert), as the mat-vec kernel does
    check(moe, rng.integers(-1000, 1000, (300, 4)).astype(np.int32), 1, 16, bn)
    check(moe, np.array([[np.iinfo(np.int32).min, np.iinfo(np.int32).max]], np.int32), 1, 4, bn)
    # most experts empty, a token choosing the same expert twice
    ids = np.where(rng.random((257, 2)) < 0.5, 3, 250).astype(np.int32); ids[::5, 1] = ids[::5, 0]
    check(moe, ids, 2, 256, bn)
    # counts one above / below a tile
    ids = np.concatenate([np.zeros(bn + 1, np.int32), np.ones(bn - 1, np.int32)]).reshape(-1, 1)
    check(moe, ids, 1, 2, bn)


def test_clamp_and_bound(moe):
    assert [moe.emul_moe_clamp(i, 8) for i in (-5, -1, 0, 7, 8, 1 << 30)] == [0, 0, 0, 7, 7, 7]
    for n_rows, n_expert, bn in [(1, 128, 128), (4096, 128, 128), (1024, 8, 512), (100000, 512, 256)]:
        assert moe.emul_moe_tiles_bound(n_rows, n_expert, bn) == -(-n_rows // bn) + min(n_expert, n_rows)
