// b200q_moe.cu — grouped MoE prefill: device-side routing, gather of the routed activations, then the grouped mode of k_gemm_q
// (b200q_gemm.cu) over expert-sorted token tiles.  Nothing is read back to the host, so the whole sequence can be captured in a CUDA graph.
//
//   k_moe_route          ids -> counts, bounds, row_src, row_dst, tile table, number of tiles (one CTA)
//   k_moe_gather_bf16    x f32 [n_tokens * nb1][K] -> bf16 [n_rows][K] in sorted order (row r = column row_src[r])
//   k_gemm_q<T, NB, 1>   blockIdx.x: 128-row weight tile (of up, then gate), blockIdx.y: tile-table entry; the expert is the third
//                        coordinate of the weight tensor maps; column c of the tile is stored at output row row_dst[col0 + c]
//   k_mul_unary          MOE_FUSED_UP_GATE only: dst = unary(gate) * up over all n_rows x M results
#include "b200q_internal.h"
#include "b200q_moe.cuh"
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstring>

namespace {

constexpr int ROUTE_WARPS = 16;
constexpr int MOE_MAX_EXPERTS = 512;             // routing histogram: ROUTE_WARPS x n_expert ints of shared memory

// One CTA.  Pass 1: each warp counts a contiguous segment of the slots per expert (lanes with the same expert are grouped with
// __match_any_sync; the group leader adds its size).  A column scan over the warps turns the per-warp counts into per-warp starting
// offsets, thread 0 scans the experts (b200q_moe_scan).  Pass 2: each warp walks its segment again in order and places every slot at
// bounds[e] + (rows of e in earlier warps) + (rows of e earlier in this warp): a stable sort by expert, identical to b200q_moe_route_serial.
__global__ void __launch_bounds__(32 * ROUTE_WARPS) k_moe_route(const int32_t * __restrict__ ids, int n_tokens, int n_used, int nb1, int n_expert, int bn,
                                                              int * __restrict__ bounds_out, int * __restrict__ row_src, int * __restrict__ row_dst,
                                                              b200q_moe_tile * __restrict__ tiles, int * __restrict__ n_tiles) {
    extern __shared__ int sm[];
    int * hist = sm;                                      // [ROUTE_WARPS][n_expert]
    int * counts = hist + ROUTE_WARPS * n_expert;         // [n_expert]
    int * bounds = counts + n_expert;                     // [n_expert + 1]
    int * toff = bounds + n_expert + 1;                   // [n_expert + 1]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_rows = n_tokens * n_used;
    const int seg = (n_rows + ROUTE_WARPS - 1) / ROUTE_WARPS, s0 = warp * seg, s1 = min(n_rows, s0 + seg);
    int * h = hist + warp * n_expert;
    for (int i = threadIdx.x; i < ROUTE_WARPS * n_expert; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int base = s0; base < s1; base += 32) {          // warp-uniform bounds
        const int s = base + lane;
        const int e = s < s1 ? b200q_moe_clamp(__ldg(ids + s), n_expert) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, e);
        if (e >= 0 && lane == __ffs(peers) - 1) h[e] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n_expert; e += blockDim.x) {
        int run = 0;
        for (int w = 0; w < ROUTE_WARPS; ++w) { const int v = hist[w * n_expert + e]; hist[w * n_expert + e] = run; run += v; }
        counts[e] = run;
    }
    __syncthreads();
    if (threadIdx.x == 0) *n_tiles = b200q_moe_scan(counts, n_expert, bn, bounds, toff);
    __syncthreads();
    for (int e = threadIdx.x; e <= n_expert; e += blockDim.x) bounds_out[e] = bounds[e];
    for (int e = threadIdx.x; e < n_expert; e += blockDim.x) b200q_moe_expert_tiles(e, bounds, toff, bn, tiles);
    const unsigned lt = (1u << lane) - 1u;
    for (int base = s0; base < s1; base += 32) {
        const int s = base + lane;
        const int e = s < s1 ? b200q_moe_clamp(__ldg(ids + s), n_expert) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, e);
        if (e >= 0) {
            const int r = bounds[e] + h[e] + __popc(peers & lt);
            const int t = s / n_used, slot = s - t * n_used;
            row_src[r] = b200q_moe_src_col(t, slot, nb1); row_dst[r] = b200q_moe_dst_row(t, slot, n_used);
        }
        __syncwarp();
        if (e >= 0 && lane == __ffs(peers) - 1) h[e] += __popc(peers);
        __syncwarp();
    }
}

// out[r][:] = bf16(x[row_src[r]][:]): a thread converts 8 consecutive values (two LDG.128 -> one STG.128), U groups in flight (as k_f32_to_bf16)
__global__ void __launch_bounds__(256) k_moe_gather_bf16(const float * __restrict__ x, const int * __restrict__ row_src, __nv_bfloat16 * __restrict__ out,
                                                         int64_t K, int64_t n_rows) {
    constexpr int U = 4;
    const int64_t k8 = K / 8, total8 = n_rows * k8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < total8; i0 += U * stride) {
        float4 a[U], b[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i < total8) {
                const int64_t r = i / k8, c = i % k8;
                const float4 * p = reinterpret_cast<const float4 *>(x + (int64_t)__ldg(row_src + r) * K + 8 * c);
                a[u] = __ldg(p); b[u] = __ldg(p + 1);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i < total8) {
                __nv_bfloat162 p0 = __floats2bfloat162_rn(a[u].x, a[u].y), p1 = __floats2bfloat162_rn(a[u].z, a[u].w), p2 = __floats2bfloat162_rn(b[u].x, b[u].y), p3 = __floats2bfloat162_rn(b[u].z, b[u].w);
                uint4 o; o.x = *reinterpret_cast<uint32_t *>(&p0); o.y = *reinterpret_cast<uint32_t *>(&p1); o.z = *reinterpret_cast<uint32_t *>(&p2); o.w = *reinterpret_cast<uint32_t *>(&p3);
                *reinterpret_cast<uint4 *>(out + i * 8) = o;
            }
        }
    }
}

}  // namespace

// Tile width from the average rows per expert.  A CTA decodes its 128 x K weight slab once per token tile, so a tile at least as wide as
// the rows an expert typically receives decodes each active expert's weights about once; a wider tile only adds masked MMA columns and
// B-tile loads (cheap next to the decode, which bounds k_gemm_q).  Hence the smallest of BN = 128 / 256 / 512 that covers the average:
// NB = 0 for many small experts (Qwen3-30B-A3B at 512 tokens: 32 rows per expert), NB = 1 or 2 for few large ones (Mixtral: 128+).
static int moe_choose_nb(int64_t n_rows, int n_expert) {
    const int64_t avg = (n_rows + n_expert - 1) / n_expert;
    return avg <= 128 ? 0 : (avg <= 256 ? 1 : 2);
}

int b200q_moe_plan(int type, int64_t m, int64_t k, int n_expert, int n_used, int nb1, int n_tokens, int up_gate, b200q_moe_plan_t * p) {
    if (!b200q_gemmq_type(type)) return -1;
    if (m < 1 || k < 256 || k % 256 || n_expert < 1 || n_expert > MOE_MAX_EXPERTS || n_used < 1 || nb1 < 1 || n_used % nb1 || n_tokens < 1) return -2;
    const int64_t n_rows = (int64_t)n_tokens * n_used;
    if (n_rows > (1 << 24) || m > (1 << 24) || k > (1 << 20)) return -2;
    if (up_gate && (m * n_rows) % 4) return -2;                                   // k_mul_unary walks float4
    b200q_layout L; if (b200q_make_layout(type, m, k, &L)) return -1;
    const int bound128 = b200q_moe_tiles_bound((int)n_rows, n_expert, 128);      // the largest bound of any tile width: sizes the table
    if (bound128 > 65535) return -2;                                              // gridDim.y
    p->estride = L.total_bytes; p->n_rows = n_rows; p->nb = moe_choose_nb(n_rows, n_expert);
    p->max_tiles = b200q_moe_tiles_bound((int)n_rows, n_expert, p->nb == 0 ? 128 : 256 * p->nb);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (size_t)b200q_align_up((int64_t)bytes, 256); return o; };
    p->off_xb = take((size_t)n_rows * k * 2);
    p->off_up = up_gate ? take((size_t)n_rows * m * 4) : 0;
    p->off_bounds = take((size_t)(n_expert + 1) * 4);
    p->off_src = take((size_t)n_rows * 4);
    p->off_dst = take((size_t)n_rows * 4);
    p->off_tiles = take((size_t)bound128 * sizeof(b200q_moe_tile));
    p->off_ntiles = take(16);
    p->total = off;
    return 0;
}

int b200q_launch_moe_gemm(const b200q_moe_desc & d, const b200q_moe_plan_t & p, void * ws, cudaStream_t st) {
    char * w = (char *)ws;
    int * bounds = (int *)(w + p.off_bounds), * row_src = (int *)(w + p.off_src), * row_dst = (int *)(w + p.off_dst), * n_tiles = (int *)(w + p.off_ntiles);
    b200q_moe_tile * tiles = (b200q_moe_tile *)(w + p.off_tiles);
    const int bn = p.nb == 0 ? 128 : 256 * p.nb;
    const size_t smem = (size_t)(ROUTE_WARPS * d.n_expert + 3 * (d.n_expert + 1)) * sizeof(int);
    k_moe_route<<<1, 32 * ROUTE_WARPS, smem, st>>>(d.ids, d.n_tokens, d.n_used, d.nb1, d.n_expert, bn, bounds, row_src, row_dst, tiles, n_tiles);
    cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) return (int)e;
    const int64_t total8 = p.n_rows * (d.K / 8);
    int64_t nb = (total8 + 256 * 4 - 1) / (256 * 4); if (nb > 148 * 8) nb = 148 * 8; if (nb < 1) nb = 1;
    k_moe_gather_bf16<<<(unsigned)nb, 256, 0, st>>>(d.x, row_src, (__nv_bfloat16 *)(w + p.off_xb), d.K, p.n_rows);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
    b200q_gemm_grouped g; memset(&g, 0, sizeof g);
    g.type = d.type; g.n_seg = d.W_gate ? 2 : 1; g.M = d.M; g.K = d.K; g.n_expert = d.n_expert; g.estride = p.estride;
    g.xb = w + p.off_xb; g.n_rows = p.n_rows; g.tiles = tiles; g.n_tiles = n_tiles; g.row_dst = row_dst; g.max_tiles = p.max_tiles; g.nb = p.nb;
    float * up = (float *)(w + p.off_up);
    if (d.W_gate) { g.W[0] = d.W; g.dst[0] = up; g.W[1] = d.W_gate; g.dst[1] = d.dst; }      // up -> scratch, gate -> dst, then the unary-mul in place
    else { g.W[0] = d.W; g.dst[0] = d.dst; }
    int rc = b200q_launch_gemm_q_grouped(g, st);
    if (rc || !d.W_gate) return rc;
    return b200q_launch_mul_unary(d.dst, up, d.dst, nullptr, p.n_rows * d.M, d.act, d.limit, st);
}
