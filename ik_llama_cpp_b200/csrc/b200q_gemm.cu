// b200q_gemm.cu — prefill (n_batch > 8) path: tcgen05 / TMEM / TMA GEMM for sm_100a.
//
//   dst[n][m] (f32, ggml layout dst[n*M + m]) = sum_k W[m][k] * X[n][k]
//
// replaces the reference's quantize_mmq_q8_1 + mul_mat_q<type> (mma.sync m16n8k32 s8, ggml-cuda/mmq.cuh:3849-4173)
// and its dequantize + cublasGemmEx fallback (ggml-cuda.cu:1723-1894).
//
// Kernel k_gemm_bf16<BN> (warp-specialised, 192 threads, 1 CTA/SM, one 128 x BN output tile per CTA):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D loads of the A (weights, bf16 [M][K]) and B (activations,
//               bf16 [N][K]) tiles, 128-byte swizzle, into a STAGES-deep smem ring guarded by full/empty mbarriers
//   warp 1      allocates TMEM, then one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16)
//               4x per 64-wide k-block; tcgen05.commit releases the smem stage / signals the epilogue
//   warps 2..5  epilogue: tcgen05.ld 32x32b.x32 (TMEM lane = output feature m, column = token n) -> registers ->
//               coalesced f32 stores (the 32 lanes of a warp hold 32 consecutive m of the same token)
// A comes either from the bf16 scratch written by k_dequant_bf16 (generic types) or ... (fused dequant: see k_gemm_q).
#include "b200q_internal.h"
#include "b200q_moe.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <unordered_map>

namespace {

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void * p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t * bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t * bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t * bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t * bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void * smem_dst, const CUtensorMap * tm, uint64_t * bar, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tm), "r"(smem_u32(bar)), "r"(x), "r"(y) : "memory");
}
// 3-D map {bytes along the row, row, expert}: the expert matrices of a MUL_MAT_ID weight tensor
__device__ __forceinline__ void tma_load_3d(void * smem_dst, const CUtensorMap * tm, uint64_t * bar, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tm), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap * tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tm) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t * smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t * bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile in smem, rows of 64 bf16 = 128 bytes, SWIZZLE_128B, 8-row groups 1024 bytes apart
// (UMMA::SmemDescriptor: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout=SWIZZLE_128B(2) [61,64))
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;                 // LBO (ignored for swizzled K-major), canonical value 1
    d |= (uint64_t)(1024 >> 4) << 32;       // SBO: 8 rows * 128 B
    d |= (uint64_t)1 << 46;                 // descriptor version for sm_100
    d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
    return d;
}
// UMMA::InstrDescriptor for kind::f16: D=f32, A=B=bf16, both K-major, M x N
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

constexpr int BM = 128, BK = 64, UMMA_K = 16;

template <int BN> struct gemm_cfg {
    static constexpr int STAGES = BN == 256 ? 4 : 6;
    static constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr size_t SMEM = 1024 /*align slack*/ + (size_t)STAGES * STAGE_BYTES + 256 /*barriers*/;
};

template <int BN>
__global__ void __launch_bounds__(192, 1)
k_gemm_bf16(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            float * __restrict__ dst, int M, int N, int K, int k_split) {
    using cfg = gemm_cfg<BN>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char * smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t * full_bar  = reinterpret_cast<uint64_t *>(smem + (size_t)cfg::STAGES * cfg::STAGE_BYTES);
    uint64_t * empty_bar = full_bar + cfg::STAGES;
    uint64_t * tmem_full = empty_bar + cfg::STAGES;
    uint32_t * tmem_slot = reinterpret_cast<uint32_t *>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int nk_total = (K + BK - 1) / BK;
    const int nk_per = (nk_total + k_split - 1) / k_split;
    const int kb0 = blockIdx.z * nk_per;
    const int kb1 = min(nk_total, kb0 + nk_per);
    const int nk = kb1 - kb0;                                   // may be <= 0 for trailing splits

    if (threadIdx.x == 0) {
        for (int s = 0; s < cfg::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
    }
    if (warp == 1) tmem_alloc(tmem_slot, BN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < nk; ++i) {
                const int s = i % cfg::STAGES; const uint32_t ph = (i / cfg::STAGES) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                unsigned char * sa = smem + (size_t)s * cfg::STAGE_BYTES; unsigned char * sb = sa + cfg::A_BYTES;
                mbar_expect_tx(&full_bar[s], cfg::STAGE_BYTES);
                tma_load_2d(sa, &tmA, &full_bar[s], (kb0 + i) * BK, m0);
                tma_load_2d(sb, &tmB, &full_bar[s], (kb0 + i) * BK, n0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(BM, BN);
            for (int i = 0; i < nk; ++i) {
                const int s = i % cfg::STAGES; const uint32_t ph = (i / cfg::STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(smem + (size_t)s * cfg::STAGE_BYTES), b_addr = a_addr + cfg::A_BYTES;
                const uint64_t a_desc = make_kmajor_sw128_desc(a_addr), b_desc = make_kmajor_sw128_desc(b_addr);
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    // advance 32 bytes (16 bf16) along K inside the 128-byte swizzle row: +2 in 16-byte units of the start address
                    umma_f16_ss(tmem_base, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (i > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(&empty_bar[s]);               // frees this smem stage when the MMAs have read it
            }
            umma_commit(tmem_full);                       // accumulator complete
        }
    } else {
        // epilogue warps 2..5: TMEM lane quadrant = warp % 4
        const int q = warp & 3;
        if (nk > 0) {
            mbar_wait(tmem_full, 0);
            tc_fence_after();
            const int m = m0 + 32 * q + lane;
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                if (n0 + c0 >= N) break;                  // warp-uniform
                uint32_t r[32];
                tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, r);
                tmem_ld_wait();
                if (m < M) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + c0 + j;
                        if (n < N) {
                            float * p = dst + (size_t)n * M + m;
                            if (k_split > 1) atomicAdd(p, __uint_as_float(r[j])); else *p = __uint_as_float(r[j]);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, BN);
}

// ---------------------------------------------------------------------------------------------------------------
// Fused prefill kernel: the A operand is dequantised INSIDE the kernel (no bf16 weight scratch in HBM).
//   warp 0      TMA producer: (a) packed weight planes of a 128-row x 256-weight block (low-bit plane 128 B/row with
//               SWIZZLE_128B, scale/meta plane 16 B/row) into a 2-deep RAW ring, (b) bf16 activation tiles into the B ring
//   warp 1      MMA issuer (tcgen05.mma kind::f16, M=128, N=BN, K=16), A and B from shared memory
//   warps 2..5  thread = one weight row: canonical decode (PRMT-LUT / mask) of 2 items per 64-wide k-block ->
//               bf16(dl*q - ml) -> the 128-byte K-major SWIZZLE_128B row of the A stage; after the main loop the same
//               warps run the epilogue (their warp%4 is their TMEM lane quadrant)
// Pipelines: raw_full/raw_empty (TMA <-> dequant), a_full/a_empty (dequant <-> MMA), b_full/b_empty (TMA <-> MMA),
// tmem_full (MMA -> epilogue).  Generic-proxy smem writes of the dequant warps are published to the tensor core with
// fence.proxy.async before the a_full arrive.
// ---------------------------------------------------------------------------------------------------------------
constexpr int RAW_K = 256;                       // weights per row per raw stage (= 8 items, 4 MMA k-blocks)
constexpr int DQ_WARPS = 8;                      // dequant / epilogue warps (warps 2..9)

// bytes per 256 weights of the planes after the 128-byte low-bit plane (every one a multiple of 16: the inner box of a TMA map)
template <int TYPE> struct gemmq_planes { static constexpr int P1 = 16, P2 = 0; };                    // IQ4_NL / Q4_0 (8 halfs), Q4_K, IQ4_K
template <> struct gemmq_planes<B200Q_TYPE_Q4_1>  { static constexpr int P1 = 32, P2 = 0; };          // {d,m} per item
template <> struct gemmq_planes<B200Q_TYPE_Q5_0>  { static constexpr int P1 = 32, P2 = 16; };         // qh | d
template <> struct gemmq_planes<B200Q_TYPE_Q5_1>  { static constexpr int P1 = 32, P2 = 32; };         // qh | {d,m}
template <> struct gemmq_planes<B200Q_TYPE_Q5_K>  { static constexpr int P1 = 32, P2 = 16; };         // qh | {d,dmin,scales}
template <> struct gemmq_planes<B200Q_TYPE_IQ5_K> { static constexpr int P1 = 32, P2 = 16; };         // qh | {d,extra,scales}
// NB = number of 256-column accumulators (BN = 256*NB), or BN = 128 when NB == 0
template <int TYPE, int NB> struct gemmq_cfg {
    static constexpr int BN = NB == 0 ? 128 : 256 * NB;
    static constexpr int A_STAGES = 3, B_STAGES = NB == 2 ? 2 : 3, RAW_STAGES = 2;
    static constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
    static constexpr int P1 = gemmq_planes<TYPE>::P1, P2 = gemmq_planes<TYPE>::P2;
    static constexpr int RAW_P0 = BM * 128, RAW_P1 = BM * P1, RAW_P2 = BM * P2, RAW_BYTES = RAW_P0 + RAW_P1 + RAW_P2;     // low-bit plane | high bits / meta | meta
    static constexpr int TMEM_COLS = BN;
    static constexpr size_t SMEM = 1024 + (size_t)A_STAGES * A_BYTES + (size_t)B_STAGES * B_BYTES + (size_t)RAW_STAGES * RAW_BYTES + 256;
    static_assert(SMEM <= 227 * 1024, "k_gemm_q: shared memory");
};

// Up to GEMMQ_MAX_SEGS weight tensors that share the activation tile (Q,K,V: the reference's look-ahead fusion,
// ggml-cuda.cu:2573-2601) are covered by ONE launch: blockIdx.x walks the concatenated 128-row tiles of all segments.
// Epilogue options per segment (only with k_split == 1): mul != nullptr -> dst = act(clamp(acc)) * clamp(mul[n][m])
// (the gate half of GGML_OP_FUSED_UP_GATE for n > 8, ggml-cuda.cu:3588-3618), dst_bf != nullptr -> bf16 copy of dst
// (the activation operand of the next MUL_MAT, saves its f32 -> bf16 pass).
constexpr int GEMMQ_MAX_SEGS = 3;
struct gemmq_seg { float * dst; const float * mul; __nv_bfloat16 * dst_bf; int M; int tile0; };
struct gemmq_args {
    CUtensorMap tmP0[GEMMQ_MAX_SEGS], tmP1[GEMMQ_MAX_SEGS], tmP2[GEMMQ_MAX_SEGS], tmB;
    gemmq_seg seg[GEMMQ_MAX_SEGS];
    int n_seg, N, K, k_split, act; float limit;
};
// grouped mode (MoE prefill, b200q_moe.cu): tmP* are 3-D maps {row bytes, M, n_expert}, tmB covers the expert-sorted bf16 activations
// [n_rows][K]; blockIdx.y indexes the tile table, tiles at or beyond *n_tiles exit at once; column c of a tile is stored at output row
// row_dst[col0 + c] of seg.dst.  Always k_split == 1: no memset, no atomics, every output is written exactly once.
struct gemmq_gargs : gemmq_args {
    const b200q_moe_tile * tiles; const int * n_tiles; const int * row_dst;
};

// carry-less per-byte add of two packed int8x4 (the A/B halves of the sign-fill LUT)
__device__ __forceinline__ uint32_t vadd4_wrap(uint32_t a, uint32_t b) {
    return ((a & 0x7f7f7f7fu) + (b & 0x7f7f7f7fu)) ^ ((a ^ b) & 0x80808080u);
}
// signed int8 lane J of a word already XOR-ed with 0x80808080 (biased by +128) -> float(v), exact:
// place the byte under the exponent of 2^23 and subtract 2^23 + 128
template <int J> __device__ __forceinline__ float biased_byte_to_float(uint32_t wb) {
    const uint32_t bits = __byte_perm(wb, 0x4B000000u, 0x7650 + J);       // {byte J, 0x00, 0x00, 0x4B}
    return __uint_as_float(bits) - 8388736.0f;
}

// Fused prefill kernel: the A operand is dequantised INSIDE the kernel (no bf16 weight scratch in HBM).
//   warp 0      TMA producer: (a) packed weight planes of a 128-row x 256-weight block (low-bit plane 128 B/row with
//               SWIZZLE_128B, scale/meta plane 16 B/row) into a 2-deep RAW ring, (b) bf16 activation tiles into the B ring
//   warp 1      MMA issuer: tcgen05.mma kind::f16, M=128, N=256 (or 128), K=16; with NB=2 the SAME dequantised A stage feeds two
//               accumulators (512 TMEM columns = 512 tokens), so every weight is decoded once per 512 tokens
//   warps 2..9  thread = (weight row, 32-weight item): canonical decode (PRMT-LUT / mask) -> exact int8->f32 via the 2^23
//               exponent trick -> bf16(dl*q - ml) -> its 64 bytes of the 128-byte K-major SWIZZLE_128B row of the A stage;
//               after the main loop the same warps run the epilogue (warp%4 = TMEM lane quadrant, warp/4 = column half)
// Pipelines: raw_full/raw_empty (TMA <-> dequant), a_full/a_empty (dequant <-> MMA), b_full/b_empty (TMA <-> MMA),
// tmem_full (MMA -> epilogue).  Generic-proxy smem writes of the dequant warps are published to the tensor core with
// fence.proxy.async before the a_full arrive.
template <int TYPE, int NB, bool GROUPED = false>
__global__ void __launch_bounds__(64 + 32 * DQ_WARPS, 1)
k_gemm_q(const __grid_constant__ std::conditional_t<GROUPED, gemmq_gargs, gemmq_args> a) {
    using cfg = gemmq_cfg<TYPE, NB>;
    int ex = 0, n_cols = 0;                                     // grouped: expert and valid columns of this tile
    int n0 = blockIdx.y * cfg::BN;
    if constexpr (GROUPED) {
        if ((int)blockIdx.y >= __ldg(a.n_tiles)) return;        // beyond the routed tiles: leave before any barrier or TMEM allocation
        const int4 tl = __ldg(reinterpret_cast<const int4 *>(a.tiles) + blockIdx.y);
        ex = tl.x; n0 = tl.y; n_cols = tl.z - tl.y;
    }
    int sg = 0;
#pragma unroll
    for (int s = 1; s < GEMMQ_MAX_SEGS; ++s) if (s < a.n_seg && (int)blockIdx.x >= a.seg[s].tile0) sg = s;
    const CUtensorMap * tmP0 = &a.tmP0[sg], * tmP1 = &a.tmP1[sg], * tmP2 = &a.tmP2[sg], * tmB = &a.tmB;
    float * __restrict__ dst = a.seg[sg].dst; const float * __restrict__ mul = a.seg[sg].mul; __nv_bfloat16 * __restrict__ dst_bf = a.seg[sg].dst_bf;
    const int M = a.seg[sg].M, N = a.N, K = a.K, k_split = a.k_split;
    constexpr int BN = cfg::BN;
    constexpr int MMA_N = NB == 0 ? 128 : 256;
    constexpr int N_ACC = NB == 0 ? 1 : NB;
    extern __shared__ unsigned char smem_raw[];
    unsigned char * smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char * sA = smem;
    unsigned char * sB = sA + (size_t)cfg::A_STAGES * cfg::A_BYTES;
    unsigned char * sR = sB + (size_t)cfg::B_STAGES * cfg::B_BYTES;
    uint64_t * bars = reinterpret_cast<uint64_t *>(sR + (size_t)cfg::RAW_STAGES * cfg::RAW_BYTES);
    uint64_t * a_full = bars, * a_empty = a_full + cfg::A_STAGES, * b_full = a_empty + cfg::A_STAGES, * b_empty = b_full + cfg::B_STAGES;
    uint64_t * raw_full = b_empty + cfg::B_STAGES, * raw_empty = raw_full + cfg::RAW_STAGES, * tmem_full = raw_empty + cfg::RAW_STAGES;
    uint32_t * tmem_slot = reinterpret_cast<uint32_t *>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = ((int)blockIdx.x - a.seg[sg].tile0) * BM;
    // K is walked in raw blocks of 256 weights; split-K over blockIdx.z in units of raw blocks
    const int nr_total = (K + RAW_K - 1) / RAW_K;
    const int nr_per = (nr_total + k_split - 1) / k_split;
    const int rb0 = blockIdx.z * nr_per, rb1 = min(nr_total, rb0 + nr_per);
    const int nr = rb1 - rb0;                                   // raw blocks of this CTA (may be <= 0)
    const int kb_begin = rb0 * (RAW_K / BK);
    const int kb_end = min((K + BK - 1) / BK, rb1 * (RAW_K / BK));
    const int nk = kb_end - kb_begin;                           // 64-wide MMA k-blocks of this CTA

    if (threadIdx.x == 0) {
        for (int s = 0; s < cfg::A_STAGES; ++s) { mbar_init(&a_full[s], DQ_WARPS); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < cfg::B_STAGES; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < cfg::RAW_STAGES; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], DQ_WARPS); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
        tma_prefetch_desc(tmP0); tma_prefetch_desc(tmP1); if (cfg::P2) tma_prefetch_desc(tmP2); tma_prefetch_desc(tmB);
    }
    if (warp == 1) tmem_alloc(tmem_slot, cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int ib = 0;
            for (int r = 0; r < nr; ++r) {
                const int rs = r % cfg::RAW_STAGES; const uint32_t rph = (r / cfg::RAW_STAGES) & 1;
                mbar_wait(&raw_empty[rs], rph ^ 1);
                unsigned char * raw = sR + (size_t)rs * cfg::RAW_BYTES;
                mbar_expect_tx(&raw_full[rs], cfg::RAW_BYTES);
                if constexpr (GROUPED) {
                    tma_load_3d(raw, tmP0, &raw_full[rs], (rb0 + r) * 128, m0, ex);
                    tma_load_3d(raw + cfg::RAW_P0, tmP1, &raw_full[rs], (rb0 + r) * cfg::P1, m0, ex);
                    if (cfg::P2) tma_load_3d(raw + cfg::RAW_P0 + cfg::RAW_P1, tmP2, &raw_full[rs], (rb0 + r) * cfg::P2, m0, ex);
                } else {
                tma_load_2d(raw, tmP0, &raw_full[rs], (rb0 + r) * 128, m0);                // bytes along the row
                tma_load_2d(raw + cfg::RAW_P0, tmP1, &raw_full[rs], (rb0 + r) * cfg::P1, m0);
                if (cfg::P2) tma_load_2d(raw + cfg::RAW_P0 + cfg::RAW_P1, tmP2, &raw_full[rs], (rb0 + r) * cfg::P2, m0);
                }
                for (int q = 0; q < RAW_K / BK && ib < nk; ++q, ++ib) {
                    const int s = ib % cfg::B_STAGES; const uint32_t ph = (ib / cfg::B_STAGES) & 1;
                    mbar_wait(&b_empty[s], ph ^ 1);
                    mbar_expect_tx(&b_full[s], cfg::B_BYTES);
#pragma unroll
                    for (int j = 0; j < N_ACC; ++j)
                        tma_load_2d(sB + (size_t)s * cfg::B_BYTES + (size_t)j * MMA_N * BK * 2, tmB, &b_full[s], (kb_begin + ib) * BK, n0 + j * MMA_N);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(BM, MMA_N);
            for (int i = 0; i < nk; ++i) {
                const int sa = i % cfg::A_STAGES; const uint32_t pa = (i / cfg::A_STAGES) & 1;
                const int sb = i % cfg::B_STAGES; const uint32_t pb = (i / cfg::B_STAGES) & 1;
                mbar_wait(&a_full[sa], pa);
                mbar_wait(&b_full[sb], pb);
                tc_fence_after();
                const uint64_t a_desc = make_kmajor_sw128_desc(smem_u32(sA + (size_t)sa * cfg::A_BYTES));
#pragma unroll
                for (int j = 0; j < N_ACC; ++j) {
                    const uint64_t b_desc = make_kmajor_sw128_desc(smem_u32(sB + (size_t)sb * cfg::B_BYTES + (size_t)j * MMA_N * BK * 2));
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)
                        umma_f16_ss(tmem_base + (uint32_t)(j * MMA_N), a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (i > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(&a_empty[sa]);
                umma_commit(&b_empty[sb]);
            }
            umma_commit(tmem_full);
        }
    } else {
        // ---------------- dequant warps (then epilogue): thread = (row, item half) ----------------
        const int dq = warp - 2;                                  // 0..7
        const int q4 = warp & 3;                                  // TMEM lane quadrant of this warp (hardware rule: warp % 4)
        const int half = dq >> 2;                                 // which 32-weight item of each 64-wide k-block / which column half in the epilogue
        const int row = 32 * q4 + lane;                           // row of the tile owned by this thread
        const b200q_kv4 T = b200q_kv4_init();
        int ia = 0;
        for (int r = 0; r < nr; ++r) {
            const int rs = r % cfg::RAW_STAGES; const uint32_t rph = (r / cfg::RAW_STAGES) & 1;
            mbar_wait(&raw_full[rs], rph);
            const unsigned char * raw = sR + (size_t)rs * cfg::RAW_BYTES;
            b200q_planes SP; SP.p[0] = raw; SP.p[1] = raw + cfg::RAW_P0; SP.p[2] = raw + cfg::RAW_P0 + cfg::RAW_P1; SP.p[3] = SP.p[4] = nullptr; SP.n32 = 8; SP.nb = 1;
            for (int q = 0; q < RAW_K / BK && ia < nk; ++q, ++ia) {
                const int sa = ia % cfg::A_STAGES; const uint32_t pa = (ia / cfg::A_STAGES) & 1;
                // decode before waiting for the A slot: the raw data is already there
                const int it = 2 * q + half;
                b200q_item I; b200q_canon C;
                b200q_load_item<TYPE, b200q_ld_plain, false, int, true>(I, SP, row, it);
                b200q_decode_item<TYPE>(I, it, C, T);
                uint32_t o[16];
#pragma unroll
                for (int w = 0; w < 8; ++w) {                     // word w = weights 4w..4w+3
                    uint32_t v = (uint32_t)C.va[w];
                    if (b200q_traits<TYPE>::HAS_B) v = vadd4_wrap(v, (uint32_t)C.vb[w]);
                    v ^= 0x80808080u;                             // bias +128 -> unsigned bytes
                    const float dl = C.dl[w / 4], ml = C.ml[w / 4];
                    const float f0 = fmaf(biased_byte_to_float<0>(v), dl, -ml), f1 = fmaf(biased_byte_to_float<1>(v), dl, -ml);
                    const float f2 = fmaf(biased_byte_to_float<2>(v), dl, -ml), f3 = fmaf(biased_byte_to_float<3>(v), dl, -ml);
                    __nv_bfloat162 b01 = __floats2bfloat162_rn(f0, f1), b23 = __floats2bfloat162_rn(f2, f3);
                    o[2 * w] = *reinterpret_cast<uint32_t *>(&b01); o[2 * w + 1] = *reinterpret_cast<uint32_t *>(&b23);
                }
                mbar_wait(&a_empty[sa], pa ^ 1);
                unsigned char * arow = sA + (size_t)sa * cfg::A_BYTES + (size_t)(row >> 3) * 1024 + (size_t)(row & 7) * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int chunk = (4 * half + c) ^ (row & 7);
                    *reinterpret_cast<uint4 *>(arow + chunk * 16) = make_uint4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
                }
                fence_proxy_async();                              // make the generic-proxy writes visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[sa]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&raw_empty[rs]);
        }
        // ---------------- epilogue: quadrant q4, column half `half` ----------------
        if constexpr (GROUPED) {
            // columns past n_cols belong to the next expert or lie beyond n_rows: masked.  Lane j fetches the output row of column
            // c0 + j once; the warp's 32 lanes (consecutive m) then store each column coalesced along M.
            if (nk > 0) {
                mbar_wait(tmem_full, 0);
                tc_fence_after();
                const int m = m0 + row;
                constexpr int COLS_PER = BN / 2;
                const int c_begin = half * COLS_PER, c_end = min((half + 1) * COLS_PER, n_cols);
                const bool mrow = m < M;
#pragma unroll 1
                for (int c0 = c_begin; c0 < c_end; c0 += 32) {
                    uint32_t rr[32];
                    tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q4) << 16) + (uint32_t)c0, rr);
                    const int rd = c0 + lane < c_end ? __ldg(a.row_dst + n0 + c0 + lane) : 0;
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int r = __shfl_sync(0xffffffffu, rd, j);
                        if (mrow && c0 + j < c_end) dst[(size_t)r * M + m] = __uint_as_float(rr[j]);
                    }
                }
            }
        } else
        if (nk > 0) {
            mbar_wait(tmem_full, 0);
            tc_fence_after();
            const int m = m0 + row;
            constexpr int COLS_PER = BN / 2;
            const int c_begin = half * COLS_PER, c_end = min((half + 1) * COLS_PER, N - n0);
            const bool mrow = m < M;
            if (k_split > 1 || (mul == nullptr && dst_bf == nullptr)) {
#pragma unroll 1
                for (int c0 = c_begin; c0 < c_end; c0 += 32) {
                    uint32_t rr[32];
                    tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q4) << 16) + (uint32_t)c0, rr);
                    tmem_ld_wait();
                    if (mrow) {
                        if (k_split > 1) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) { const int n = n0 + c0 + j; if (n < N) atomicAdd(dst + (size_t)n * M + m, __uint_as_float(rr[j])); }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) { const int n = n0 + c0 + j; if (n < N) dst[(size_t)n * M + m] = __uint_as_float(rr[j]); }
                        }
                    }
                }
            } else {
                // fused unary-mul (+ bf16 copy): the `mul` operand of chunk c+1 is fetched (32 loads in flight per thread) while
                // chunk c is computed, so the L2 latency hides behind the activation math
                const float lim = a.limit; const int act = a.act;
                float u[32], un[32];
                auto fetch = [&](float (&dstu)[32], int c0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) { const int n = n0 + c0 + j; dstu[j] = (mul != nullptr && mrow && c0 < c_end && n < N) ? __ldg(mul + (size_t)n * M + m) : 1.0f; }
                };
                auto finish = [&](const uint32_t (&rr)[32], const float (&uu)[32], int c0) {
                    if (!mrow) return;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + c0 + j;
                        if (n < N) {
                            float v = __uint_as_float(rr[j]);
                            if (mul != nullptr) v = b200q_glu<true>(act, v, uu[j], lim);
                            dst[(size_t)n * M + m] = v;
                            if (dst_bf != nullptr) dst_bf[(size_t)n * M + m] = __float2bfloat16_rn(v);
                        }
                    }
                };
                fetch(u, c_begin);
#pragma unroll 1
                for (int c0 = c_begin; c0 < c_end; c0 += 64) {
                    uint32_t rr[32];
                    tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q4) << 16) + (uint32_t)c0, rr);
                    fetch(un, c0 + 32);
                    tmem_ld_wait();
                    finish(rr, u, c0);
                    if (c0 + 32 < c_end) {
                        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q4) << 16) + (uint32_t)(c0 + 32), rr);
                        fetch(u, c0 + 64);
                        tmem_ld_wait();
                        finish(rr, un, c0 + 32);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, cfg::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------------------------
// Ternary prefill on the INT8 tensor pipe: IQ2_BN (bitnet b1.58) weights x per-token int8 activations -> s32 in TMEM.
// (BASELINE config 4 / north_star "IQ*_BN ternary (int8 tcgen05)".  The reference has no integer tensor-core path for this type: its prefill is
//  dequantize_block_iq2_bn + cublasGemmEx in f16 with f16 accumulation, ggml-cuda.cu:1723-1894, SURVEY §8 a13.)
//   A: the 2-bit fields q in {0,1,2} of the wire blocks are expanded to UNSIGNED int8 in the K-major SWIZZLE_128B A stage (128 rows x 128 k
//      = 128 bytes per row: one shift + mask per 4 weights, no table, no scale); w = rs * (q - 1) is applied in the epilogue:
//      dst[n][m] = rs[m] * ts[n] * (acc[m][n] - S[n]),  acc = sum_k q[m][k] * xq[n][k]  (tcgen05.mma kind::i8, u8 x s8 -> s32, exact),
//      S[n] = sum_k xq[n][k] and ts[n] = amax_n / 127 come from the activation quantiser (k_quantize_rows_i8).
//   B: int8 activations [N][K], TMA (SWIZZLE_128B, 128 k = 128 bytes per row), one per-TOKEN scale: the whole K reduction is integer.
//   Zero-filled TMA tails make any K % 64 == 0 work (bitnet: K = 3200, 8640): q = 0 and xq = 0 beyond K contribute nothing, S[n] covers real k only.
// Same warp roles / pipelines as k_gemm_q; MMA K = 32 per instruction, 4 instructions per 128-byte k-block; 2 x 256 TMEM columns for 512 tokens.
// Accuracy: activations rounded to 8 bits per token (NMSE ~1e-4 for Gaussian activations; the reference's own q8_1 decode path: ~2e-5, its f16-accumulate
// prefill: ~1e-6 + f16 overflow risk); weights exact.  Tolerance in tests/test_gpu_parity.py: NMSE <= 5e-4 (the reference's test bar).
// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N) {        // D = s32 (2 << 4), A = u8 (0 << 7), B = s8 (1 << 10), K-major both
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_i8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
constexpr int BNI_BK = 128;                      // k (= bytes) per A / B stage row
constexpr int BNI_RAW_K = 512;                   // weights per row per raw stage: 128 bytes of 2-bit fields = 4 k-blocks
template <int NB> struct gemmbn_cfg {
    static constexpr int BN = NB == 0 ? 128 : 256 * NB;
    static constexpr int A_STAGES = 3, B_STAGES = 2, RAW_STAGES = 2;
    static constexpr int A_BYTES = BM * BNI_BK, B_BYTES = BN * BNI_BK, RAW_BYTES = BM * 128;
    static constexpr int TMEM_COLS = BN;
    static constexpr size_t SMEM = 1024 + (size_t)A_STAGES * A_BYTES + (size_t)B_STAGES * B_BYTES + (size_t)RAW_STAGES * RAW_BYTES + 256;
};
struct gemmbn_seg { float * dst; const float * rs; int M; int tile0; };
struct gemmbn_args {
    CUtensorMap tmP0[GEMMQ_MAX_SEGS], tmB;
    gemmbn_seg seg[GEMMQ_MAX_SEGS];
    const float * ts; const int * sx;            // per-token scale and integer sum of the quantised activations
    int n_seg, N, K;
};
template <int NB>
__global__ void __launch_bounds__(64 + 32 * DQ_WARPS, 1)
k_gemm_bn_i8(const __grid_constant__ gemmbn_args a) {
    using cfg = gemmbn_cfg<NB>;
    int sg = 0;
#pragma unroll
    for (int s = 1; s < GEMMQ_MAX_SEGS; ++s) if (s < a.n_seg && (int)blockIdx.x >= a.seg[s].tile0) sg = s;
    const CUtensorMap * tmP0 = &a.tmP0[sg], * tmB = &a.tmB;
    float * __restrict__ dst = a.seg[sg].dst; const float * __restrict__ rs = a.seg[sg].rs;
    const int M = a.seg[sg].M, N = a.N, K = a.K;
    constexpr int BN = cfg::BN, MMA_N = NB == 0 ? 128 : 256, N_ACC = NB == 0 ? 1 : NB;
    extern __shared__ unsigned char smem_raw[];
    unsigned char * smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char * sA = smem;
    unsigned char * sB = sA + (size_t)cfg::A_STAGES * cfg::A_BYTES;
    unsigned char * sR = sB + (size_t)cfg::B_STAGES * cfg::B_BYTES;
    uint64_t * bars = reinterpret_cast<uint64_t *>(sR + (size_t)cfg::RAW_STAGES * cfg::RAW_BYTES);
    uint64_t * a_full = bars, * a_empty = a_full + cfg::A_STAGES, * b_full = a_empty + cfg::A_STAGES, * b_empty = b_full + cfg::B_STAGES;
    uint64_t * raw_full = b_empty + cfg::B_STAGES, * raw_empty = raw_full + cfg::RAW_STAGES, * tmem_full = raw_empty + cfg::RAW_STAGES;
    uint32_t * tmem_slot = reinterpret_cast<uint32_t *>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = ((int)blockIdx.x - a.seg[sg].tile0) * BM, n0 = blockIdx.y * BN;
    const int nr = (K + BNI_RAW_K - 1) / BNI_RAW_K;             // raw blocks of 512 weights
    const int nk = (K + BNI_BK - 1) / BNI_BK;                   // 128-wide MMA k-blocks

    if (threadIdx.x == 0) {
        for (int s = 0; s < cfg::A_STAGES; ++s) { mbar_init(&a_full[s], DQ_WARPS); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < cfg::B_STAGES; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < cfg::RAW_STAGES; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], DQ_WARPS); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
        tma_prefetch_desc(tmP0); tma_prefetch_desc(tmB);
    }
    if (warp == 1) tmem_alloc(tmem_slot, cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int ib = 0;
            for (int r = 0; r < nr; ++r) {
                const int rsi = r % cfg::RAW_STAGES; const uint32_t rph = (r / cfg::RAW_STAGES) & 1;
                mbar_wait(&raw_empty[rsi], rph ^ 1);
                mbar_expect_tx(&raw_full[rsi], cfg::RAW_BYTES);
                tma_load_2d(sR + (size_t)rsi * cfg::RAW_BYTES, tmP0, &raw_full[rsi], r * 128, m0);       // 128 bytes of 2-bit fields per row
                for (int q = 0; q < BNI_RAW_K / BNI_BK && ib < nk; ++q, ++ib) {
                    const int s = ib % cfg::B_STAGES; const uint32_t ph = (ib / cfg::B_STAGES) & 1;
                    mbar_wait(&b_empty[s], ph ^ 1);
                    mbar_expect_tx(&b_full[s], cfg::B_BYTES);
#pragma unroll
                    for (int j = 0; j < N_ACC; ++j)
                        tma_load_2d(sB + (size_t)s * cfg::B_BYTES + (size_t)j * MMA_N * BNI_BK, tmB, &b_full[s], ib * BNI_BK, n0 + j * MMA_N);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_i8(BM, MMA_N);
            for (int i = 0; i < nk; ++i) {
                const int sa = i % cfg::A_STAGES; const uint32_t pa = (i / cfg::A_STAGES) & 1;
                const int sb = i % cfg::B_STAGES; const uint32_t pb = (i / cfg::B_STAGES) & 1;
                mbar_wait(&a_full[sa], pa);
                mbar_wait(&b_full[sb], pb);
                tc_fence_after();
                const uint64_t a_desc = make_kmajor_sw128_desc(smem_u32(sA + (size_t)sa * cfg::A_BYTES));
#pragma unroll
                for (int j = 0; j < N_ACC; ++j) {
                    const uint64_t b_desc = make_kmajor_sw128_desc(smem_u32(sB + (size_t)sb * cfg::B_BYTES + (size_t)j * MMA_N * BNI_BK));
#pragma unroll
                    for (int k = 0; k < BNI_BK / 32; ++k)        // K = 32 int8 = 32 bytes per instruction: +2 in 16-byte units of the start address
                        umma_i8_ss(tmem_base + (uint32_t)(j * MMA_N), a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (i > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(&a_empty[sa]);
                umma_commit(&b_empty[sb]);
            }
            umma_commit(tmem_full);
        }
    } else {
        // ---------------- expand warps (then epilogue): thread = (row, wire block of the k-block) ----------------
        const int dq = warp - 2, q4 = warp & 3, half = dq >> 2, row = 32 * q4 + lane;
        int ia = 0;
        for (int r = 0; r < nr; ++r) {
            const int rsi = r % cfg::RAW_STAGES; const uint32_t rph = (r / cfg::RAW_STAGES) & 1;
            mbar_wait(&raw_full[rsi], rph);
            const unsigned char * raw = sR + (size_t)rsi * cfg::RAW_BYTES + (size_t)row * 128;
            for (int q = 0; q < BNI_RAW_K / BNI_BK && ia < nk; ++q, ++ia) {
                const int sa = ia % cfg::A_STAGES; const uint32_t pa = (ia / cfg::A_STAGES) & 1;
                // wire block (64 weights, 16 bytes) number 2q + half of this raw row; SWIZZLE_128B: 16-byte chunk c sits at c ^ (row & 7)
                const uint4 wv = *reinterpret_cast<const uint4 *>(raw + (((2 * q + half) ^ (row & 7)) << 4));
                const uint32_t w[4] = {wv.x, wv.y, wv.z, wv.w};
                mbar_wait(&a_empty[sa], pa ^ 1);
                unsigned char * arow = sA + (size_t)sa * cfg::A_BYTES + (size_t)(row >> 3) * 1024 + (size_t)(row & 7) * 128;
#pragma unroll
                for (int f = 0; f < 4; ++f) {                    // field f of byte j = weight 16 f + j of the block: one 16-byte chunk of 16 consecutive k
                    const int chunk = (4 * half + f) ^ (row & 7);
                    *reinterpret_cast<uint4 *>(arow + chunk * 16) = make_uint4((w[0] >> (2 * f)) & 0x03030303u, (w[1] >> (2 * f)) & 0x03030303u,
                                                                               (w[2] >> (2 * f)) & 0x03030303u, (w[3] >> (2 * f)) & 0x03030303u);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[sa]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&raw_empty[rsi]);
        }
        // ---------------- epilogue: dst = rs[m] * ts[n] * (acc - S[n]) ----------------
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int m = m0 + row;
        constexpr int COLS_PER = BN / 2;
        const int c_begin = half * COLS_PER, c_end = min((half + 1) * COLS_PER, N - n0);
        const bool mrow = m < M;
        const float rsm = mrow ? __ldg(rs + m) : 0.0f;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            uint32_t rr[32];
            tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q4) << 16) + (uint32_t)c0, rr);
            tmem_ld_wait();
            if (mrow) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int n = n0 + c0 + j;
                    if (n < N) dst[(size_t)n * M + m] = rsm * __ldg(a.ts + n) * (float)((int)rr[j] - __ldg(a.sx + n));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, cfg::TMEM_COLS);
}

// f32 [N][K] (row stride xs) -> int8 [N][K] with ONE scale per token: q = rint(x * 127 / amax_n); ts[n] = amax_n / 127; sx[n] = sum_k q
__global__ void __launch_bounds__(256) k_quantize_rows_i8(const float * __restrict__ x, int64_t xs, int8_t * __restrict__ q, float * __restrict__ ts, int * __restrict__ sx, int64_t K) {
    const int64_t n = blockIdx.x; const float * xr = x + n * xs; int8_t * qr = q + n * K;
    __shared__ float s_amax[8]; __shared__ int s_sum[8];
    float amax = 0.0f;
    for (int64_t k = threadIdx.x * 4; k < K; k += blockDim.x * 4) { const float4 v = *reinterpret_cast<const float4 *>(xr + k); amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)))); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if ((threadIdx.x & 31) == 0) s_amax[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = s_amax[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) amax = fmaxf(amax, s_amax[i]);
    const float d = __fdiv_rn(amax, 127.0f), inv = d > 0.0f ? __frcp_rn(d) : 0.0f;
    int sum = 0;
    for (int64_t k = threadIdx.x * 4; k < K; k += blockDim.x * 4) {
        const float4 v = *reinterpret_cast<const float4 *>(xr + k);
        const int a = max(-127, min(127, __float2int_rn(v.x * inv))), b = max(-127, min(127, __float2int_rn(v.y * inv)));
        const int c = max(-127, min(127, __float2int_rn(v.z * inv))), e = max(-127, min(127, __float2int_rn(v.w * inv)));
        sum += a + b + c + e;
        *reinterpret_cast<uint32_t *>(qr + k) = (uint32_t)(a & 0xff) | ((uint32_t)(b & 0xff) << 8) | ((uint32_t)(c & 0xff) << 16) | ((uint32_t)(e & 0xff) << 24);
    }
    sum = __reduce_add_sync(0xffffffffu, sum);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int i = 0; i < 8; ++i) t += s_sum[i]; sx[n] = t; ts[n] = d; }
}

// dst = act(clamp(gate)) * clamp(up) elementwise (the reference's ggml_fused_mul_unary after two MMQs, ggml-cuda.cu:3588-3618);
// gate may alias dst; optional bf16 copy for the following MUL_MAT
__global__ void k_mul_unary(const float * gate /* may alias dst: no __restrict__ */, const float * __restrict__ up, float * dst, __nv_bfloat16 * __restrict__ dst_bf,
                            int64_t total4, int act, float lim) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 g = reinterpret_cast<const float4 *>(gate)[i]; float4 u = reinterpret_cast<const float4 *>(up)[i];
        float4 r; r.x = b200q_glu<true>(act, g.x, u.x, lim); r.y = b200q_glu<true>(act, g.y, u.y, lim); r.z = b200q_glu<true>(act, g.z, u.z, lim); r.w = b200q_glu<true>(act, g.w, u.w, lim);
        reinterpret_cast<float4 *>(dst)[i] = r;
        if (dst_bf != nullptr) {
            __nv_bfloat162 b0 = __floats2bfloat162_rn(r.x, r.y), b1 = __floats2bfloat162_rn(r.z, r.w);
            uint2 o; o.x = *reinterpret_cast<uint32_t *>(&b0); o.y = *reinterpret_cast<uint32_t *>(&b1);
            reinterpret_cast<uint2 *>(dst_bf)[i] = o;
        }
    }
}

// f32 [N][K] (row stride xs) -> bf16 [N][K].  HBM-bound glue between the GEMMs (12 MB per 512 x 4096 activation): a thread converts 8 consecutive
// values (two LDG.128 -> one STG.128) and keeps U such groups in flight; round 1's one-float4-per-thread version ran at ~1 TB/s (11.8 us per call,
// profiles/r1_pp_breakdown.txt) and cost 10 % of the prefill layer.
__global__ void __launch_bounds__(256) k_f32_to_bf16(const float * __restrict__ x, int64_t xs, __nv_bfloat16 * __restrict__ out, int64_t K, int64_t N) {
    constexpr int U = 4;
    const int64_t k8 = K / 8, total8 = N * k8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < total8; i0 += U * stride) {
        float4 a[U], b[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i < total8) { const int64_t n = i / k8, c = i % k8; const float4 * p = reinterpret_cast<const float4 *>(x + n * xs + 8 * c); a[u] = __ldg(p); b[u] = __ldg(p + 1); }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i < total8) {
                __nv_bfloat162 p0 = __floats2bfloat162_rn(a[u].x, a[u].y), p1 = __floats2bfloat162_rn(a[u].z, a[u].w), p2 = __floats2bfloat162_rn(b[u].x, b[u].y), p3 = __floats2bfloat162_rn(b[u].z, b[u].w);
                uint4 o; o.x = *reinterpret_cast<uint32_t *>(&p0); o.y = *reinterpret_cast<uint32_t *>(&p1); o.z = *reinterpret_cast<uint32_t *>(&p2); o.w = *reinterpret_cast<uint32_t *>(&p3);
                const int64_t n = i / k8, c = i % k8;
                *reinterpret_cast<uint4 *>(out + n * K + 8 * c) = o;
            }
        }
    }
}
// K % 8 != 0 (K % 4 == 0): the simple version
__global__ void k_f32_to_bf16_k4(const float * __restrict__ x, int64_t xs, __nv_bfloat16 * __restrict__ out, int64_t K, int64_t N) {
    const int64_t total4 = N * (K / 4);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = i / (K / 4), k4 = i % (K / 4);
        const float4 v = *reinterpret_cast<const float4 *>(x + n * xs + 4 * k4);
        __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        uint2 u; u.x = *reinterpret_cast<uint32_t *>(&a); u.y = *reinterpret_cast<uint32_t *>(&b);
        *reinterpret_cast<uint2 *>(out + n * K + 4 * k4) = u;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host side: tensor maps
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
encode_tiled_fn get_encode() {
    static encode_tiled_fn fn = nullptr; static std::once_flag once;
    std::call_once(once, [] {
        void * p = nullptr; cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess) fn = (encode_tiled_fn)p;
    });
    return fn;
}
// bf16 matrix [rows][cols] row-major (cols contiguous), box = 64 cols x box_rows, 128B swizzle
int make_tmap_bf16(CUtensorMap * tm, const void * ptr, int64_t rows, int64_t cols, int box_rows) {
    encode_tiled_fn enc = get_encode(); if (!enc) return -1;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -2;
}

template <int BN>
int launch_gemm_bf16(const void * A_bf16, const void * B_bf16, float * dst, int64_t M, int64_t N, int64_t K, int k_split, cudaStream_t st) {
    using cfg = gemm_cfg<BN>;
    CUtensorMap tmA, tmB;
    if (make_tmap_bf16(&tmA, A_bf16, M, K, BM)) return -10;
    if (make_tmap_bf16(&tmB, B_bf16, N, K, BN)) return -11;
    static bool configured[B200Q_MAX_DEVICES] = {};
    const int dev = b200q_current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(k_gemm_bf16<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg::SMEM) != cudaSuccess) return -12;
        configured[dev] = true;
    }
    dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN), (unsigned)k_split);
    k_gemm_bf16<BN><<<grid, 192, cfg::SMEM, st>>>(tmA, tmB, dst, (int)M, (int)N, (int)K, k_split);
    return (int)cudaGetLastError();
}


// uint8 matrix [rows][row_bytes] (row_bytes contiguous), box = box_bytes x box_rows
int make_tmap_u8(CUtensorMap * tm, const void * ptr, int64_t rows, int64_t row_bytes, int box_bytes, int box_rows, bool swizzle128) {
    encode_tiled_fn enc = get_encode(); if (!enc) return -1;
    cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)box_bytes, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -2;
}

// types whose plane 0 is 16 B / item of low bits and whose other planes are 16 or 32 B per 256 weights (gemmq_planes): the weight slab is decoded
// inside the GEMM.  (Q6_K / Q6_0 / Q8_0 would not fit the shared memory next to a 512-token B tile, Q3_K / IQ2_K / *_KS have planes that are not a
// multiple of 16 bytes per 256 weights: those keep the bf16 scratch.)
constexpr bool gemmq_supported(int type) {
    return type == B200Q_TYPE_IQ4_NL || type == B200Q_TYPE_Q4_0 || type == B200Q_TYPE_Q4_K || type == B200Q_TYPE_IQ4_K ||
           type == B200Q_TYPE_Q4_1 || type == B200Q_TYPE_Q5_0 || type == B200Q_TYPE_Q5_1 || type == B200Q_TYPE_Q5_K || type == B200Q_TYPE_IQ5_K;
}

template <int TYPE, int NB>
int launch_gemm_q(const b200q_gemm_multi & d, int k_split, cudaStream_t st) {
    using cfg = gemmq_cfg<TYPE, NB>;
    gemmq_args a; memset(&a, 0, sizeof a);
    const int64_t p1_row = (d.K / 256) * cfg::P1, p2_row = (d.K / 256) * cfg::P2;
    int tiles = 0;
    for (int i = 0; i < d.n_seg; ++i) {
        b200q_layout L; if (b200q_make_layout(TYPE, d.M[i], d.K, &L)) return -1;
        if (make_tmap_u8(&a.tmP0[i], (const char *)d.W[i] + L.plane_off[0], d.M[i], d.K / 2, 128, BM, true)) return -10;
        if (make_tmap_u8(&a.tmP1[i], (const char *)d.W[i] + L.plane_off[1], d.M[i], p1_row, cfg::P1, BM, false)) return -13;
        if (cfg::P2 && make_tmap_u8(&a.tmP2[i], (const char *)d.W[i] + L.plane_off[2], d.M[i], p2_row, cfg::P2, BM, false)) return -13;
        a.seg[i].dst = d.dst[i]; a.seg[i].mul = d.mul[i]; a.seg[i].dst_bf = (__nv_bfloat16 *)d.dst_bf[i]; a.seg[i].M = (int)d.M[i]; a.seg[i].tile0 = tiles;
        tiles += (int)((d.M[i] + BM - 1) / BM);
    }
    if (make_tmap_bf16(&a.tmB, d.xb, d.N, d.K, NB == 0 ? 128 : 256)) return -11;
    a.n_seg = d.n_seg; a.N = (int)d.N; a.K = (int)d.K; a.k_split = k_split; a.act = d.act; a.limit = d.limit;
    static bool configured[B200Q_MAX_DEVICES] = {};
    const int dev = b200q_current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(k_gemm_q<TYPE, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg::SMEM) != cudaSuccess) return -12;
        configured[dev] = true;
    }
    dim3 grid((unsigned)tiles, (unsigned)((d.N + cfg::BN - 1) / cfg::BN), (unsigned)k_split);
    k_gemm_q<TYPE, NB><<<grid, 64 + 32 * DQ_WARPS, cfg::SMEM, st>>>(a);
    return (int)cudaGetLastError();
}

// n_mat uint8 matrices [rows][row_bytes], mat_stride bytes apart: box = box_bytes x box_rows x 1 (one matrix per load)
int make_tmap_u8_3d(CUtensorMap * tm, const void * ptr, int64_t n_mat, int64_t mat_stride, int64_t rows, int64_t row_bytes, int box_bytes, int box_rows, bool swizzle128) {
    encode_tiled_fn enc = get_encode(); if (!enc) return -1;
    cuuint64_t dims[3] = {(cuuint64_t)row_bytes, (cuuint64_t)rows, (cuuint64_t)n_mat};
    cuuint64_t strides[2] = {(cuuint64_t)row_bytes, (cuuint64_t)mat_stride};
    cuuint32_t box[3] = {(cuuint32_t)box_bytes, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -2;
}

// grouped (MoE) launch: ONE 3-D map per weight plane and segment, whatever n_expert; the grid covers the host-known bound on the tiles
template <int TYPE, int NB>
int launch_gemm_q_grouped(const b200q_gemm_grouped & g, cudaStream_t st) {
    using cfg = gemmq_cfg<TYPE, NB>;
    gemmq_gargs a; memset(&a, 0, sizeof a);
    b200q_layout L; if (b200q_make_layout(TYPE, g.M, g.K, &L)) return -1;
    const int64_t p1_row = (g.K / 256) * cfg::P1, p2_row = (g.K / 256) * cfg::P2;
    int tiles = 0;
    for (int i = 0; i < g.n_seg; ++i) {
        const char * W = (const char *)g.W[i];
        if (make_tmap_u8_3d(&a.tmP0[i], W + L.plane_off[0], g.n_expert, g.estride, g.M, g.K / 2, 128, BM, true)) return -10;
        if (make_tmap_u8_3d(&a.tmP1[i], W + L.plane_off[1], g.n_expert, g.estride, g.M, p1_row, cfg::P1, BM, false)) return -13;
        if (cfg::P2 && make_tmap_u8_3d(&a.tmP2[i], W + L.plane_off[2], g.n_expert, g.estride, g.M, p2_row, cfg::P2, BM, false)) return -13;
        a.seg[i].dst = g.dst[i]; a.seg[i].M = (int)g.M; a.seg[i].tile0 = tiles;
        tiles += (int)((g.M + BM - 1) / BM);
    }
    if (make_tmap_bf16(&a.tmB, g.xb, g.n_rows, g.K, NB == 0 ? 128 : 256)) return -11;
    a.n_seg = g.n_seg; a.N = (int)g.n_rows; a.K = (int)g.K; a.k_split = 1;
    a.tiles = (const b200q_moe_tile *)g.tiles; a.n_tiles = g.n_tiles; a.row_dst = g.row_dst;
    static bool configured[B200Q_MAX_DEVICES] = {};
    const int dev = b200q_current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(k_gemm_q<TYPE, NB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg::SMEM) != cudaSuccess) return -12;
        configured[dev] = true;
    }
    dim3 grid((unsigned)tiles, (unsigned)g.max_tiles, 1);
    k_gemm_q<TYPE, NB, true><<<grid, 64 + 32 * DQ_WARPS, cfg::SMEM, st>>>(a);
    return (int)cudaGetLastError();
}

// int8 activation tensor map: [rows][K bytes], box 128 bytes x box_rows, 128B swizzle, zero fill beyond K
static int make_tmap_i8(CUtensorMap * tm, const void * ptr, int64_t rows, int64_t K, int box_rows) { return make_tmap_u8(tm, ptr, rows, K, 128, box_rows, true); }

template <int NB>
static int launch_gemm_bn_i8(const b200q_gemm_multi & d, const int8_t * xq, const float * ts, const int * sx, cudaStream_t st) {
    using cfg = gemmbn_cfg<NB>;
    gemmbn_args a; memset(&a, 0, sizeof a);
    int tiles = 0;
    for (int i = 0; i < d.n_seg; ++i) {
        b200q_layout L; if (b200q_make_layout(B200Q_TYPE_IQ2_BN, d.M[i], d.K, &L)) return -1;
        if (make_tmap_u8(&a.tmP0[i], (const char *)d.W[i] + L.plane_off[0], d.M[i], d.K / 4, 128, BM, true)) return -10;
        a.seg[i].dst = d.dst[i]; a.seg[i].rs = reinterpret_cast<const float *>((const char *)d.W[i] + L.plane_off[1]); a.seg[i].M = (int)d.M[i]; a.seg[i].tile0 = tiles;
        tiles += (int)((d.M[i] + BM - 1) / BM);
    }
    if (make_tmap_i8(&a.tmB, xq, d.N, d.K, NB == 0 ? 128 : 256)) return -11;
    a.ts = ts; a.sx = sx; a.n_seg = d.n_seg; a.N = (int)d.N; a.K = (int)d.K;
    static bool configured[B200Q_MAX_DEVICES] = {};
    const int dev = b200q_current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(k_gemm_bn_i8<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg::SMEM) != cudaSuccess) return -12;
        configured[dev] = true;
    }
    dim3 grid((unsigned)tiles, (unsigned)((d.N + cfg::BN - 1) / cfg::BN), 1);
    k_gemm_bn_i8<NB><<<grid, 64 + 32 * DQ_WARPS, cfg::SMEM, st>>>(a);
    return (int)cudaGetLastError();
}

// split-K factor of the fused kernel: minimise waves x (raw blocks per CTA + fixed cost), the fixed cost (pipeline fill,
// TMEM round trip, epilogue) being worth ~4 raw blocks; split-K pays memset + f32 atomics
int gemmq_choose_split(int64_t tiles, int64_t nr, int sm_count, bool allow_split) {
    if (!allow_split) return 1;
    static const int forced = [] { const char * e = getenv("B200Q_GEMM_SPLIT"); return e ? atoi(e) : 0; }();      // experiments only
    if (forced > 0) return forced <= nr ? forced : (int)nr;
    int best = 1; int64_t best_cost = INT64_MAX;
    for (int ks = 1; ks <= 16 && ks <= nr; ++ks) {
        const int64_t per = (nr + ks - 1) / ks;
        if (ks > 1 && per * (ks - 1) >= nr) continue;                 // an empty split
        const int64_t waves = (tiles * ks + sm_count - 1) / sm_count;
        const int64_t cost = waves * (per + 4) + (ks > 1 ? 2 : 0);
        if (cost < best_cost) { best_cost = cost; best = ks; }
    }
    return best;
}

}  // namespace


int b200q_gemmq_type(int type) { return gemmq_supported(type) ? 1 : 0; }

int b200q_launch_gemm_q_grouped(const b200q_gemm_grouped & g, cudaStream_t st) {
    if (g.n_seg < 1 || g.n_seg > 2 || g.K % 256 || g.nb < 0 || g.nb > 2 || g.max_tiles < 1) return -2;
    switch (g.type) {
#define GQ(T) case T: return g.nb == 2 ? launch_gemm_q_grouped<T, 2>(g, st) : g.nb == 1 ? launch_gemm_q_grouped<T, 1>(g, st) : launch_gemm_q_grouped<T, 0>(g, st);
        GQ(B200Q_TYPE_IQ4_NL) GQ(B200Q_TYPE_Q4_0) GQ(B200Q_TYPE_Q4_K) GQ(B200Q_TYPE_IQ4_K)
        GQ(B200Q_TYPE_Q4_1) GQ(B200Q_TYPE_Q5_0) GQ(B200Q_TYPE_Q5_1) GQ(B200Q_TYPE_Q5_K) GQ(B200Q_TYPE_IQ5_K)
#undef GQ
        default: return -1;
    }
}

// IQ2_BN prefill on the int8 tensor pipe.  X f32 [N][K] is quantised per token into `ws` (int8 [N][K] | ts[N] | sx[N]); up to 3 tensors share it.
// Requires K % 64 == 0 (16-byte TMA strides); returns -100 when the shape is not eligible (callers use the bf16 path).
size_t b200q_gemm_i8_workspace_bytes(int64_t K, int64_t N) { return (size_t)b200q_align_up(N * K, 256) + (size_t)b200q_align_up(N * 8, 256); }
int b200q_launch_gemm_bn_i8(const b200q_gemm_multi & d, const float * x, int64_t x_stride, void * ws, size_t ws_bytes, cudaStream_t st) {
    if (d.type != B200Q_TYPE_IQ2_BN || d.K % 64 || d.N < 1 || d.n_seg < 1 || d.n_seg > GEMMQ_MAX_SEGS) return -100;
    const int64_t xs = x_stride ? x_stride : d.K;
    if (((uintptr_t)x & 15) || (xs & 3) || ws_bytes < b200q_gemm_i8_workspace_bytes(d.K, d.N)) return -100;
    int8_t * xq = (int8_t *)ws; float * ts = (float *)((char *)ws + b200q_align_up(d.N * d.K, 256)); int * sx = (int *)(ts + d.N);
    k_quantize_rows_i8<<<(unsigned)d.N, 256, 0, st>>>(x, xs, xq, ts, sx, d.K);
    cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) return (int)e;
    const int nb = d.N > 256 ? 2 : (d.N > 128 ? 1 : 0);
    return nb == 2 ? launch_gemm_bn_i8<2>(d, xq, ts, sx, st) : nb == 1 ? launch_gemm_bn_i8<1>(d, xq, ts, sx, st) : launch_gemm_bn_i8<0>(d, xq, ts, sx, st);
}

// dst[j][i] = a[j][i] + b[j % nb][i]  (GGML_OP_ADD of a mat-mul result with a bias row / a same-shape tensor, when it is NOT fused into the mat-vec)
__global__ void k_add_rows(const float * __restrict__ a, const float * __restrict__ b, float * __restrict__ dst, int64_t m, int64_t n, int64_t nb) {
    const int64_t total = m * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) dst[i] = a[i] + b[((i / m) % nb) * m + i % m];
}
int b200q_launch_add_rows(const float * a, const float * b, float * dst, int64_t m, int64_t n, int64_t nb, cudaStream_t st) {
    if (m < 1 || n < 1 || nb < 1) return -2;
    int64_t g = (m * n + 255) / 256; if (g > 148 * 16) g = 148 * 16;
    k_add_rows<<<(unsigned)g, 256, 0, st>>>(a, b, dst, m, n, nb);
    return (int)cudaGetLastError();
}

// elementwise tail of GGML_OP_FUSED_UP_GATE for n > 8 when it cannot ride in the gate GEMM's epilogue
int b200q_launch_mul_unary(const float * gate, const float * up, float * dst, void * dst_bf16, int64_t total, int act, float limit, cudaStream_t st) {
    if (total % 4) return -2;
    int64_t nb = (total / 4 + 255) / 256; if (nb > 148 * 16) nb = 148 * 16; if (nb < 1) nb = 1;
    k_mul_unary<<<(unsigned)nb, 256, 0, st>>>(gate, up, dst, (__nv_bfloat16 *)dst_bf16, total / 4, act, limit);
    return (int)cudaGetLastError();
}

// would the fused kernel run this shape without split-K (so that a non-linear epilogue can be fused)?
int b200q_gemm_epilogue_fusable(int type, int64_t M, int64_t K, int64_t N, int sm_count, int fused) {
    if (!(fused && gemmq_supported(type) && K % 256 == 0)) return 0;
    // Measured (scripts/pp_breakdown.py, Llama-3-8B up/gate, 512 tokens): gate GEMM with the unary-mul in its epilogue 98 us vs
    // plain gate GEMM 60 us + k_mul_unary 20 us: the grid is a single wave, every CTA reaches its epilogue at the same time and the
    // extra loads are fully exposed.  The fused epilogue therefore stays opt-in until the kernel is persistent (epilogue of tile i
    // under the main loop of tile i+1): option "fuse_epilogue" / B200Q_FUSE_EPILOGUE=1 (passed here as fused == 2).
    if (fused < 2) return 0;
    const int bn = N > 256 ? 512 : (N > 128 ? 256 : 128);
    const int64_t tiles = ((M + BM - 1) / BM) * ((N + bn - 1) / bn);
    return gemmq_choose_split(tiles, K / 256, sm_count, true) == 1;
}

size_t b200q_gemm_workspace_bytes(int type, int64_t M, int64_t K, int64_t N) {
    (void)type;
    return (size_t)b200q_align_up(N * K * 2, 256) + (size_t)b200q_align_up(M * K * 2, 256);
}

// f32 [N][K] -> bf16 [N][K] (shared by the mat-muls that consume the same activation)
int b200q_launch_f32_to_bf16(const float * x, int64_t x_stride, void * out, int64_t K, int64_t N, cudaStream_t st) {
    if (K % 4) return -2;
    const int64_t xs = x_stride ? x_stride : K;
    if (K % 8 == 0 && xs % 4 == 0 && !((uintptr_t)x & 15) && !((uintptr_t)out & 15)) {
        const int64_t total8 = N * (K / 8); int64_t nb = (total8 + 256 * 4 - 1) / (256 * 4); if (nb > 148 * 8) nb = 148 * 8; if (nb < 1) nb = 1;
        k_f32_to_bf16<<<(unsigned)nb, 256, 0, st>>>(x, xs, (__nv_bfloat16 *)out, K, N);
    } else {
        const int64_t total4 = N * (K / 4); int64_t nb = (total4 + 255) / 256; if (nb > 148 * 32) nb = 148 * 32; if (nb < 1) nb = 1;
        k_f32_to_bf16_k4<<<(unsigned)nb, 256, 0, st>>>(x, xs, (__nv_bfloat16 *)out, K, N);
    }
    return (int)cudaGetLastError();
}

// n_seg weight tensors of one type and K sharing X = bf16 [N][K] (already converted); dst[i] f32 [N][M_i].
// wscratch: bf16 W scratch (max M_i x K) for the unfused path.
int b200q_launch_gemm_multi_bf16x(const b200q_gemm_multi & d, void * wscratch, size_t ws_bytes, int sm_count, int fused, cudaStream_t st) {
    if (d.K % 8) return -2;
    if (d.n_seg < 1 || d.n_seg > GEMMQ_MAX_SEGS) return -2;
    const int type = d.type; const int64_t K = d.K, N = d.N;
    bool epi = false; for (int i = 0; i < d.n_seg; ++i) epi = epi || d.mul[i] || d.dst_bf[i];
    const bool use_fused = fused && gemmq_supported(type) && K % 256 == 0;
    if (use_fused) {
        // one CTA dequantises a 128-row block once for up to 512 tokens (two 256-column accumulators in TMEM);
        // split-K (f32 atomics) fills the SMs when there are few row blocks
        const int nb = N > 256 ? 2 : (N > 128 ? 1 : 0);
        const int bn = nb == 0 ? 128 : 256 * nb;
        int64_t mt = 0; for (int i = 0; i < d.n_seg; ++i) mt += (d.M[i] + BM - 1) / BM;
        const int64_t tiles = mt * ((N + bn - 1) / bn);
        const int k_split = gemmq_choose_split(tiles, K / 256, sm_count, !epi);
        if (k_split > 1) for (int i = 0; i < d.n_seg; ++i) { cudaError_t e = cudaMemsetAsync(d.dst[i], 0, (size_t)d.M[i] * N * sizeof(float), st); if (e != cudaSuccess) return -3; }
        switch (type) {
#define GQ(T) case T: return nb == 2 ? launch_gemm_q<T, 2>(d, k_split, st) : nb == 1 ? launch_gemm_q<T, 1>(d, k_split, st) : launch_gemm_q<T, 0>(d, k_split, st);
            GQ(B200Q_TYPE_IQ4_NL) GQ(B200Q_TYPE_Q4_0) GQ(B200Q_TYPE_Q4_K) GQ(B200Q_TYPE_IQ4_K)
            GQ(B200Q_TYPE_Q4_1) GQ(B200Q_TYPE_Q5_0) GQ(B200Q_TYPE_Q5_1) GQ(B200Q_TYPE_Q5_K) GQ(B200Q_TYPE_IQ5_K)
#undef GQ
            default: break;
        }
    }
    if (epi) return -6;     // the generic path has no fused epilogue: callers use b200q_launch_mul_unary
    // unfused: bf16 weight scratch + plain bf16 GEMM per tensor; tile / split selection: fill ~1 wave of the SMs
    for (int i = 0; i < d.n_seg; ++i) {
        const int64_t M = d.M[i];
        b200q_layout L; if (b200q_make_layout(type, M, K, &L)) return -1;
        const int64_t mt = (M + BM - 1) / BM;
        const bool bn256 = N >= 256 && mt * ((N + 255) / 256) >= sm_count / 2;
        const int64_t tiles = bn256 ? mt * ((N + 255) / 256) : mt * ((N + 127) / 128);
        int k_split = 1;
        const int64_t nk = (K + BK - 1) / BK;
        while (tiles * k_split * 2 <= sm_count && k_split * 2 <= 8 && nk / (k_split * 2) >= 8) k_split *= 2;
        if (k_split > 1) { cudaError_t e = cudaMemsetAsync(d.dst[i], 0, (size_t)M * N * sizeof(float), st); if (e != cudaSuccess) return -3; }
        if (ws_bytes < (size_t)b200q_align_up(M * K * 2, 256)) return -5;
        int rc = b200q_launch_dequant_bf16(d.W[i], L, wscratch, st); if (rc) return rc;
        rc = bn256 ? launch_gemm_bf16<256>(wscratch, d.xb, d.dst[i], M, N, K, k_split, st) : launch_gemm_bf16<128>(wscratch, d.xb, d.dst[i], M, N, K, k_split, st);
        if (rc) return rc;
    }
    return 0;
}

int b200q_launch_gemm_bf16x(int type, const void * W, const void * xb, float * dst, int64_t M, int64_t K, int64_t N,
                            void * wscratch, size_t ws_bytes, int sm_count, int fused, cudaStream_t st) {
    b200q_gemm_multi d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = 1; d.W[0] = W; d.dst[0] = dst; d.M[0] = M; d.K = K; d.N = N; d.xb = xb;
    return b200q_launch_gemm_multi_bf16x(d, wscratch, ws_bytes, sm_count, fused, st);
}

// A = planes of `type` [M][K]; X = f32 [N][K]; dst f32 [N][M].  Workspace: bf16 X followed by bf16 W (unfused path only).
int b200q_launch_gemm(int type, const void * W, const float * x, int64_t x_stride, float * dst, int64_t M, int64_t K, int64_t N,
                      void * ws, size_t ws_bytes, int sm_count, int fused, cudaStream_t st) {
    if (ws_bytes < b200q_gemm_workspace_bytes(type, M, K, N)) return -5;
    static const int use_i8 = [] { const char * e = getenv("B200Q_BN_INT8"); return e ? atoi(e) : 1; }();
    if (type == B200Q_TYPE_IQ2_BN && use_i8 && fused) {          // ternary weights: int8 tensor pipe (kind::i8), exact integer accumulation
        b200q_gemm_multi d; memset(&d, 0, sizeof d);
        d.type = type; d.n_seg = 1; d.W[0] = W; d.dst[0] = dst; d.M[0] = M; d.K = K; d.N = N;
        const int rc = b200q_launch_gemm_bn_i8(d, x, x_stride, ws, ws_bytes, st);
        if (rc != -100) return rc;
    }
    void * xb = ws;
    void * wb = (char *)ws + b200q_align_up(N * K * 2, 256);
    int rc = b200q_launch_f32_to_bf16(x, x_stride, xb, K, N, st); if (rc) return rc;
    return b200q_launch_gemm_bf16x(type, W, xb, dst, M, K, N, wb, ws_bytes - (size_t)b200q_align_up(N * K * 2, 256), sm_count, fused, st);
}
