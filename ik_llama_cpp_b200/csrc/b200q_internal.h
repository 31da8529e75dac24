// b200q_internal.h — declarations shared by the translation units of libb200q.so (not part of the public ABI).
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>
#include "b200q_types.cuh"

#define B200Q_MAX_SEGS 4
// function attributes (opt-in shared memory size) are per device: remember per device whether a kernel has been configured
#define B200Q_MAX_DEVICES 16
static inline int b200q_current_device() { int d = 0; if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= B200Q_MAX_DEVICES) d = 0; return d; }

enum { B200Q_ACT_NONE = 0, B200Q_ACT_SILU = 1, B200Q_ACT_GELU = 2, B200Q_ACT_RELU = 3, B200Q_ACT_SWIGLU_OAI = 4 };

#if defined(__CUDACC__)
// act(gate) * up of GGML_OP_FUSED_UP_GATE, with the reference's order of operations (fused_mul_mat_vec_q, mmvq-templates.cuh:240-275;
// fused_mul_silu_f32 with limit, ggml-cuda/unary.cu:63-72; CPU: ggml.c:16939-16945):
//   SILU:  g = silu(g); if (limit > 1e-6) { g = min(g, limit); u = clamp(u, -limit, limit); }  r = g * u      (the clamp follows the activation)
//   GELU / RELU: limit is ignored;   SWIGLU_OAI (no bias): g = min(g, 7), u = clamp(u, -7, 7), r = g / (1 + exp(-1.702 g)) * (1 + u)
// FAST: __expf / __fdividef (prefill epilogue: |rel err| ~1e-6, far below the bf16 operand noise of that path)
template <bool FAST>
__device__ __forceinline__ float b200q_glu(int act, float g, float u, float limit) {
    switch (act) {
        case B200Q_ACT_SILU: {
            g = FAST ? __fdividef(g, 1.0f + __expf(-g)) : g / (1.0f + expf(-g));
            if (limit > 1e-6f) { g = fminf(g, limit); u = fmaxf(-limit, fminf(limit, u)); }
            return g * u;
        }
        case B200Q_ACT_GELU: { const float c = 0.79788456080286535587989211986876f, a = 0.044715f; return 0.5f * g * (1.0f + tanhf(c * g * (1.0f + a * g * g))) * u; }
        case B200Q_ACT_RELU: return fmaxf(g, 0.0f) * u;
        case B200Q_ACT_SWIGLU_OAI: {
            g = fminf(g, 7.0f); u = fmaxf(fminf(u, 7.0f), -7.0f);
            return (FAST ? __fdividef(g, 1.0f + __expf(-g * 1.702f)) : g / (1.0f + expf(-g * 1.702f))) * (1.0f + u);
        }
        default: return g * u;
    }
}
#endif

// types whose canonical decode has a non-zero subtracted offset (ml) -> the kernel needs the integer activation sums
B200Q_HD constexpr bool b200q_mmvq_has_ml(int type) {
    return !(type == B200Q_TYPE_IQ4_NL || type == B200Q_TYPE_Q8_0 || type == B200Q_TYPE_IQ4_XS || type == B200Q_TYPE_MXFP4);
}
// types whose two 16-weight halves of an item carry different scales / offsets
B200Q_HD constexpr bool b200q_split16(int type) {
    return type == B200Q_TYPE_Q6_K || type == B200Q_TYPE_IQ4_K || type == B200Q_TYPE_IQ5_K || type == B200Q_TYPE_Q2_K || type == B200Q_TYPE_Q3_K ||
           type == B200Q_TYPE_IQ2_K || type == B200Q_TYPE_IQ3_K;
}

// device view of the NVLS communicator of include/b200q.h (b200q_nvls_comm) + the direction flags of one launch
struct b200q_tp_comm {
    // tagged-slot exchange of the fused decode reduce (k_mmvq_ring<..., TP>): entry = {f32 value, u32 id of the reduce}, one 8-byte store
    float2 * ll_mc;              // multicast address of slots[2 parities][world][ll_stride]
    const float2 * ll_local;     // this rank's mapping of the same
    float2 * ll_red;             // rank-local [2 parities][ll_stride]: the summed vector, same tagging (filled cooperatively by the consumer's CTAs)
    int64_t ll_stride; uint32_t world, rank;
    float2 * ll_peer[8];         // optional: every rank's mapping of the slot array (peer memory over NVLink); ll_peer[0] != nullptr selects unicast stores
    uint32_t * seq;              // rank-local: [0] reduces issued by this rank, [1] CTA arrival counter
    int in; int out;
};
struct b200q_mmvq_seg_desc { const void * W; const void * W2; float * dst; const float * bias; int64_t M; };
struct b200q_mmvq_desc {
    int type; int n_seg; b200q_mmvq_seg_desc seg[B200Q_MAX_SEGS];
    int64_t K; const float * x; int64_t x_stride; int ncols; int act; float limit; int sm_count; int pdl; int ring;
    b200q_tp_comm tp;
    const void * q8_in;     // n = 1: activations already quantised by the producing launch (b200q_q8 image); x is still passed for the fallback
    void * q8_out;          // fused up/gate, n = 1: also emit dst as a b200q_q8 image for the next MUL_MAT
    const b200q_mmvq_desc * next;   // optional: the decode launch that will follow this one; its first weight stages are warmed in L2 (b200q_decode_prefetch_next)
};
// b200q_q8 image of a K-vector: [K int8][K/32 f32 d][K/32 i32 sums][K/32 u32 arrival counters] (+ 16 B slack)
static inline size_t b200q_q8_image_bytes(int64_t k) { return (size_t)(k + 12 * (k / 32) + 16); }

int b200q_launch_repack(const void * wire, void * planes, const b200q_layout & L, int inverse, cudaStream_t st);
int b200q_launch_dequant_bf16(const void * W, const b200q_layout & L, void * out, cudaStream_t st);
int b200q_launch_mmvq(const b200q_mmvq_desc & d, cudaStream_t st);
// MoE decode: W = n_expert matrices [M x K], b200q_plane_bytes(type, M, K) apart; ids device int32 [n_tokens][n_used]; x f32 [n_tokens][nb1][K]; dst f32 [n_tokens][n_used][M]
struct b200q_mmvq_id_desc {
    int type; const void * W; const void * W2; const int32_t * ids; const float * x; float * dst;
    int64_t M, K; int n_expert, n_used, nb1, n_tokens; int act; float limit; int sm_count; int pdl;
};
int b200q_launch_mmvq_id(const b200q_mmvq_id_desc & d, cudaStream_t st);
int b200q_launch_wire_mmvq_id(const b200q_mmvq_id_desc & d, cudaStream_t st);
// wire-layout types (b200q_wire.cu)
int b200q_launch_wire_mmvq(const b200q_mmvq_desc & d, cudaStream_t st);
int b200q_launch_wire_dequant_bf16(int type, const void * W, int64_t M, int64_t K, void * out, cudaStream_t st);

// prefill: up to 3 weight tensors of one type / K that share the bf16 activation operand xb [N][K]
struct b200q_gemm_multi {
    int type; int n_seg; const void * W[3]; float * dst[3]; const float * mul[3]; void * dst_bf[3]; int64_t M[3];
    int64_t K, N; const void * xb; int act; float limit;
};
size_t b200q_gemm_workspace_bytes(int type, int64_t M, int64_t K, int64_t N);
int b200q_launch_gemm(int type, const void * W, const float * x, int64_t x_stride, float * dst, int64_t M, int64_t K, int64_t N,
                      void * ws, size_t ws_bytes, int sm_count, int fused, cudaStream_t st);
int b200q_launch_gemm_bf16x(int type, const void * W, const void * xb, float * dst, int64_t M, int64_t K, int64_t N,
                            void * wscratch, size_t ws_bytes, int sm_count, int fused, cudaStream_t st);
int b200q_launch_gemm_multi_bf16x(const b200q_gemm_multi & d, void * wscratch, size_t ws_bytes, int sm_count, int fused, cudaStream_t st);
int b200q_launch_mul_unary(const float * gate, const float * up, float * dst, void * dst_bf16, int64_t total, int act, float limit, cudaStream_t st);
int b200q_gemm_epilogue_fusable(int type, int64_t M, int64_t K, int64_t N, int sm_count, int fused);
size_t b200q_gemm_i8_workspace_bytes(int64_t K, int64_t N);
int b200q_launch_gemm_bn_i8(const b200q_gemm_multi & d, const float * x, int64_t x_stride, void * ws, size_t ws_bytes, cudaStream_t st);
int b200q_launch_add_rows(const float * a, const float * b, float * dst, int64_t m, int64_t n, int64_t nb, cudaStream_t st);
int b200q_launch_f32_to_bf16(const float * x, int64_t x_stride, void * out, int64_t K, int64_t N, cudaStream_t st);

// MoE prefill (b200q_moe.cu): grouped k_gemm_q over expert-sorted token tiles
int b200q_gemmq_type(int type);          // 1 if k_gemm_q decodes this type inside the kernel
struct b200q_gemm_grouped {
    int type; int n_seg; const void * W[2]; float * dst[2];      // n_seg = 2: up (-> dst[0]) and gate (-> dst[1]) in one launch
    int64_t M, K; int n_expert; int64_t estride;                 // the n_expert matrices of W[i] lie estride bytes apart
    const void * xb; int64_t n_rows;                             // bf16 [n_rows][K], expert-sorted
    const void * tiles; const int * n_tiles; const int * row_dst; int max_tiles; int nb;
};
int b200q_launch_gemm_q_grouped(const b200q_gemm_grouped & g, cudaStream_t st);
struct b200q_moe_plan_t {
    int64_t n_rows; int nb; int max_tiles; int64_t estride;
    size_t off_xb, off_up, off_bounds, off_src, off_dst, off_tiles, off_ntiles, total;     // workspace layout
};
// 0: the grouped path covers this type and shape (p filled); -1: type not covered; -2: shape not covered
int b200q_moe_plan(int type, int64_t m, int64_t k, int n_expert, int n_used, int nb1, int n_tokens, int up_gate, b200q_moe_plan_t * p);
struct b200q_moe_desc {
    int type; const void * W; const void * W_gate; int n_expert; const int32_t * ids; const float * x; float * dst;
    int64_t M, K; int n_used, nb1, n_tokens; int act; float limit;
};
int b200q_launch_moe_gemm(const b200q_moe_desc & d, const b200q_moe_plan_t & p, void * ws, cudaStream_t st);
