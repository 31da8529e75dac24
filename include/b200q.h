/* b200q.h — C ABI of libb200q.so: the Blackwell (sm_100a) quantized mat-mul hot path of ik_llama.cpp.
 *
 * Plain C: pointers, sizes, ggml_type ids.  No torch / ggml types.  All device pointers are CUDA device
 * addresses on the current device; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Every function returns 0 on success, a negative B200Q_E_* code otherwise (b200q_last_error() has the text).
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with B200Q_E_CUDA.
 *
 * What each entry point replaces in the reference (paths relative to the ik_llama.cpp tree):
 *   b200q_set_tensor / b200q_get_tensor    ggml_backend_cuda_buffer_set_tensor / _get_tensor   ggml/src/ggml-cuda.cu:641-672
 *                                          (+ the wire->device re-layout, cf. run-time repack `-rtr`)
 *   b200q_mul_mat                          ggml_cuda_mul_mat dispatcher                        ggml/src/ggml-cuda.cu:2645-2727
 *   b200q_mul_mat_vec[_multi]              quantize_row_q8_1_cuda + ggml_cuda_op_mul_mat_vec_q ggml/src/ggml-cuda.cu:2503-2604,
 *                                          (mul_mat_vec_q / iqk_mul_mat_vec_q kernels)         ggml-cuda/mmvq-templates.cuh:68-150,287-303
 *                                          incl. the "following MUL_MATs share src1" fusion    ggml/src/ggml-cuda.cu:2573-2601
 *   b200q_fused_up_gate_vec                ggml_cuda_up_gate_unary / fused_mul_mat_vec_q       ggml/src/ggml-cuda.cu:3542-3620, mmvq-templates.cuh:152-330
 *   b200q_mul_mat_gemm                     quantize_mmq_q8_1_cuda + mul_mat_q (MMQ)            ggml-cuda/mmq.cuh:3849-4173; dequant+cuBLAS fallback ggml-cuda.cu:1723-1894
 *   b200q_dequantize_bf16                  dequantize_block_* (convert.cu)                     ggml-cuda/convert.cu
 *   b200q_reduce_*                         ggml_cuda_op_reduce                                 ggml-cuda/reduce.cu:125-598
 * Tensor conventions are ggml's: W is [M rows][K cols] in the GGUF wire format of `type`
 * (row stride = ggml_row_size(type, K)); x is f32 [N][K]; dst is f32 [N][M]  (dst[j*M + i]).
 */
#ifndef B200Q_H
#define B200Q_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B200Q_ABI_VERSION 1
#if defined(__GNUC__)
#define B200Q_API __attribute__((visibility("default")))
#else
#define B200Q_API
#endif

enum { B200Q_OK = 0, B200Q_E_TYPE = -1, B200Q_E_SHAPE = -2, B200Q_E_CUDA = -3, B200Q_E_ARG = -4, B200Q_E_NOMEM = -5 };
/* unary of GGML_OP_FUSED_UP_GATE.  `limit` (op_params[1]) follows the reference: SILU only, applied AFTER the activation
 * (g = min(silu(g), limit), u = clamp(u, +-limit)), ignored when <= 1e-6 (mmvq-templates.cuh:253-258, unary.cu:63-72).
 * SWIGLU_OAI: alpha 1.702, limit 7, no bias (ggml-cuda.cu:3607-3611). */
enum { B200Q_UNARY_NONE = 0, B200Q_UNARY_SILU = 1, B200Q_UNARY_GELU = 2, B200Q_UNARY_RELU = 3, B200Q_UNARY_SWIGLU_OAI = 4 };

B200Q_API int          b200q_abi_version(void);
B200Q_API const char * b200q_last_error(void);
B200Q_API int          b200q_set_option(const char * key, int value);   /* "pdl": programmatic dependent launch of the decode kernels (cf. the "-cuda k=v" string of ggml_backend_cuda_init, ggml-cuda.cu:5339) */
B200Q_API int          b200q_device_count(void);                      /* ggml_backend_cuda_get_device_count, ggml-cuda.h:38 */

/* ---- type geometry (mirrors ggml_type_traits: ggml/src/ggml.c:640-1460) ---- */
B200Q_API int     b200q_type_supported(int ggml_type);                /* 1 if MUL_MAT with this src0 type is implemented   */
B200Q_API int64_t b200q_wire_row_size(int ggml_type, int64_t k);      /* == ggml_row_size(type, k); <0 on error            */
B200Q_API int64_t b200q_plane_bytes(int ggml_type, int64_t m, int64_t k); /* device bytes of the re-laid-out tensor        */

/* ---- weights: wire <-> device layout ---- */
B200Q_API int b200q_repack  (int type, const void * wire_dev,   void * planes_dev, int64_t m, int64_t k, void * stream);
B200Q_API int b200q_unrepack(int type, const void * planes_dev, void * wire_dev,   int64_t m, int64_t k, void * stream);
B200Q_API int b200q_set_tensor(int type, const void * wire_host, void * planes_dev, int64_t m, int64_t k, void * stream); /* H2D + repack, synchronous */
B200Q_API int b200q_get_tensor(int type, const void * planes_dev, void * wire_host, int64_t m, int64_t k, void * stream); /* unrepack + D2H, synchronous */

/* ---- decode: n <= 8 activation columns ---- */
B200Q_API int b200q_mul_mat_vec(int type, const void * W, const float * x, float * dst,
                      int64_t m, int64_t k, int n, int64_t x_stride, const float * bias, void * stream);
/* several weight tensors of the same type and K sharing one activation (Q,K,V): one launch */
B200Q_API int b200q_mul_mat_vec_multi(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m,
                            int64_t k, const float * x, int n, int64_t x_stride, void * stream);
/* dst = unary(gate.x) * (up.x)   (optionally clamped: limit > 0) */
B200Q_API int b200q_fused_up_gate_vec(int type, const void * W_up, const void * W_gate, const float * x, float * dst,
                            int64_t m, int64_t k, int n, int64_t x_stride, int unary, float limit, void * stream);

/* q8_1 hand-off FUSED_UP_GATE -> MUL_MAT(ffn_down) for n = 1 (the reference quantises each activation once, quantize_row_q8_1_cuda in
 * ggml_cuda_op_mul_mat_vec_q, ggml-cuda.cu:2503-2604; here the producer's epilogue does it): `q8` is a device scratch of
 * b200q_q8_scratch_bytes(m_of_up_gate) bytes, zeroed ONCE with b200q_q8_scratch_init.  *q8_produced = 1 if the launch emitted the image
 * (eligible shape and kernel); pass q8_in = NULL to b200q_mul_mat_vec_q8 otherwise.  x / dst are always read / written as usual. */
B200Q_API size_t b200q_q8_scratch_bytes(int64_t k);
B200Q_API int b200q_q8_scratch_init(void * q8, int64_t k, void * stream);
B200Q_API int b200q_fused_up_gate_vec_q8(int type, const void * W_up, const void * W_gate, const float * x, float * dst, int64_t m, int64_t k,
                               int unary, float limit, void * q8_out, int * q8_produced, void * stream);
B200Q_API int b200q_mul_mat_vec_q8(int type, const void * W, const float * x, const void * q8_in, float * dst, int64_t m, int64_t k,
                         const float * bias, void * stream);

/* Decode chains: tell the NEXT decode launch of this thread which weights the launch AFTER it will stream, so that it can warm their first
 * stages in L2 (cp.async.bulk.prefetch.L2) while it runs; a kernel cannot prefetch into shared memory before the previous one has left the SM.
 * The hint is consumed (cleared) by the next b200q_mul_mat_vec* / b200q_fused_up_gate_vec* call.  W_gate != NULL: fused up/gate (n_tensors = 1). */
B200Q_API int b200q_decode_prefetch_next(int type, int n_tensors, const void * const * W, const void * W_gate, const int64_t * m, int64_t k);

/* ---- prefill: tcgen05 GEMM ---- */
B200Q_API size_t b200q_mul_mat_workspace(int type, int64_t m, int64_t k, int64_t n);
B200Q_API int b200q_mul_mat_gemm(int type, const void * W, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                       void * workspace, size_t workspace_bytes, void * stream);
/* activations shared by several mat-muls (Q,K,V / up,gate): convert once, then call the _bf16 variant per weight tensor */
B200Q_API int b200q_convert_f32_bf16(const float * x, int64_t x_stride, void * out_bf16, int64_t k, int64_t n, void * stream);
B200Q_API int b200q_mul_mat_gemm_bf16(int type, const void * W, const void * x_bf16, float * dst, int64_t m, int64_t k, int64_t n,
                            void * workspace /* bf16 [m][k] scratch, only for types without a fused kernel */, size_t workspace_bytes, void * stream);
B200Q_API int b200q_dequantize_bf16(int type, const void * W, void * out_bf16, int64_t m, int64_t k, void * stream);
/* several MUL_MATs of one type / K that share src1, n > 8 (the look-ahead fusion of ggml_cuda_mul_mat_q, ggml-cuda.cu:2573-2601):
 * ONE launch walks the row tiles of up to 3 tensors (Q,K,V) */
B200Q_API int b200q_mul_mat_gemm_multi_bf16(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m, int64_t k,
                                  const void * x_bf16, int64_t n, void * workspace, size_t workspace_bytes, void * stream);
/* GGML_OP_FUSED_UP_GATE for n > 8 (ggml_cuda_up_gate_unary, ggml-cuda.cu:3588-3618: two MMQ + ggml_fused_mul_unary): the unary-mul
 * rides in the epilogue of the gate GEMM; dst_bf16 (optional, may be NULL) receives a bf16 copy = the operand of ffn_down.
 * workspace >= align256(m*n*4) + align256(m*k*2) */
B200Q_API int b200q_fused_up_gate_gemm_bf16(int type, const void * W_up, const void * W_gate, const void * x_bf16, float * dst, void * dst_bf16,
                                  int64_t m, int64_t k, int64_t n, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream);

/* ---- GGML_OP_REDUCE (sum) for the row-parallel mat-muls of split-mode-graph: NVLS all-reduce in ONE kernel ----
 * One process per GPU; the reduction buffers live in symmetric memory: `mc_base` / `mc_flag` = multicast (NVLS) addresses,
 * `local_base` / `local_flag` = this rank's own mapping of the same allocation.  Two parity buffers of `parity_stride` floats
 * alternate (base + parity*stride); the parity and the flag target come from the device counter `seq_counter` (rank-local,
 * zero-initialised), so the call has constant arguments and can be captured in a CUDA graph.  `seq_counter` points at FOUR u32
 * {reduces done, dirty floats of parity buffer 0, of parity buffer 1, pad}, zero-initialised.  `cta_counter`: rank-local u32, zero. */
B200Q_API int b200q_reduce_sum_nvls(const float * in, float * out, int64_t n, void * mc_base, void * local_base, int64_t parity_stride,
                          void * mc_flag, const void * local_flag, uint32_t world_size, void * seq_counter, void * cta_counter, void * stream);

/* Prefill-sized REDUCE: two-shot bf16 all-reduce in ONE kernel (the reference casts the partial to bf16/f16 when ne[1] > 32,
 * src/llama-build-context.cpp:1198-1200, and runs reduce-scatter + all-gather, ggml-cuda/reduce.cu:306-372): f32 partial -> bf16 staging in
 * symmetric memory, barrier, multimem.ld_reduce of the rank's 1/world slice (f32 accumulation in the switch) + multimem.st of the sum to every
 * rank, barrier, copy-out as bf16 (out_bf16: the activation operand of the next GEMM) and / or f32 (out_f32).  `state`: rank-local u32[4], zero. */
typedef struct b200q_nvls_stage {
    void * mc_stage; void * local_stage; int64_t stage_elems;   /* bf16 staging buffer: multicast address / this rank's mapping / capacity in elements */
    void * mc_flag; const void * local_flag;                    /* u32 flag word in symmetric memory (multicast / local), zero-initialised */
    uint32_t world_size; uint32_t rank;
    void * state;
} b200q_nvls_stage;
B200Q_API int b200q_reduce_sum_nvls_bf16(const float * in, float * out_f32, void * out_bf16, int64_t n, const b200q_nvls_stage * stage, void * stream);

/* ---- tensor-parallel decode (n = 1): the GGML_OP_REDUCE after a row-parallel mat-vec fused INTO the mat-vec kernels ----
 * (reference: ggml_cuda_op_reduce runs as its own node after wo / ffn_down under -sm graph, ggml-cuda/reduce.cu:125-598).
 * Tagged-slot exchange, no flag, no fence, no acknowledgement round trip: an entry is {f32 value, u32 number of the reduce}, written with one
 * 8-byte store.  reduce_out: the kernel's epilogue broadcasts each finished partial row to slot [parity][this rank][row] of EVERY rank with
 * multimem.st through the NVLS multicast mapping (dst is not written; m_total <= ll_stride).  reduce_in: `x` is ignored; the CTAs of the consumer
 * sum the per-rank slots in rank order (bit-identical on every rank), each its own slice, publish the sums in ll_reduced with the same tagging and
 * quantise their activations from there (k <= ll_stride).  W_gate != NULL: fused up/gate mode (n_tensors = 1).
 * CONTRACT: on one communicator every reduce_out launch must be followed, on every rank, by at least one reduce_in launch before the next
 * reduce_out (the two parities are reused every second reduce); all ranks issue the same sequence.
 *   ll_mc / ll_local: multicast / local address of the symmetric slot array, 2 * world_size * ll_stride entries of 8 bytes, zero-initialised;
 *   ll_reduced: rank-local, 2 * ll_stride entries, zero-initialised; ll_state: rank-local u32[2], zero-initialised; all 16-byte aligned. */
typedef struct b200q_nvls_comm {
    void * ll_mc; const void * ll_local; void * ll_reduced; int64_t ll_stride; uint32_t world_size; uint32_t rank; void * ll_state;
    void * const * ll_peers;    /* optional (HOST array of world_size device pointers, world_size <= 8): every rank's mapping of the slot array in THIS
                                 * rank's address space (peer memory).  When given, reduce_out writes each peer's copy with ordinary stores, the rows of
                                 * a CTA as consecutive 16-byte lanes of one warp (coalesced into 128-byte NVLink packets), instead of one multicast
                                 * store per row pair.  NULL: multimem.st only. */
} b200q_nvls_comm;
B200Q_API int b200q_mul_mat_vec_tp(int type, int n_tensors, const void * const * W, const void * W_gate, float * const * dst, const int64_t * m,
                         int64_t k, const float * x, int unary, float limit, const b200q_nvls_comm * comm, int reduce_in, int reduce_out, void * stream);

/* ---- dispatcher (what GGML_OP_MUL_MAT calls): n <= 8 -> mat-vec, else GEMM ---- */
B200Q_API int b200q_mul_mat(int type, const void * W, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                  void * workspace, size_t workspace_bytes, void * stream);
/* any-n variants of the multi-tensor and fused up/gate ops with f32 activations (what the graph nodes carry) */
B200Q_API size_t b200q_mul_mat_multi_workspace(int type, int n_tensors, const int64_t * m, int64_t k, int64_t n);
B200Q_API int b200q_mul_mat_multi(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m, int64_t k,
                        const float * x, int64_t n, void * workspace, size_t workspace_bytes, void * stream);
B200Q_API size_t b200q_fused_up_gate_workspace(int type, int64_t m, int64_t k, int64_t n);
B200Q_API int b200q_fused_up_gate(int type, const void * W_up, const void * W_gate, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                        int unary, float limit, void * workspace, size_t workspace_bytes, void * stream);
/* GGML_OP_ADD of a mat-mul result with its bias row(s): dst[j][i] = a[j][i] + b[j % nb][i] (i < m, j < n) */
B200Q_API int b200q_add_rows(const float * a, const float * b, float * dst, int64_t m, int64_t n, int64_t nb, void * stream);
/* ---- MoE decode: GGML_OP_MUL_MAT_ID / GGML_OP_MOE_FUSED_UP_GATE for small batches (ggml_cuda_mul_mat_id / ggml_cuda_moe_up_gate_unary,
 * ggml-cuda.cu:2836-3540; mul_mat_vec_q with ids, mmvq-templates.cuh:293-302).  W: n_expert matrices [m x k] of `type`, each in the device layout,
 * b200q_plane_bytes(type, m, k) apart; ids: DEVICE int32 [n_tokens][n_used]; x f32 [n_tokens][nb1][k] (nb1 = 1: the column is shared by the slots of
 * a token, nb1 = n_used: one column per slot); dst f32 [n_tokens][n_used][m]:  dst[t][e] = W[ids[t][e]] . x[t][e % nb1]
 * (W_gate != NULL: unary(W_gate[id] . x) * (W[id] . x)).  Expert ids are resolved on the device.  The quantised activation columns of a launch live
 * in shared memory (200 KB of q8_1): batches whose n_tokens * nb1 columns exceed that are walked in token chunks by the same kernel (functional
 * path for MoE prefill when the type or shape has no grouped GEMM, see below). */
B200Q_API int b200q_mul_mat_id_vec(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                         int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * stream);
/* ---- MoE prefill: the same ops as a grouped tcgen05 GEMM over expert-sorted tokens (ggml_cuda_mul_mat_id with mul_mat_q_id, ggml-cuda.cu:3210-3307).
 * On the device: route (count the slots per expert, scan, sort the slots by expert, one tile-table entry per 128/256/512-token tile of each
 * expert), gather the routed activation columns as bf16, one GEMM launch that dequantises the expert weights inside the kernel (up and gate
 * as two segments of that launch for W_gate != NULL, then the unary-mul).  Nothing is read back to the host: the call can be captured in
 * a CUDA graph.  No split-K: the result is bit-identical from run to run.  Types: IQ4_NL, Q4_0, Q4_1, Q5_0, Q5_1, Q4_K, Q5_K, IQ4_K,
 * IQ5_K with k % 256 == 0 and n_expert <= 512 (b200q_mul_mat_id_gemm returns B200Q_E_TYPE / B200Q_E_SHAPE otherwise).
 * b200q_mul_mat_id_workspace: device bytes the grouped path needs (256-byte aligned workspace), 0 if the type / shape is not covered;
 * up_gate != 0 for GGML_OP_MOE_FUSED_UP_GATE.  b200q_mul_mat_id: the dispatcher (what the graph nodes call): the grouped GEMM for covered
 * types and shapes at or above a batch threshold set from measurement (scripts/moe_prefill_bench.py, DESIGN.md §4), b200q_mul_mat_id_vec
 * otherwise (workspace may then be NULL). */
B200Q_API size_t b200q_mul_mat_id_workspace(int type, int64_t m, int64_t k, int n_expert, int n_used, int nb1, int n_tokens, int up_gate);
B200Q_API int b200q_mul_mat_id_gemm(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                          int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream);
B200Q_API int b200q_mul_mat_id(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                     int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream);
/* same through HOST activations/results: H2D(x) -> mul_mat -> D2H(dst), synchronous (end-to-end entry point) */
B200Q_API int b200q_mul_mat_host(int type, const void * W_planes_dev, const float * x_host, float * dst_host,
                       int64_t m, int64_t k, int64_t n, void * stream);

#ifdef __cplusplus
}
#endif
#endif /* B200Q_H */
