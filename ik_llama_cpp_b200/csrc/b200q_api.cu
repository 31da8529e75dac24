// b200q_api.cu — the C ABI of libb200q.so (see include/b200q.h for the reference interfaces each entry replaces).
#include "../../include/b200q.h"
#include "b200q_internal.h"
#include <cuda_runtime.h>
#include <mutex>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

int b200q_launch_allreduce_nvls(const float * in, float * out, int64_t n, void * mc_base, void * local_base, int64_t stride,
                                void * mc_flag, const void * local_flag, uint32_t world, void * seq, void * cta_counter, int sm_count, cudaStream_t st);

int b200q_launch_allreduce_nvls_2shot(const float * in, float * out_f32, void * out_bf16, int64_t n, void * mc_stage, void * local_stage,
                                      void * mc_flag, const void * local_flag, uint32_t world, uint32_t rank, void * state, int sm_count, cudaStream_t st);

namespace {
thread_local char g_err[512] = "";
int fail(int code, const char * fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
    return code;
}
int cuda_fail(const char * what, cudaError_t e) { return fail(B200Q_E_CUDA, "%s: %s", what, cudaGetErrorString(e)); }

struct dev_info { int sm_count = 0; bool ok = false; };
dev_info & device_info() {
    static dev_info info[16]; static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) { static dev_info bad; return bad; }
    std::lock_guard<std::mutex> lk(mu);
    if (!info[dev].ok) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, dev) == cudaSuccess) { info[dev].sm_count = p.multiProcessorCount; info[dev].ok = true; }
    }
    return info[dev];
}
int check_launch(int rc, const char * what) {
    if (rc == 0) return B200Q_OK;
    if (rc == -1) return fail(B200Q_E_TYPE, "%s: unsupported ggml type", what);
    if (rc == -2) return fail(B200Q_E_SHAPE, "%s: unsupported shape", what);
    if (rc == -5) return fail(B200Q_E_NOMEM, "%s: workspace too small", what);
    if (rc > 0) return cuda_fail(what, (cudaError_t)rc);
    return fail(B200Q_E_CUDA, "%s: launch failed (%d)", what, rc);
}
// per-thread scratch for the host-buffer entry points
// (device-aware: a loader thread may serve several GPUs in turn; an allocation made on another device is never reused)
struct scratch { void * p = nullptr; size_t n = 0; int dev = -1; };
void release(scratch & s) {
    if (!s.p) return;
    int cur = 0; cudaGetDevice(&cur);
    if (s.dev >= 0 && s.dev != cur) { cudaSetDevice(s.dev); cudaFree(s.p); cudaSetDevice(cur); } else cudaFree(s.p);
    s.p = nullptr; s.n = 0; s.dev = -1;
}
int ensure(scratch & s, size_t n) {
    int cur = 0; cudaGetDevice(&cur);
    if (s.p && s.dev == cur && s.n >= n) return 0;
    release(s);
    cudaError_t e = cudaMalloc(&s.p, n);
    if (e != cudaSuccess) { s.p = nullptr; return cuda_fail("cudaMalloc(scratch)", e); }
    s.n = n; s.dev = cur; return 0;
}
constexpr size_t STAGE_KEEP = (size_t)64 << 20;      // upload staging above this size is freed right after use (model load)
thread_local scratch g_x, g_y, g_ws, g_stage;
// programmatic dependent launch for the decode kernels (default on; B200Q_PDL=0 or b200q_set_option("pdl",0) disables)
int & opt_ring() { static int v = [] { const char * e = getenv("B200Q_RING"); return e ? atoi(e) : 1; }(); return v; }
int & opt_fuse_epi() { static int v = [] { const char * e = getenv("B200Q_FUSE_EPILOGUE"); return e ? atoi(e) : 0; }(); return v; }
int & opt_fused() { static int v = [] { const char * e = getenv("B200Q_FUSED_GEMM"); return e ? atoi(e) : 1; }(); return v; }
// L2 warm-up of the next launch's weights: measured 753 vs 771 tok/s (slower: the prefetch competes with the running kernel's own stream) -> opt-in
int & opt_pf() { static int v = [] { const char * e = getenv("B200Q_PREFETCH_NEXT"); return e ? atoi(e) : 0; }(); return v; }
int & opt_q8() { static int v = [] { const char * e = getenv("B200Q_Q8_HANDOFF"); return e ? atoi(e) : 1; }(); return v; }
int & opt_pdl() { static int v = [] { const char * e = getenv("B200Q_PDL"); return e ? atoi(e) : 1; }(); return v; }
}  // namespace

extern "C" {

int b200q_abi_version(void) { return B200Q_ABI_VERSION; }
const char * b200q_last_error(void) { return g_err; }
int b200q_set_option(const char * key, int value) {
    if (key && !strcmp(key, "pdl")) { opt_pdl() = value; return B200Q_OK; }
    if (key && !strcmp(key, "prefetch_next")) { opt_pf() = value; return B200Q_OK; }
    if (key && !strcmp(key, "q8_handoff")) { opt_q8() = value; return B200Q_OK; }
    if (key && !strcmp(key, "ring")) { opt_ring() = value; return B200Q_OK; }
    if (key && !strcmp(key, "fused_gemm")) { opt_fused() = value; return B200Q_OK; }
    if (key && !strcmp(key, "fuse_epilogue")) { opt_fuse_epi() = value; return B200Q_OK; }
    return fail(B200Q_E_ARG, "b200q_set_option: unknown option");
}
int b200q_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

int b200q_type_supported(int type) { b200q_layout L; return b200q_make_layout(type, 4, 256, &L) == 0 ? 1 : 0; }
int64_t b200q_wire_row_size(int type, int64_t k) { b200q_layout L; if (b200q_make_layout(type, 4, k, &L)) return -1; return b200q_wire_row_size(L); }
int64_t b200q_plane_bytes(int type, int64_t m, int64_t k) { b200q_layout L; if (b200q_make_layout(type, m, k, &L)) return -1; return L.total_bytes; }

int b200q_repack(int type, const void * wire_dev, void * planes_dev, int64_t m, int64_t k, void * stream) {
    b200q_layout L; int rc = b200q_make_layout(type, m, k, &L);
    if (rc) return check_launch(rc, "b200q_repack");
    return check_launch(b200q_launch_repack(wire_dev, planes_dev, L, 0, (cudaStream_t)stream), "b200q_repack");
}
int b200q_unrepack(int type, const void * planes_dev, void * wire_dev, int64_t m, int64_t k, void * stream) {
    b200q_layout L; int rc = b200q_make_layout(type, m, k, &L);
    if (rc) return check_launch(rc, "b200q_unrepack");
    // the inverse pass ORs bits into the wire buffer for some types: it clears what it needs itself
    return check_launch(b200q_launch_repack(wire_dev, const_cast<void *>(planes_dev), L, 1, (cudaStream_t)stream), "b200q_unrepack");
}
int b200q_set_tensor(int type, const void * wire_host, void * planes_dev, int64_t m, int64_t k, void * stream) {
    b200q_layout L; int rc = b200q_make_layout(type, m, k, &L);
    if (rc) return check_launch(rc, "b200q_set_tensor");
    const size_t nbytes = (size_t)b200q_wire_row_size(L) * m;
    if ((rc = ensure(g_stage, nbytes))) return rc;
    cudaStream_t st = (cudaStream_t)stream; cudaError_t e;
    if ((e = cudaMemcpyAsync(g_stage.p, wire_host, nbytes, cudaMemcpyHostToDevice, st)) != cudaSuccess) return cuda_fail("set_tensor H2D", e);
    if ((rc = check_launch(b200q_launch_repack(g_stage.p, planes_dev, L, 0, st), "b200q_set_tensor"))) return rc;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail("set_tensor sync", e);
    if (g_stage.n > STAGE_KEEP) release(g_stage);
    return B200Q_OK;
}
int b200q_get_tensor(int type, const void * planes_dev, void * wire_host, int64_t m, int64_t k, void * stream) {
    b200q_layout L; int rc = b200q_make_layout(type, m, k, &L);
    if (rc) return check_launch(rc, "b200q_get_tensor");
    const size_t nbytes = (size_t)b200q_wire_row_size(L) * m;
    if ((rc = ensure(g_stage, nbytes))) return rc;
    cudaStream_t st = (cudaStream_t)stream; cudaError_t e;
    if ((rc = check_launch(b200q_launch_repack(g_stage.p, const_cast<void *>(planes_dev), L, 1, st), "b200q_get_tensor"))) return rc;
    if ((e = cudaMemcpyAsync(wire_host, g_stage.p, nbytes, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return cuda_fail("get_tensor D2H", e);
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail("get_tensor sync", e);
    if (g_stage.n > STAGE_KEEP) release(g_stage);
    return B200Q_OK;
}

// pending "next weights" hint of this thread (b200q_decode_prefetch_next): consumed by the next decode launch
static thread_local b200q_mmvq_desc g_next; static thread_local bool g_next_valid = false;
static inline void attach_next(b200q_mmvq_desc & d) { d.next = nullptr; if (g_next_valid && opt_pf()) d.next = &g_next; g_next_valid = false; }

int b200q_decode_prefetch_next(int type, int n_tensors, const void * const * W, const void * W_gate, const int64_t * m, int64_t k) {
    g_next_valid = false;
    if (n_tensors < 1 || n_tensors > B200Q_MAX_SEGS || !W || !m || (W_gate && n_tensors != 1)) return fail(B200Q_E_ARG, "b200q_decode_prefetch_next: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_decode_prefetch_next: no CUDA device");
    memset(&g_next, 0, sizeof g_next);
    g_next.type = type; g_next.n_seg = n_tensors; g_next.K = k; g_next.ncols = 1; g_next.sm_count = di.sm_count; g_next.ring = opt_ring();
    for (int i = 0; i < n_tensors; ++i) g_next.seg[i] = {W[i], i == 0 ? W_gate : nullptr, nullptr, nullptr, m[i]};
    g_next_valid = true;
    return B200Q_OK;
}

static int mmvq_cols(b200q_mmvq_desc & d, int n, int64_t x_stride, cudaStream_t st, const char * what) {
    attach_next(d);
    // the kernel is instantiated for 1/2/4/8 columns: cover n with the largest pieces
    int done = 0;
    const int64_t xs = x_stride ? x_stride : d.K;
    if (((uintptr_t)d.x & 15) || (xs & 3)) return fail(B200Q_E_ARG, "%s: activations must be 16-byte aligned with a row stride multiple of 4 floats", what);
    float * dst0[B200Q_MAX_SEGS]; for (int i = 0; i < d.n_seg; ++i) dst0[i] = d.seg[i].dst;
    const float * x0 = d.x;
    while (done < n) {
        int c = 8; while (c > n - done) c >>= 1;
        // shared memory budget: c*K int8 + c*(K/32)*8 bytes must fit in ~200 KB
        while (c > 1 && (size_t)c * d.K + (size_t)c * (d.K / 32) * 8 > 200 * 1024) c >>= 1;
        if ((size_t)c * d.K + (size_t)c * (d.K / 32) * 8 > 200 * 1024) return fail(B200Q_E_SHAPE, "%s: K=%lld too large for the mat-vec kernel", what, (long long)d.K);
        d.ncols = c; d.x = x0 + (int64_t)done * xs; d.x_stride = xs;
        for (int i = 0; i < d.n_seg; ++i) d.seg[i].dst = dst0[i] + (int64_t)done * d.seg[i].M;
        int rc = check_launch(b200q_launch_mmvq(d, st), what);
        if (rc) return rc;
        d.next = nullptr;
        done += c;
    }
    return B200Q_OK;
}

int b200q_mul_mat_vec(int type, const void * W, const float * x, float * dst, int64_t m, int64_t k, int n, int64_t x_stride,
                      const float * bias, void * stream) {
    if (!W || !x || !dst || m <= 0 || n < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_vec: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_vec: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = 1; d.seg[0] = {W, nullptr, dst, bias, m}; d.K = k; d.x = x; d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = opt_ring();
    return mmvq_cols(d, n, x_stride, (cudaStream_t)stream, "b200q_mul_mat_vec");
}
int b200q_mul_mat_vec_multi(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m, int64_t k,
                            const float * x, int n, int64_t x_stride, void * stream) {
    if (n_tensors < 1 || n_tensors > B200Q_MAX_SEGS || !W || !dst || !m || !x || n < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_multi: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_vec_multi: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = n_tensors; d.K = k; d.x = x; d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = opt_ring();
    for (int i = 0; i < n_tensors; ++i) d.seg[i] = {W[i], nullptr, dst[i], nullptr, m[i]};
    return mmvq_cols(d, n, x_stride, (cudaStream_t)stream, "b200q_mul_mat_vec_multi");
}
int b200q_fused_up_gate_vec(int type, const void * W_up, const void * W_gate, const float * x, float * dst, int64_t m, int64_t k, int n,
                            int64_t x_stride, int unary, float limit, void * stream) {
    if (!W_up || !W_gate || !x || !dst || m <= 0 || n < 1) return fail(B200Q_E_ARG, "b200q_fused_up_gate_vec: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_fused_up_gate_vec: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = 1; d.seg[0] = {W_up, W_gate, dst, nullptr, m}; d.K = k; d.x = x; d.act = unary; d.limit = limit; d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = opt_ring();
    return mmvq_cols(d, n, x_stride, (cudaStream_t)stream, "b200q_fused_up_gate_vec");
}

/* q8 hand-off between FUSED_UP_GATE and the following MUL_MAT (ffn_down), n = 1: the up/gate launch also emits its result quantised to
 * q8_1 (by the warp that completes each 32-row block), the next mat-vec bulk-copies that image instead of re-quantising per CTA. */
size_t b200q_q8_scratch_bytes(int64_t k) { return k > 0 && k % 32 == 0 ? b200q_q8_image_bytes(k) : 0; }
int b200q_q8_scratch_init(void * q8, int64_t k, void * stream) {
    if (!q8 || k <= 0 || k % 32) return fail(B200Q_E_ARG, "b200q_q8_scratch_init: bad argument");
    cudaError_t e = cudaMemsetAsync(q8, 0, b200q_q8_image_bytes(k), (cudaStream_t)stream);
    return e == cudaSuccess ? B200Q_OK : cuda_fail("b200q_q8_scratch_init", e);
}
int b200q_fused_up_gate_vec_q8(int type, const void * W_up, const void * W_gate, const float * x, float * dst, int64_t m, int64_t k,
                               int unary, float limit, void * q8_out, int * q8_produced, void * stream) {
    if (q8_produced) *q8_produced = 0;
    if (!W_up || !W_gate || !x || !dst || m <= 0) return fail(B200Q_E_ARG, "b200q_fused_up_gate_vec_q8: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_fused_up_gate_vec_q8: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = 1; d.seg[0] = {W_up, W_gate, dst, nullptr, m}; d.K = k; d.x = x; d.x_stride = k; d.ncols = 1; d.act = unary; d.limit = limit;
    d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = opt_ring();
    if (((uintptr_t)x & 15) || (k & 3)) return fail(B200Q_E_ARG, "b200q_fused_up_gate_vec_q8: activations must be 16-byte aligned");
    attach_next(d);
    if (q8_out && opt_q8()) {
        d.q8_out = q8_out;
        const int rc = b200q_launch_mmvq(d, (cudaStream_t)stream);
        if (rc == 0) { if (q8_produced) *q8_produced = 1; return B200Q_OK; }
        if (rc != -8) return check_launch(rc, "b200q_fused_up_gate_vec_q8");
        d.q8_out = nullptr;              // shape not eligible for the hand-off: plain launch
    }
    return check_launch(b200q_launch_mmvq(d, (cudaStream_t)stream), "b200q_fused_up_gate_vec_q8");
}
int b200q_mul_mat_vec_q8(int type, const void * W, const float * x, const void * q8_in, float * dst, int64_t m, int64_t k,
                         const float * bias, void * stream) {
    if (!W || !x || !dst || m <= 0) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_q8: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_vec_q8: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = 1; d.seg[0] = {W, nullptr, dst, bias, m}; d.K = k; d.x = x; d.x_stride = k; d.ncols = 1; d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = opt_ring();
    if (((uintptr_t)x & 15) || (k & 3)) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_q8: activations must be 16-byte aligned");
    attach_next(d);
    if (q8_in && opt_q8()) {
        d.q8_in = q8_in;
        const int rc = b200q_launch_mmvq(d, (cudaStream_t)stream);
        if (rc == 0) return B200Q_OK;
        if (rc != -8) return check_launch(rc, "b200q_mul_mat_vec_q8");
        d.q8_in = nullptr;
    }
    return check_launch(b200q_launch_mmvq(d, (cudaStream_t)stream), "b200q_mul_mat_vec_q8");
}

int b200q_mul_mat_vec_tp(int type, int n_tensors, const void * const * W, const void * W_gate, float * const * dst, const int64_t * m,
                         int64_t k, const float * x, int unary, float limit, const b200q_nvls_comm * comm, int reduce_in, int reduce_out, void * stream) {
    if (n_tensors < 1 || n_tensors > B200Q_MAX_SEGS || !W || !m || (W_gate && n_tensors != 1)) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_tp: bad argument");
    if ((reduce_in || reduce_out) && (!comm || !comm->ll_mc || !comm->ll_local || !comm->ll_reduced || !comm->ll_state || comm->ll_stride < 1 || comm->world_size < 2 || comm->rank >= comm->world_size
                                      || ((uintptr_t)comm->ll_mc & 15) || ((uintptr_t)comm->ll_local & 15) || ((uintptr_t)comm->ll_reduced & 15) || (comm->ll_stride & 1)))
        return fail(B200Q_E_ARG, "b200q_mul_mat_vec_tp: incomplete communicator");
    if (!reduce_in && !x) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_tp: x is NULL");
    if (!reduce_out && !dst) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_tp: dst is NULL");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_vec_tp: no CUDA device");
    b200q_mmvq_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = n_tensors; d.K = k; d.x = x; d.x_stride = k; d.ncols = 1; d.act = unary; d.limit = limit; d.sm_count = di.sm_count; d.pdl = opt_pdl(); d.ring = 1;
    for (int i = 0; i < n_tensors; ++i) d.seg[i] = {W[i], i == 0 ? W_gate : nullptr, dst ? dst[i] : nullptr, nullptr, m[i]};
    if (comm) {
        d.tp.ll_mc = (float2 *)comm->ll_mc; d.tp.ll_local = (const float2 *)comm->ll_local; d.tp.ll_red = (float2 *)comm->ll_reduced; d.tp.ll_stride = comm->ll_stride;
        d.tp.world = comm->world_size; d.tp.rank = comm->rank; d.tp.seq = (uint32_t *)comm->ll_state; d.tp.in = reduce_in != 0; d.tp.out = reduce_out != 0;
        // unicast variant (peer stores, rows of a CTA coalesced): measured SLOWER than the multicast stores at 2 GPUs (578-583 vs 626 tok/s, same box,
        // profiles/r2_tp_timeline.md) -> opt-in only
        static const int ucast = [] { const char * e = getenv("B200Q_TP_UNICAST"); return e ? atoi(e) : 0; }();
        if (ucast && comm->ll_peers && comm->world_size <= 8) {
            for (uint32_t r = 0; r < comm->world_size; ++r) {
                if (!comm->ll_peers[r] || ((uintptr_t)comm->ll_peers[r] & 15)) return fail(B200Q_E_ARG, "b200q_mul_mat_vec_tp: bad peer mapping");
                d.tp.ll_peer[r] = (float2 *)comm->ll_peers[r];
            }
        }
    }
    return check_launch(b200q_launch_mmvq(d, (cudaStream_t)stream), "b200q_mul_mat_vec_tp");
}

int b200q_reduce_sum_nvls(const float * in, float * out, int64_t n, void * mc_base, void * local_base, int64_t parity_stride,
                          void * mc_flag, const void * local_flag, uint32_t world_size, void * seq_counter, void * cta_counter, void * stream) {
    if (!in || !out || !mc_base || !local_base || !mc_flag || !local_flag || !seq_counter || !cta_counter || world_size < 2) return fail(B200Q_E_ARG, "b200q_reduce_sum_nvls: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_reduce_sum_nvls: no CUDA device");
    return check_launch(b200q_launch_allreduce_nvls(in, out, n, mc_base, local_base, parity_stride, mc_flag, local_flag, world_size, seq_counter, cta_counter,
                                                    di.sm_count, (cudaStream_t)stream), "b200q_reduce_sum_nvls");
}

int b200q_reduce_sum_nvls_bf16(const float * in, float * out_f32, void * out_bf16, int64_t n, const b200q_nvls_stage * sg, void * stream) {
    if (!in || (!out_f32 && !out_bf16) || !sg || !sg->mc_stage || !sg->local_stage || !sg->mc_flag || !sg->local_flag || !sg->state || sg->world_size < 2 || sg->rank >= sg->world_size)
        return fail(B200Q_E_ARG, "b200q_reduce_sum_nvls_bf16: bad argument");
    if (n > sg->stage_elems || (n & 7)) return fail(B200Q_E_SHAPE, "b200q_reduce_sum_nvls_bf16: n must be a multiple of 8 and fit the staging buffer");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_reduce_sum_nvls_bf16: no CUDA device");
    return check_launch(b200q_launch_allreduce_nvls_2shot(in, out_f32, out_bf16, n, sg->mc_stage, sg->local_stage, sg->mc_flag, sg->local_flag, sg->world_size, sg->rank,
                                                          sg->state, di.sm_count, (cudaStream_t)stream), "b200q_reduce_sum_nvls_bf16");
}

size_t b200q_mul_mat_workspace(int type, int64_t m, int64_t k, int64_t n) { return n <= 8 ? 0 : b200q_gemm_workspace_bytes(type, m, k, n); }

int b200q_dequantize_bf16(int type, const void * W, void * out, int64_t m, int64_t k, void * stream) {
    b200q_layout L; int rc = b200q_make_layout(type, m, k, &L);
    if (rc) return check_launch(rc, "b200q_dequantize_bf16");
    return check_launch(b200q_launch_dequant_bf16(W, L, out, (cudaStream_t)stream), "b200q_dequantize_bf16");
}
int b200q_mul_mat_gemm(int type, const void * W, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                       void * workspace, size_t workspace_bytes, void * stream) {
    if (!W || !x || !dst || !workspace || m <= 0 || n < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_gemm: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_gemm: no CUDA device");
    return check_launch(b200q_launch_gemm(type, W, x, k, dst, m, k, n, workspace, workspace_bytes, di.sm_count, opt_fused(), (cudaStream_t)stream), "b200q_mul_mat_gemm");
}
int b200q_convert_f32_bf16(const float * x, int64_t x_stride, void * out_bf16, int64_t k, int64_t n, void * stream) {
    if (!x || !out_bf16 || n < 1) return fail(B200Q_E_ARG, "b200q_convert_f32_bf16: bad argument");
    return check_launch(b200q_launch_f32_to_bf16(x, x_stride, out_bf16, k, n, (cudaStream_t)stream), "b200q_convert_f32_bf16");
}
int b200q_mul_mat_gemm_bf16(int type, const void * W, const void * x_bf16, float * dst, int64_t m, int64_t k, int64_t n,
                            void * workspace, size_t workspace_bytes, void * stream) {
    if (!W || !x_bf16 || !dst || m <= 0 || n < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_gemm_bf16: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_gemm_bf16: no CUDA device");
    return check_launch(b200q_launch_gemm_bf16x(type, W, x_bf16, dst, m, k, n, workspace, workspace_bytes, di.sm_count, opt_fused(), (cudaStream_t)stream), "b200q_mul_mat_gemm_bf16");
}
int b200q_mul_mat_gemm_multi_bf16(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m, int64_t k,
                                  const void * x_bf16, int64_t n, void * workspace, size_t workspace_bytes, void * stream) {
    if (n_tensors < 1 || n_tensors > 3 || !W || !dst || !m || !x_bf16 || n < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_gemm_multi_bf16: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_gemm_multi_bf16: no CUDA device");
    b200q_gemm_multi d; memset(&d, 0, sizeof d);
    d.type = type; d.n_seg = n_tensors; d.K = k; d.N = n; d.xb = x_bf16;
    for (int i = 0; i < n_tensors; ++i) { if (!W[i] || !dst[i] || m[i] <= 0) return fail(B200Q_E_ARG, "b200q_mul_mat_gemm_multi_bf16: bad tensor %d", i); d.W[i] = W[i]; d.dst[i] = dst[i]; d.M[i] = m[i]; }
    return check_launch(b200q_launch_gemm_multi_bf16x(d, workspace, workspace_bytes, di.sm_count, opt_fused(), (cudaStream_t)stream), "b200q_mul_mat_gemm_multi_bf16");
}
size_t b200q_mul_mat_multi_workspace(int type, int n_tensors, const int64_t * m, int64_t k, int64_t n) {
    if (n <= 8 || !m) return 0;
    int64_t mm = 0; for (int i = 0; i < n_tensors; ++i) mm = m[i] > mm ? m[i] : mm;
    return b200q_gemm_workspace_bytes(type, mm, k, n);
}
int b200q_mul_mat_multi(int type, int n_tensors, const void * const * W, float * const * dst, const int64_t * m, int64_t k,
                        const float * x, int64_t n, void * workspace, size_t workspace_bytes, void * stream) {
    if (n <= 8) return b200q_mul_mat_vec_multi(type, n_tensors, W, dst, m, k, x, (int)n, k, stream);
    if (!x || !workspace || workspace_bytes < b200q_mul_mat_multi_workspace(type, n_tensors, m, k, n)) return fail(B200Q_E_ARG, "b200q_mul_mat_multi: bad argument / workspace too small");
    int rc = b200q_convert_f32_bf16(x, k, workspace, k, n, stream); if (rc) return rc;
    const size_t off = (size_t)b200q_align_up(n * k * 2, 256);
    return b200q_mul_mat_gemm_multi_bf16(type, n_tensors, W, dst, m, k, workspace, n, (char *)workspace + off, workspace_bytes - off, stream);
}

size_t b200q_fused_up_gate_workspace(int type, int64_t m, int64_t k, int64_t n) {
    if (n <= 8) return 0;
    (void)type;     // bf16 activations + f32 up result + bf16 weight scratch (types without a fused kernel)
    return (size_t)b200q_align_up(n * k * 2, 256) + (size_t)b200q_align_up(m * n * 4, 256) + (size_t)b200q_align_up(m * k * 2, 256);
}
// x already bf16 [n][k]; workspace >= align(m*n*4) + align(m*k*2)
int b200q_fused_up_gate_gemm_bf16(int type, const void * W_up, const void * W_gate, const void * x_bf16, float * dst, void * dst_bf16,
                                  int64_t m, int64_t k, int64_t n, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream) {
    if (!W_up || !W_gate || !x_bf16 || !dst || !workspace || m <= 0 || n < 1) return fail(B200Q_E_ARG, "b200q_fused_up_gate_gemm_bf16: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_fused_up_gate_gemm_bf16: no CUDA device");
    const size_t up_bytes = (size_t)b200q_align_up(m * n * 4, 256);
    if (workspace_bytes < up_bytes) return fail(B200Q_E_ARG, "b200q_fused_up_gate_gemm_bf16: workspace too small");
    float * up_res = (float *)workspace; void * wsc = (char *)workspace + up_bytes; const size_t wsc_bytes = workspace_bytes - up_bytes;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (!b200q_gemm_epilogue_fusable(type, m, k, n, di.sm_count, opt_fused() && opt_fuse_epi() ? 2 : 0)) {
        // default: up and gate as the two segments of ONE launch (up -> workspace, gate -> dst), then the unary-mul tail in place
        b200q_gemm_multi d; memset(&d, 0, sizeof d);
        d.type = type; d.n_seg = 2; d.W[0] = W_up; d.dst[0] = up_res; d.M[0] = m; d.W[1] = W_gate; d.dst[1] = dst; d.M[1] = m; d.K = k; d.N = n; d.xb = x_bf16;
        rc = check_launch(b200q_launch_gemm_multi_bf16x(d, wsc, wsc_bytes, di.sm_count, opt_fused(), st), "b200q_fused_up_gate_gemm_bf16(up,gate)");
        if (rc) return rc;
        return check_launch(b200q_launch_mul_unary(dst, up_res, dst, dst_bf16, m * n, unary, limit, st), "b200q_fused_up_gate_gemm_bf16(unary)");
    }
    rc = check_launch(b200q_launch_gemm_bf16x(type, W_up, x_bf16, up_res, m, k, n, wsc, wsc_bytes, di.sm_count, opt_fused(), st), "b200q_fused_up_gate_gemm_bf16(up)");
    if (rc) return rc;
    if (b200q_gemm_epilogue_fusable(type, m, k, n, di.sm_count, opt_fused() && opt_fuse_epi() ? 2 : 0)) {
        // gate GEMM whose epilogue applies unary(gate) * up and (optionally) emits the bf16 operand of ffn_down
        b200q_gemm_multi d; memset(&d, 0, sizeof d);
        d.type = type; d.n_seg = 1; d.W[0] = W_gate; d.dst[0] = dst; d.mul[0] = up_res; d.dst_bf[0] = dst_bf16; d.M[0] = m; d.K = k; d.N = n; d.xb = x_bf16;
        d.act = unary; d.limit = limit;
        return check_launch(b200q_launch_gemm_multi_bf16x(d, wsc, wsc_bytes, di.sm_count, opt_fused(), st), "b200q_fused_up_gate_gemm_bf16(gate)");
    }
    rc = check_launch(b200q_launch_gemm_bf16x(type, W_gate, x_bf16, dst, m, k, n, wsc, wsc_bytes, di.sm_count, opt_fused(), st), "b200q_fused_up_gate_gemm_bf16(gate)");
    if (rc) return rc;
    return check_launch(b200q_launch_mul_unary(dst, up_res, dst, dst_bf16, m * n, unary, limit, st), "b200q_fused_up_gate_gemm_bf16(unary)");
}
int b200q_fused_up_gate(int type, const void * W_up, const void * W_gate, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                        int unary, float limit, void * workspace, size_t workspace_bytes, void * stream) {
    if (n <= 8) return b200q_fused_up_gate_vec(type, W_up, W_gate, x, dst, m, k, (int)n, k, unary, limit, stream);
    if (!x || !workspace || workspace_bytes < b200q_fused_up_gate_workspace(type, m, k, n)) return fail(B200Q_E_ARG, "b200q_fused_up_gate: bad argument / workspace too small");
    if ((m * n) % 4) return fail(B200Q_E_SHAPE, "b200q_fused_up_gate: m*n must be a multiple of 4");
    int rc;
    {   // ternary weights: both GEMMs on the int8 tensor pipe (one activation quantisation, one launch over the up and gate row tiles), then the unary-mul tail
        static const int use_i8 = [] { const char * e = getenv("B200Q_BN_INT8"); return e ? atoi(e) : 1; }();
        dev_info & di = device_info();
        const size_t up_bytes = (size_t)b200q_align_up(m * n * 4, 256);
        if (type == B200Q_TYPE_IQ2_BN && use_i8 && opt_fused() && di.ok && workspace_bytes >= up_bytes + b200q_gemm_i8_workspace_bytes(k, n)) {
            float * up_res = (float *)workspace;
            b200q_gemm_multi d; memset(&d, 0, sizeof d);
            d.type = type; d.n_seg = 2; d.W[0] = W_up; d.dst[0] = up_res; d.M[0] = m; d.W[1] = W_gate; d.dst[1] = dst; d.M[1] = m; d.K = k; d.N = n;
            rc = b200q_launch_gemm_bn_i8(d, x, k, (char *)workspace + up_bytes, workspace_bytes - up_bytes, (cudaStream_t)stream);
            if (rc == 0) return check_launch(b200q_launch_mul_unary(dst, up_res, dst, nullptr, m * n, unary, limit, (cudaStream_t)stream), "b200q_fused_up_gate(unary)");
            if (rc != -100) return check_launch(rc, "b200q_fused_up_gate(int8)");
        }
    }
    rc = b200q_convert_f32_bf16(x, k, workspace, k, n, stream); if (rc) return rc;
    const size_t off = (size_t)b200q_align_up(n * k * 2, 256);
    return b200q_fused_up_gate_gemm_bf16(type, W_up, W_gate, workspace, dst, nullptr, m, k, n, unary, limit, (char *)workspace + off, workspace_bytes - off, stream);
}
int b200q_mul_mat(int type, const void * W, const float * x, float * dst, int64_t m, int64_t k, int64_t n,
                  void * workspace, size_t workspace_bytes, void * stream) {
    if (n <= 8) return b200q_mul_mat_vec(type, W, x, dst, m, k, (int)n, k, nullptr, stream);
    return b200q_mul_mat_gemm(type, W, x, dst, m, k, n, workspace, workspace_bytes, stream);
}
/* GGML_OP_ADD of a mat-mul result with its bias (bias [m] broadcast over the n columns, nb = 1) or with a same-shape tensor (nb = n): the node as
 * its own launch, for graphs that compute it separately; inside a graph the mat-vec fuses it (bias operand of b200q_mul_mat_vec). */
int b200q_add_rows(const float * a, const float * b, float * dst, int64_t m, int64_t n, int64_t nb, void * stream) {
    if (!a || !b || !dst) return fail(B200Q_E_ARG, "b200q_add_rows: bad argument");
    return check_launch(b200q_launch_add_rows(a, b, dst, m, n, nb, (cudaStream_t)stream), "b200q_add_rows");
}
int b200q_mul_mat_id_vec(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                         int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * stream) {
    if (!W || !ids || !x || !dst || m <= 0 || n_expert < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_id_vec: bad argument");
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_id_vec: no CUDA device");
    if (((uintptr_t)x & 15) || (k & 3)) return fail(B200Q_E_ARG, "b200q_mul_mat_id_vec: activations must be 16-byte aligned");
    if (n_tokens < 1 || n_used < 1 || nb1 < 1 || n_used % nb1) return fail(B200Q_E_ARG, "b200q_mul_mat_id_vec: bad token / slot counts");
    // the quantised activation columns of a launch live in shared memory: larger batches are walked in token chunks (same kernel, the expert ids
    // never leave the device).  b200q_mul_mat_id sends larger batches of the types the grouped tcgen05 GEMM covers there instead.
    const int64_t col_bytes = (int64_t)nb1 * (k + k / 4);
    int chunk = (int)((200 * 1024) / (col_bytes > 0 ? col_bytes : 1));
    static const int forced = [] { const char * e = getenv("B200Q_MOE_CHUNK_TOKENS"); return e ? atoi(e) : 0; }();
    if (forced > 0 && forced < chunk) chunk = forced;
    if (chunk < 1) return fail(B200Q_E_SHAPE, "b200q_mul_mat_id_vec: one token's activation columns do not fit shared memory");
    for (int t0 = 0; t0 < n_tokens; t0 += chunk) {
        const int nt = n_tokens - t0 < chunk ? n_tokens - t0 : chunk;
        b200q_mmvq_id_desc d; memset(&d, 0, sizeof d);
        d.type = type; d.W = W; d.W2 = W_gate; d.ids = ids + (int64_t)t0 * n_used; d.x = x + (int64_t)t0 * nb1 * k; d.dst = dst + (int64_t)t0 * n_used * m;
        d.M = m; d.K = k; d.n_expert = n_expert; d.n_used = n_used; d.nb1 = nb1; d.n_tokens = nt;
        d.act = unary; d.limit = limit; d.sm_count = di.sm_count; d.pdl = opt_pdl();
        const int rc = check_launch(b200q_launch_mmvq_id(d, (cudaStream_t)stream), "b200q_mul_mat_id_vec");
        if (rc) return rc;
    }
    return B200Q_OK;
}
size_t b200q_mul_mat_id_workspace(int type, int64_t m, int64_t k, int n_expert, int n_used, int nb1, int n_tokens, int up_gate) {
    b200q_moe_plan_t p;
    return b200q_moe_plan(type, m, k, n_expert, n_used, nb1, n_tokens, up_gate, &p) == 0 ? p.total : 0;
}
int b200q_mul_mat_id_gemm(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                          int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream) {
    if (!W || !ids || !x || !dst || !workspace || m <= 0 || k <= 0 || n_expert < 1) return fail(B200Q_E_ARG, "b200q_mul_mat_id_gemm: bad argument");
    if (n_tokens < 1 || n_used < 1 || nb1 < 1 || n_used % nb1) return fail(B200Q_E_ARG, "b200q_mul_mat_id_gemm: bad token / slot counts");
    if (((uintptr_t)x & 15) || ((uintptr_t)workspace & 255)) return fail(B200Q_E_ARG, "b200q_mul_mat_id_gemm: x must be 16-byte and the workspace 256-byte aligned");
    b200q_moe_plan_t p;
    const int rc = b200q_moe_plan(type, m, k, n_expert, n_used, nb1, n_tokens, W_gate != nullptr, &p);
    if (rc == -1) return fail(B200Q_E_TYPE, "b200q_mul_mat_id_gemm: type %d has no grouped GEMM", type);
    if (rc) return fail(B200Q_E_SHAPE, "b200q_mul_mat_id_gemm: shape not covered by the grouped GEMM (k %% 256 == 0, n_expert <= 512)");
    if (workspace_bytes < p.total) return fail(B200Q_E_ARG, "b200q_mul_mat_id_gemm: workspace too small (%zu < %zu)", workspace_bytes, p.total);
    dev_info & di = device_info(); if (!di.ok) return fail(B200Q_E_CUDA, "b200q_mul_mat_id_gemm: no CUDA device");
    b200q_moe_desc d; memset(&d, 0, sizeof d);
    d.type = type; d.W = W; d.W_gate = W_gate; d.n_expert = n_expert; d.ids = ids; d.x = x; d.dst = dst; d.M = m; d.K = k;
    d.n_used = n_used; d.nb1 = nb1; d.n_tokens = n_tokens; d.act = unary; d.limit = limit;
    return check_launch(b200q_launch_moe_gemm(d, p, workspace, (cudaStream_t)stream), "b200q_mul_mat_id_gemm");
}
// Smallest batch (routed rows n_tokens * n_used) that takes the grouped GEMM.  Measured with scripts/moe_prefill_bench.py on a B200 at a
// 1000 W power limit (profiles/moe_prefill_b200.json, one MoE FFN layer, grouped GEMM vs mat-vec time): at 8 tokens the mat-vec kernel is
// about as fast or faster (Qwen3-30B-A3B shape, 64 rows: IQ4_NL 1.05-1.15x, Q4_K 0.84-0.92x; Mixtral-8x7B shape, 16 rows: 1.03-1.10x /
// 0.83-0.89x), at 16 tokens the grouped GEMM wins at every point (1.25-1.74x).  The crossover lies between 64 and 128 rows with 128
// experts and between 16 and 32 rows with 8 experts: max(32, n_expert) rows puts both shapes on the measured winning side.
static int64_t moe_gemm_min_rows(int n_expert) { return n_expert > 32 ? n_expert : 32; }
int b200q_mul_mat_id(int type, const void * W, const void * W_gate, int n_expert, const int32_t * ids, const float * x, float * dst,
                     int64_t m, int64_t k, int n_used, int nb1, int n_tokens, int unary, float limit, void * workspace, size_t workspace_bytes, void * stream) {
    b200q_moe_plan_t p;
    if (n_expert >= 1 && (int64_t)n_tokens * n_used >= moe_gemm_min_rows(n_expert) &&
        b200q_moe_plan(type, m, k, n_expert, n_used, nb1, n_tokens, W_gate != nullptr, &p) == 0)
        return b200q_mul_mat_id_gemm(type, W, W_gate, n_expert, ids, x, dst, m, k, n_used, nb1, n_tokens, unary, limit, workspace, workspace_bytes, stream);
    return b200q_mul_mat_id_vec(type, W, W_gate, n_expert, ids, x, dst, m, k, n_used, nb1, n_tokens, unary, limit, stream);
}
int b200q_mul_mat_host(int type, const void * W, const float * x_host, float * dst_host, int64_t m, int64_t k, int64_t n, void * stream) {
    cudaStream_t st = (cudaStream_t)stream; cudaError_t e; int rc;
    const size_t xb = (size_t)n * k * sizeof(float), yb = (size_t)n * m * sizeof(float), wsb = b200q_mul_mat_workspace(type, m, k, n);
    if ((rc = ensure(g_x, xb)) || (rc = ensure(g_y, yb)) || (wsb && (rc = ensure(g_ws, wsb)))) return rc;
    if ((e = cudaMemcpyAsync(g_x.p, x_host, xb, cudaMemcpyHostToDevice, st)) != cudaSuccess) return cuda_fail("mul_mat_host H2D", e);
    if ((rc = b200q_mul_mat(type, W, (const float *)g_x.p, (float *)g_y.p, m, k, n, g_ws.p, g_ws.n, stream))) return rc;
    if ((e = cudaMemcpyAsync(dst_host, g_y.p, yb, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return cuda_fail("mul_mat_host D2H", e);
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail("mul_mat_host sync", e);
    return B200Q_OK;
}

}  // extern "C"
