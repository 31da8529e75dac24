// ggml_b200_backend.cpp — the drop-in boundary at the ggml-backend level (SURVEY.md §8b).
//
// Implements the reference's backend vtable (struct ggml_backend_i, ggml/src/ggml-backend-impl.h:81-130) and buffer vtables
// (:18-51) on top of libb200q.so, and exports the C symbols of ggml/include/ggml-cuda.h:24-46 under their original names.
// graph_compute owns the hot path: GGML_OP_MUL_MAT on block-quantized src0 (2-D and batched), GGML_OP_FUSED_UP_GATE, the look-ahead
// fusions of ggml_cuda_mul_mat_q (Q,K,V sharing src1; a trailing bias ADD, ggml-cuda.cu:2573-2601) and the q8_1 hand-off from
// FUSED_UP_GATE to the following MUL_MAT (ffn_down).  Every other op is reported as unsupported (supports_op == false): this library is the
// quantized-mat-mul backend; the pass-through kernels (norm, rope, attention ...) of a full llama graph are outside SURVEY §8a.
// graph_compute never allocates or synchronises once warm: scratch comes from a grow-only pool sized at first use (capture-safe afterwards).
// Compiled against the reference's headers where they lie (-I/root/reference/ggml/include -I.../ggml/src); nothing is copied.
#include "ggml.h"
#include "ggml-backend.h"
#include "ggml-backend-impl.h"
#include "ggml-cuda.h"      // the reference's own header: the prototypes this library implements
#include "b200q.h"

#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#define B200_MAX_DEVICES 16

static ggml_log_callback g_log_cb = nullptr; static void * g_log_ud = nullptr;
static void b200_log(enum ggml_log_level lvl, const char * fmt, ...) {
    char buf[512]; va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (g_log_cb) g_log_cb(lvl, buf, g_log_ud); else fputs(buf, stderr);
}
// abort-on-error convention of the reference (CUDA_CHECK -> GGML_ABORT, ggml-cuda.cu:135-145)
#define B200_CUDA_CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { b200_log(GGML_LOG_LEVEL_ERROR, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); GGML_ABORT("CUDA error"); } } while (0)
#define B200Q_CHECK(x) do { int rc_ = (x); if (rc_ != 0) { b200_log(GGML_LOG_LEVEL_ERROR, "b200q error %d: %s at %s:%d\n", rc_, b200q_last_error(), __FILE__, __LINE__); GGML_ABORT("b200q error"); } } while (0)

// ------------------------------------------------------------------------------------------------------------------
// buffers
// ------------------------------------------------------------------------------------------------------------------
struct b200_buft_ctx { int device; std::string name; };
struct b200_buffer_ctx { int device; void * base; };

static bool b200_tensor_is_repacked(const ggml_tensor * t) {
    // quantized weight matrices are stored in the plane layout (ik_llama_cpp_b200/csrc/b200q_types.cuh)
    return ggml_is_quantized(t->type) && b200q_type_supported(t->type) && ggml_is_contiguous(t) && t->view_src == nullptr && b200q_plane_bytes(t->type, t->ne[1], t->ne[0]) > 0;
}

GGML_CALL static const char * b200_buffer_get_name(ggml_backend_buffer_t) { return "B200"; }
GGML_CALL static bool b200_buffer_is_ours(ggml_backend_buffer_t b) { return b->iface.get_name == b200_buffer_get_name; }   // identity idiom of ggml-cuda.cu:607-609
GGML_CALL static void b200_buffer_free(ggml_backend_buffer_t buffer) {
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; cudaSetDevice(c->device); cudaFree(c->base); delete c;
}
GGML_CALL static void * b200_buffer_get_base(ggml_backend_buffer_t buffer) { return ((b200_buffer_ctx *)buffer->context)->base; }
static size_t b200_alloc_size(const ggml_tensor * t);
GGML_CALL static void b200_buffer_init_tensor(ggml_backend_buffer_t buffer, ggml_tensor * t) {
    // zero the bytes the allocation has beyond the wire size (plane alignment gaps): kernels never read them, but a state dump / compare should
    // see deterministic memory (the reference zeroes its row padding here too, ggml-cuda.cu:621-639)
    if (t->view_src != nullptr || !b200_tensor_is_repacked(t)) return;
    const size_t have = b200_alloc_size(t), wire = ggml_nbytes(t);
    if (have > wire) {
        b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
        B200_CUDA_CHECK(cudaMemsetAsync((char *)t->data + wire, 0, have - wire, cudaStreamPerThread)); B200_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
    }
}
GGML_CALL static void b200_buffer_memset_tensor(ggml_backend_buffer_t buffer, ggml_tensor * t, uint8_t v, size_t off, size_t size) {
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    B200_CUDA_CHECK(cudaMemsetAsync((char *)t->data + off, v, size, cudaStreamPerThread)); B200_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
}
GGML_CALL static void b200_buffer_set_tensor(ggml_backend_buffer_t buffer, ggml_tensor * t, const void * data, size_t off, size_t size) {
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    if (b200_tensor_is_repacked(t)) {
        GGML_ASSERT(off == 0 && size == ggml_nbytes(t) && "quantized tensors are uploaded whole (they are re-laid-out on the device)");
        // 3-D tensors (MoE experts [K, M, E]): every [M x K] matrix is re-laid-out on its own, matrices are b200q_plane_bytes(M, K) apart
        const int64_t nmat = t->ne[2] * t->ne[3]; const size_t wire_mat = ggml_nbytes(t) / (size_t)nmat, dev_mat = (size_t)b200q_plane_bytes(t->type, t->ne[1], t->ne[0]);
        for (int64_t e = 0; e < nmat; ++e)
            B200Q_CHECK(b200q_set_tensor(t->type, (const char *)data + e * wire_mat, (char *)t->data + e * dev_mat, t->ne[1], t->ne[0], cudaStreamPerThread));
        return;
    }
    B200_CUDA_CHECK(cudaMemcpyAsync((char *)t->data + off, data, size, cudaMemcpyHostToDevice, cudaStreamPerThread));
    B200_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
}
GGML_CALL static void b200_buffer_get_tensor(ggml_backend_buffer_t buffer, const ggml_tensor * t, void * data, size_t off, size_t size) {
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    if (b200_tensor_is_repacked(t)) {
        GGML_ASSERT(off == 0 && size == ggml_nbytes(t));
        const int64_t nmat = t->ne[2] * t->ne[3]; const size_t wire_mat = ggml_nbytes(t) / (size_t)nmat, dev_mat = (size_t)b200q_plane_bytes(t->type, t->ne[1], t->ne[0]);
        for (int64_t e = 0; e < nmat; ++e)      // original GGUF bytes, bit-for-bit
            B200Q_CHECK(b200q_get_tensor(t->type, (const char *)t->data + e * dev_mat, (char *)data + e * wire_mat, t->ne[1], t->ne[0], cudaStreamPerThread));
        return;
    }
    B200_CUDA_CHECK(cudaMemcpyAsync(data, (const char *)t->data + off, size, cudaMemcpyDeviceToHost, cudaStreamPerThread));
    B200_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
}
static size_t b200_alloc_size(const ggml_tensor * t) {
    size_t n = ggml_nbytes(t);
    if (b200_tensor_is_repacked(t)) { const int64_t pb = b200q_plane_bytes(t->type, t->ne[1], t->ne[0]) * t->ne[2] * t->ne[3]; if (pb > (int64_t)n) n = (size_t)pb; }
    return n;
}
GGML_CALL static bool b200_buffer_cpy_tensor(ggml_backend_buffer_t buffer, const ggml_tensor * src, ggml_tensor * dst) {
    if (!src->buffer || !b200_buffer_is_ours(src->buffer)) return false;       // host sources go through set_tensor
    if (src->type != dst->type || ggml_nbytes(src) != ggml_nbytes(dst) || b200_alloc_size(src) != b200_alloc_size(dst)) return false;    // same layout on both sides only
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    B200_CUDA_CHECK(cudaMemcpyAsync(dst->data, src->data, b200_alloc_size(src), cudaMemcpyDeviceToDevice, cudaStreamPerThread));
    B200_CUDA_CHECK(cudaStreamSynchronize(cudaStreamPerThread));
    return true;
}
GGML_CALL static void b200_buffer_clear(ggml_backend_buffer_t buffer, uint8_t v) {
    b200_buffer_ctx * c = (b200_buffer_ctx *)buffer->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    B200_CUDA_CHECK(cudaMemset(c->base, v, buffer->size));
}
static const ggml_backend_buffer_i b200_buffer_iface = {
    /* get_name */ b200_buffer_get_name, /* free_buffer */ b200_buffer_free, /* get_base */ b200_buffer_get_base, /* init_tensor */ b200_buffer_init_tensor,
    /* memset_tensor */ b200_buffer_memset_tensor, /* set_tensor */ b200_buffer_set_tensor, /* get_tensor */ b200_buffer_get_tensor,
    /* cpy_tensor */ b200_buffer_cpy_tensor, /* clear */ b200_buffer_clear, /* reset */ nullptr,
};

GGML_CALL static const char * b200_buft_get_name(ggml_backend_buffer_type_t buft) { return ((b200_buft_ctx *)buft->context)->name.c_str(); }
GGML_CALL static ggml_backend_buffer_t b200_buft_alloc(ggml_backend_buffer_type_t buft, size_t size) {
    b200_buft_ctx * bc = (b200_buft_ctx *)buft->context;
    if (cudaSetDevice(bc->device) != cudaSuccess) return nullptr;
    void * p = nullptr; size = size < 1 ? 1 : size;
    if (cudaMalloc(&p, size) != cudaSuccess) { cudaGetLastError(); b200_log(GGML_LOG_LEVEL_ERROR, "%s: allocating %.2f MiB on device %d failed\n", __func__, size / 1048576.0, bc->device); return nullptr; }
    return ggml_backend_buffer_init(buft, b200_buffer_iface, new b200_buffer_ctx{bc->device, p}, size);
}
GGML_CALL static size_t b200_buft_alignment(ggml_backend_buffer_type_t) { return 256; }     // plane offsets are 256-byte aligned
GGML_CALL static size_t b200_buft_alloc_size(ggml_backend_buffer_type_t, const ggml_tensor * t) { return b200_alloc_size(t); }
GGML_CALL static bool b200_buft_is_host(ggml_backend_buffer_type_t) { return false; }
static const ggml_backend_buffer_type_i b200_buft_iface = { b200_buft_get_name, b200_buft_alloc, b200_buft_alignment, /* get_max_size */ nullptr, b200_buft_alloc_size, b200_buft_is_host };

// pinned host buffer type (ggml-cuda.cu:1408-1520)
GGML_CALL static const char * b200_host_buffer_name(ggml_backend_buffer_t) { return "B200_Host"; }
GGML_CALL static void b200_host_buffer_free(ggml_backend_buffer_t buffer) { cudaFreeHost(buffer->context); }
GGML_CALL static const char * b200_host_buft_name(ggml_backend_buffer_type_t) { return "B200_Host"; }
GGML_CALL static ggml_backend_buffer_t b200_host_buft_alloc(ggml_backend_buffer_type_t buft, size_t size) {
    void * p = nullptr;
    if (cudaMallocHost(&p, size < 1 ? 1 : size) != cudaSuccess) { cudaGetLastError(); return ggml_backend_buft_alloc_buffer(ggml_backend_cpu_buffer_type(), size); }
    ggml_backend_buffer_t b = ggml_backend_cpu_buffer_from_ptr(p, size);
    b->buft = buft; b->iface.get_name = b200_host_buffer_name; b->iface.free_buffer = b200_host_buffer_free;
    return b;
}

// ------------------------------------------------------------------------------------------------------------------
// backend
// ------------------------------------------------------------------------------------------------------------------
struct b200_backend_ctx {
    int device; std::string name; cudaStream_t stream = nullptr; void * ws = nullptr; size_t ws_size = 0; const void * model = nullptr;
    std::vector<void *> retired;    // outgrown scratch blocks: kernels already enqueued may still use them -> freed in synchronize() / free()
    void * q8 = nullptr; int64_t q8_k = 0;     // q8_1 hand-off scratch FUSED_UP_GATE -> MUL_MAT (b200q_q8_scratch_*)
    // Scratch for one op.  Grow-only: a larger request allocates a new block (stream-ordered use of the old one stays valid, it is retired, not
    // freed) -> no synchronisation and, once the largest shape has been seen, no allocation inside graph_compute (CUDA-graph capture safe).
    void * workspace(size_t n) {
        if (n > ws_size) {
            if (ws) retired.push_back(ws);
            const size_t want = n + n / 4;
            B200_CUDA_CHECK(cudaMalloc(&ws, want)); ws_size = want;
        }
        return ws;
    }
    void * q8_scratch(int64_t k) {
        if (k != q8_k) {
            if (q8) retired.push_back(q8);
            B200_CUDA_CHECK(cudaMalloc(&q8, b200q_q8_scratch_bytes(k))); q8_k = k;
            B200Q_CHECK(b200q_q8_scratch_init(q8, k, stream));
        }
        return q8;
    }
    void release_retired() { for (void * p : retired) cudaFree(p); retired.clear(); }
};
static ggml_guid_t b200_guid() { static ggml_guid g = {0xb2, 0x00, 0x51, 0x0a, 0x71, 0x63, 0x67, 0x65, 0x6e, 0x30, 0x35, 0x2d, 0x71, 0x6d, 0x6d, 0x01}; return &g; }

GGML_CALL static const char * b200_backend_name(ggml_backend_t b) { return ((b200_backend_ctx *)b->context)->name.c_str(); }
GGML_CALL static void b200_backend_free(ggml_backend_t b) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; cudaSetDevice(c->device);
    if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    if (c->ws) cudaFree(c->ws);
    if (c->q8) cudaFree(c->q8);
    c->release_retired();
    delete c; delete b;
}
GGML_CALL static ggml_backend_buffer_type_t b200_backend_default_buft(ggml_backend_t b) { return ggml_backend_cuda_buffer_type(((b200_backend_ctx *)b->context)->device); }
GGML_CALL static void b200_backend_synchronize(ggml_backend_t b) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; B200_CUDA_CHECK(cudaSetDevice(c->device)); B200_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    c->release_retired();
}
// asynchronous tensor access on the backend stream (ggml_backend_cuda_set/get_tensor_async, ggml-cuda.cu:4280-4297); quantized weights go through
// the synchronous buffer path (they are re-laid-out on upload)
GGML_CALL static void b200_backend_set_tensor_async(ggml_backend_t b, ggml_tensor * t, const void * data, size_t off, size_t size) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    if (b200_tensor_is_repacked(t)) { B200_CUDA_CHECK(cudaStreamSynchronize(c->stream)); t->buffer->iface.set_tensor(t->buffer, t, data, off, size); return; }
    B200_CUDA_CHECK(cudaMemcpyAsync((char *)t->data + off, data, size, cudaMemcpyHostToDevice, c->stream));
}
GGML_CALL static void b200_backend_get_tensor_async(ggml_backend_t b, const ggml_tensor * t, void * data, size_t off, size_t size) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    if (b200_tensor_is_repacked(t)) { B200_CUDA_CHECK(cudaStreamSynchronize(c->stream)); t->buffer->iface.get_tensor(t->buffer, t, data, off, size); return; }
    B200_CUDA_CHECK(cudaMemcpyAsync(data, (const char *)t->data + off, size, cudaMemcpyDeviceToHost, c->stream));
}
GGML_CALL static bool b200_backend_cpy_tensor_async(ggml_backend_t bsrc, ggml_backend_t bdst, const ggml_tensor * src, ggml_tensor * dst) {
    if (!ggml_backend_is_cuda(bsrc) || !ggml_backend_is_cuda(bdst) || !src->buffer || !dst->buffer || !b200_buffer_is_ours(src->buffer) || !b200_buffer_is_ours(dst->buffer)) return false;
    if (ggml_is_quantized(src->type) || ggml_nbytes(src) != ggml_nbytes(dst)) return false;       // weights are not copied between devices on this path
    b200_backend_ctx * cs = (b200_backend_ctx *)bsrc->context; b200_backend_ctx * cd = (b200_backend_ctx *)bdst->context;
    B200_CUDA_CHECK(cudaSetDevice(cs->device));
    if (cs->device == cd->device) B200_CUDA_CHECK(cudaMemcpyAsync(dst->data, src->data, ggml_nbytes(dst), cudaMemcpyDeviceToDevice, cs->stream));
    else B200_CUDA_CHECK(cudaMemcpyPeerAsync(dst->data, cd->device, src->data, cs->device, ggml_nbytes(dst), cs->stream));
    if (bsrc != bdst) {     // the destination stream must observe the copy (same scheme as ggml-cuda.cu:4330-4345: record on src, wait on dst)
        cudaEvent_t ev; B200_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        B200_CUDA_CHECK(cudaEventRecord(ev, cs->stream)); B200_CUDA_CHECK(cudaSetDevice(cd->device)); B200_CUDA_CHECK(cudaStreamWaitEvent(cd->stream, ev, 0));
        B200_CUDA_CHECK(cudaEventDestroy(ev));
    }
    return true;
}
// events (ggml-cuda.cu:5218-5272)
GGML_CALL static ggml_backend_event_t b200_event_new(ggml_backend_t b) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; if (cudaSetDevice(c->device) != cudaSuccess) return nullptr;
    cudaEvent_t ev; if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    return new ggml_backend_event{ b, ev };
}
GGML_CALL static void b200_event_free(ggml_backend_event_t e) { cudaEventDestroy((cudaEvent_t)e->context); delete e; }
GGML_CALL static void b200_event_record(ggml_backend_event_t e) { b200_backend_ctx * c = (b200_backend_ctx *)e->backend->context; B200_CUDA_CHECK(cudaEventRecord((cudaEvent_t)e->context, c->stream)); }
GGML_CALL static void b200_event_wait(ggml_backend_t b, ggml_backend_event_t e) {
    if (!ggml_backend_is_cuda(e->backend)) GGML_ABORT("b200: event of a foreign backend");
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; B200_CUDA_CHECK(cudaStreamWaitEvent(c->stream, (cudaEvent_t)e->context, 0));
}
GGML_CALL static void b200_event_synchronize(ggml_backend_event_t e) { B200_CUDA_CHECK(cudaEventSynchronize((cudaEvent_t)e->context)); }

static int32_t b200_op_param_i32(const ggml_tensor * t, int i) { int32_t v; memcpy(&v, (const char *)t->op_params + i * sizeof(int32_t), sizeof v); return v; }
static int b200_unary(int ggml_unary) {
    switch (ggml_unary) { case GGML_UNARY_OP_SILU: return B200Q_UNARY_SILU; case GGML_UNARY_OP_GELU: return B200Q_UNARY_GELU; case GGML_UNARY_OP_RELU: return B200Q_UNARY_RELU;
                          case GGML_UNARY_OP_SWIGLU_OAI: return B200Q_UNARY_SWIGLU_OAI; default: return -1; }
}
// src0 must be a WHOLE quantized tensor living in one of our buffers: only those are stored in the device layout (b200_tensor_is_repacked).
// A view into a quantized tensor (a row slice of a merged wqkv ...) addresses wire-byte offsets inside a plane-layout allocation: refuse it,
// the scheduler then keeps that node on the backend that owns a wire-format copy.
static bool b200_weight_ok(const ggml_tensor * w) {
    return w && b200_tensor_is_repacked(w) && w->buffer && b200_buffer_is_ours(w->buffer) && w->ne[3] == 1 &&
           w->ne[0] % ggml_blck_size(w->type) == 0 && w->ne[0] % 32 == 0 && b200q_plane_bytes(w->type, w->ne[1], w->ne[0]) > 0;
}
// MUL_MAT: w [K, M, E?] x [K, N, B2, B3] -> dst [M, N, B2, B3]; 2-D, or batched with w broadcast over the batch (ne02 == 1) or one weight matrix per
// batch entry (ne02 == ne12, ne03 == 1)
static bool b200_can_mul_mat(const ggml_tensor * w, const ggml_tensor * x, const ggml_tensor * dst) {
    if (!b200_weight_ok(w) || !x || x->type != GGML_TYPE_F32 || !ggml_is_contiguous(x) || dst->type != GGML_TYPE_F32 || !ggml_is_contiguous(dst)) return false;
    if (w->ne[0] != x->ne[0]) return false;
    if (!(w->ne[2] == 1 || (w->ne[2] == x->ne[2] && x->ne[3] == 1))) return false;
    return true;
}
GGML_CALL static bool b200_backend_supports_op(ggml_backend_t, const ggml_tensor * op) {
    switch (op->op) {
        case GGML_OP_NONE: case GGML_OP_RESHAPE: case GGML_OP_VIEW: case GGML_OP_PERMUTE: case GGML_OP_TRANSPOSE: return true;
        case GGML_OP_MUL_MAT: return b200_can_mul_mat(op->src[0], op->src[1], op);
        case GGML_OP_ADD:       // the bias of a mat-mul result ([M] broadcast over the columns) or a same-shape f32 add, on our buffers
            return op->type == GGML_TYPE_F32 && op->src[0] && op->src[1] && op->src[0]->type == GGML_TYPE_F32 && op->src[1]->type == GGML_TYPE_F32 &&
                   ggml_is_contiguous(op) && ggml_is_contiguous(op->src[0]) && ggml_is_contiguous(op->src[1]) && ggml_are_same_shape(op, op->src[0]) &&
                   op->src[1]->ne[0] == op->ne[0] && (ggml_nelements(op->src[1]) == op->ne[0] || ggml_are_same_shape(op, op->src[1]));
        case GGML_OP_MUL_MAT_ID: case GGML_OP_MOE_FUSED_UP_GATE: {
            // MoE: expert ids resolved on the device; large batches of the types the grouped GEMM covers take it, others are walked in token chunks by the mat-vec kernel
            const bool ug = op->op == GGML_OP_MOE_FUSED_UP_GATE;
            const ggml_tensor * w = op->src[0]; const ggml_tensor * g = ug ? op->src[1] : nullptr; const ggml_tensor * x = op->src[ug ? 2 : 1]; const ggml_tensor * ids = op->src[ug ? 3 : 2];
            if (!w || !x || !ids || (ug && (!g || g->type != w->type || !ggml_are_same_shape(g, w) || op->src[4] || op->src[5] || b200_unary(b200_op_param_i32(op, 0)) < 0))) return false;
            if (!b200_weight_ok(w) || (g && !b200_weight_ok(g)) || x->type != GGML_TYPE_F32 || !ggml_is_contiguous(x) || ids->type != GGML_TYPE_I32 || !ggml_is_contiguous(ids)) return false;
            if (op->type != GGML_TYPE_F32 || !ggml_is_contiguous(op) || w->ne[0] != x->ne[0] || x->ne[3] != 1 || ids->ne[1] != x->ne[2] || ids->ne[0] % x->ne[1]) return false;
            return x->ne[1] * (w->ne[0] + w->ne[0] / 4) <= 200 * 1024;      // one token's columns must fit
        }
        case GGML_OP_FUSED_UP_GATE:
            return op->src[0] && op->src[1] && !op->src[3] && !op->src[4] && op->src[0]->type == op->src[1]->type && op->src[2] && op->src[2]->ne[2] * op->src[2]->ne[3] == 1 &&
                   op->src[0]->ne[2] == 1 && op->src[1]->ne[2] == 1 && b200_can_mul_mat(op->src[0], op->src[2], op) &&
                   b200_can_mul_mat(op->src[1], op->src[2], op) && b200_unary(b200_op_param_i32(op, 0)) >= 0 &&
                   (op->src[2]->ne[1] <= 8 || (op->src[0]->ne[1] * op->src[2]->ne[1]) % 4 == 0);
        default: return false;     // no silent CPU detour inside graph_compute: unsupported ops are refused up front
    }
}
GGML_CALL static enum ggml_status b200_backend_graph_compute(ggml_backend_t b, ggml_cgraph * cgraph) {
    b200_backend_ctx * c = (b200_backend_ctx *)b->context; B200_CUDA_CHECK(cudaSetDevice(c->device));
    const ggml_tensor * q8_from = nullptr;      // FUSED_UP_GATE node whose result is also available as a q8_1 image in c->q8
    for (int i = 0; i < cgraph->n_nodes; ++i) {
        ggml_tensor * node = cgraph->nodes[i];
        switch (node->op) {
            case GGML_OP_NONE: case GGML_OP_RESHAPE: case GGML_OP_VIEW: case GGML_OP_PERMUTE: case GGML_OP_TRANSPOSE: break;
            case GGML_OP_MUL_MAT: {
                const ggml_tensor * w = node->src[0]; const ggml_tensor * x = node->src[1];
                GGML_ASSERT(b200_can_mul_mat(w, x, node));
                const int64_t m = w->ne[1], k = w->ne[0], n = x->ne[1];
                const int64_t nbatch = x->ne[2] * x->ne[3];
                if (nbatch > 1) {       // batched / broadcast MUL_MAT: one launch per batch entry (src0 broadcast over the batch or one matrix per entry)
                    const size_t wstride = (size_t)b200q_plane_bytes(w->type, m, k);
                    for (int64_t bi = 0; bi < nbatch; ++bi) {
                        const char * W = (const char *)w->data + (w->ne[2] > 1 ? (size_t)bi * wstride : 0);
                        const size_t need = b200q_mul_mat_workspace(w->type, m, k, n);
                        void * ws = need ? c->workspace(need) : nullptr;
                        B200Q_CHECK(b200q_mul_mat(w->type, W, (const float *)x->data + bi * n * k, (float *)node->data + bi * n * m, m, k, n, ws, need, c->stream));
                    }
                    break;
                }
                // q8_1 hand-off (n = 1): the previous node was the FUSED_UP_GATE that produced x and emitted its q8 image
                if (n == 1 && q8_from == x) {
                    B200Q_CHECK(b200q_mul_mat_vec_q8(w->type, w->data, (const float *)x->data, c->q8, (float *)node->data, m, k, nullptr, c->stream));
                    q8_from = nullptr;
                    break;
                }
                // a trailing bias ADD (dst = mul_mat + bias[M], ggml-cuda.cu:2590-2600) rides in the mat-vec epilogue
                if (n <= 8 && i + 1 < cgraph->n_nodes) {
                    ggml_tensor * ad = cgraph->nodes[i + 1];
                    if (ad->op == GGML_OP_ADD && ad->src[0] == node && ad->src[1] && ad->src[1]->type == GGML_TYPE_F32 && ggml_is_contiguous(ad->src[1]) &&
                        ggml_nelements(ad->src[1]) == m && ad->type == GGML_TYPE_F32 && ggml_is_contiguous(ad) && ad->src[1]->buffer && b200_buffer_is_ours(ad->src[1]->buffer)) {
                        // both nodes are written: the plain product into node->data, the biased one into the ADD node
                        B200Q_CHECK(b200q_mul_mat_vec(w->type, w->data, (const float *)x->data, (float *)node->data, m, k, (int)n, k, nullptr, c->stream));
                        B200Q_CHECK(b200q_mul_mat_vec(w->type, w->data, (const float *)x->data, (float *)ad->data, m, k, (int)n, k, (const float *)ad->src[1]->data, c->stream));
                        ++i;
                        break;
                    }
                }
                // look-ahead fusion of ggml_cuda_mul_mat_q (ggml-cuda.cu:2573-2601): following MUL_MAT nodes that share src1 (Q,K,V)
                // and the weight type join this launch; every node's data is still written
                const void * W[3] = {w->data}; float * D[3] = {(float *)node->data}; int64_t M[3] = {m}; int nt = 1;
                while (nt < 3 && i + 1 < cgraph->n_nodes) {
                    const ggml_tensor * nx = cgraph->nodes[i + 1];
                    if (nx->op != GGML_OP_MUL_MAT || nx->src[1] != x || !nx->src[0] || nx->src[0]->type != w->type || !b200_can_mul_mat(nx->src[0], x, nx) || nx->src[0]->ne[2] != 1) break;
                    if (n <= 8 && (nx->src[0]->ne[1] & 1)) break;            // the multi-tensor mat-vec walks row pairs
                    W[nt] = nx->src[0]->data; D[nt] = (float *)nx->data; M[nt] = nx->src[0]->ne[1]; ++nt; ++i;
                }
                if (nt > 1 && (n > 8 || !(m & 1))) {
                    const size_t need = b200q_mul_mat_multi_workspace(w->type, nt, M, k, n);
                    void * ws = need ? c->workspace(need) : nullptr;
                    B200Q_CHECK(b200q_mul_mat_multi(w->type, nt, W, D, M, k, (const float *)x->data, n, ws, need, c->stream));
                } else {
                    for (int j = 0; j < nt; ++j) {
                        const size_t need = b200q_mul_mat_workspace(w->type, M[j], k, n);
                        void * ws = need ? c->workspace(need) : nullptr;
                        B200Q_CHECK(b200q_mul_mat(w->type, W[j], (const float *)x->data, D[j], M[j], k, n, ws, need, c->stream));
                    }
                }
            } break;
            case GGML_OP_ADD: {
                const ggml_tensor * a0 = node->src[0]; const ggml_tensor * a1 = node->src[1];
                const int64_t m = node->ne[0], n = ggml_nelements(node) / m, nb = ggml_nelements(a1) / m;
                B200Q_CHECK(b200q_add_rows((const float *)a0->data, (const float *)a1->data, (float *)node->data, m, n, nb, c->stream));
            } break;
            case GGML_OP_MUL_MAT_ID: case GGML_OP_MOE_FUSED_UP_GATE: {
                const bool ug = node->op == GGML_OP_MOE_FUSED_UP_GATE;
                const ggml_tensor * w = node->src[0]; const ggml_tensor * g = ug ? node->src[1] : nullptr; const ggml_tensor * x = node->src[ug ? 2 : 1]; const ggml_tensor * ids = node->src[ug ? 3 : 2];
                float limit = 0.0f; if (ug) memcpy(&limit, (const char *)node->op_params + sizeof(int32_t), sizeof(float));
                // decode-sized batches: the mat-vec kernel; larger batches of the covered types: the grouped GEMM (b200q_mul_mat_id dispatches)
                const int n_expert = (int)w->ne[2], n_used = (int)ids->ne[0], nb1 = (int)x->ne[1], n_tokens = (int)x->ne[2];
                const size_t need = b200q_mul_mat_id_workspace(w->type, w->ne[1], w->ne[0], n_expert, n_used, nb1, n_tokens, ug);
                void * ws = need ? c->workspace(need) : nullptr;
                B200Q_CHECK(b200q_mul_mat_id(w->type, w->data, g ? g->data : nullptr, n_expert, (const int32_t *)ids->data, (const float *)x->data, (float *)node->data,
                                             w->ne[1], w->ne[0], n_used, nb1, n_tokens, ug ? b200_unary(b200_op_param_i32(node, 0)) : 0, limit, ws, need, c->stream));
            } break;
            case GGML_OP_FUSED_UP_GATE: {
                const ggml_tensor * up = node->src[0]; const ggml_tensor * gate = node->src[1]; const ggml_tensor * x = node->src[2];
                float limit = 0.0f; memcpy(&limit, (const char *)node->op_params + sizeof(int32_t), sizeof(float));
                const int unary = b200_unary(b200_op_param_i32(node, 0));
                // n = 1 and the next node is the MUL_MAT that consumes this result (ffn_down): quantise it once, here, in the kernel's tail
                if (x->ne[1] == 1 && i + 1 < cgraph->n_nodes && up->ne[1] % 64 == 0) {
                    const ggml_tensor * nx = cgraph->nodes[i + 1];
                    if (nx->op == GGML_OP_MUL_MAT && nx->src[1] == node && b200_can_mul_mat(nx->src[0], node, nx) && nx->src[0]->ne[2] == 1) {
                        int produced = 0;
                        B200Q_CHECK(b200q_fused_up_gate_vec_q8(up->type, up->data, gate->data, (const float *)x->data, (float *)node->data, up->ne[1], up->ne[0], unary, limit,
                                                               c->q8_scratch(up->ne[1]), &produced, c->stream));
                        q8_from = produced ? node : nullptr;
                        break;
                    }
                }
                const size_t need = b200q_fused_up_gate_workspace(up->type, up->ne[1], up->ne[0], x->ne[1]);
                void * ws = need ? c->workspace(need) : nullptr;
                B200Q_CHECK(b200q_fused_up_gate(up->type, up->data, gate->data, (const float *)x->data, (float *)node->data, up->ne[1], up->ne[0],
                                                x->ne[1], unary, limit, ws, need, c->stream));
            } break;
            default:
                b200_log(GGML_LOG_LEVEL_ERROR, "%s: op %s not supported by the B200 quantized-mat-mul backend\n", __func__, ggml_op_name(node->op));
                return GGML_STATUS_FAILED;
        }
    }
    return GGML_STATUS_SUCCESS;     // asynchronous w.r.t. the host, like ggml_backend_cuda_graph_compute (ggml-cuda.cu:4687)
}
GGML_CALL static bool b200_backend_supports_buft(ggml_backend_t b, ggml_backend_buffer_type_t buft) {
    if (buft->iface.get_name != b200_buft_get_name) return false;
    return ((b200_buft_ctx *)buft->context)->device == ((b200_backend_ctx *)b->context)->device;
}
GGML_CALL static bool b200_backend_offload_op(ggml_backend_t, const ggml_tensor *) { return false; }

static const ggml_backend_i b200_backend_iface = {
    /* get_name */ b200_backend_name, /* free */ b200_backend_free, /* get_default_buffer_type */ b200_backend_default_buft,
    /* set_tensor_async */ b200_backend_set_tensor_async, /* get_tensor_async */ b200_backend_get_tensor_async, /* cpy_tensor_async */ b200_backend_cpy_tensor_async,
    /* synchronize */ b200_backend_synchronize,
    /* graph_plan_create */ nullptr, /* graph_plan_free */ nullptr, /* graph_plan_update */ nullptr, /* graph_plan_compute */ nullptr,
    /* graph_compute */ b200_backend_graph_compute, /* supports_op */ b200_backend_supports_op, /* supports_buft */ b200_backend_supports_buft,
    /* offload_op */ b200_backend_offload_op, /* event_new */ b200_event_new, /* event_free */ b200_event_free, /* event_record */ b200_event_record,
    /* event_wait */ b200_event_wait, /* event_synchronize */ b200_event_synchronize,
};

// ------------------------------------------------------------------------------------------------------------------
// exported C ABI (names and meaning of ggml/include/ggml-cuda.h:24-46)
// ------------------------------------------------------------------------------------------------------------------
extern "C" {
GGML_API GGML_CALL int ggml_backend_cuda_get_device_count(void) { int n = b200q_device_count(); return n > B200_MAX_DEVICES ? B200_MAX_DEVICES : n; }
GGML_API GGML_CALL ggml_backend_buffer_type_t ggml_backend_cuda_buffer_type(int device) {
    static std::mutex mu; std::lock_guard<std::mutex> lk(mu);
    static ggml_backend_buffer_type types[B200_MAX_DEVICES]; static bool init = false;
    if (device < 0 || device >= ggml_backend_cuda_get_device_count()) return nullptr;
    if (!init) { for (int i = 0; i < B200_MAX_DEVICES; ++i) types[i] = { b200_buft_iface, new b200_buft_ctx{i, "B200" + std::to_string(i)} }; init = true; }
    return &types[device];
}
GGML_API GGML_CALL ggml_backend_buffer_type_t ggml_backend_cuda_split_buffer_type(const float *) {
    // One process per GPU in this design: tensor-parallel shards are ordinary device tensors of each rank (ik_llama_cpp_b200/tp.py applies the
    // reference's split rules to the wire bytes) and GGML_OP_REDUCE is the NVLS kernel family of libb200q (b200q_reduce_sum_nvls[_bf16], fused
    // multimem.red mat-vec).  The reference's single-process multi-device split buffer (ggml-cuda.cu:805-1406) is NOT provided: say so instead
    // of silently placing everything on device 0 (a caller asking for -sm row/graph in ONE process must use the reference's CUDA backend).
    b200_log(GGML_LOG_LEVEL_ERROR, "%s: single-process split buffers are not provided by the B200 quantized-mat-mul backend (one process per GPU)\n", __func__);
    return nullptr;
}
GGML_API GGML_CALL ggml_backend_buffer_type_t ggml_backend_cuda_host_buffer_type(void) {
    static ggml_backend_buffer_type t = { { b200_host_buft_name, b200_host_buft_alloc, ggml_backend_cpu_buffer_type()->iface.get_alignment, nullptr,
                                            ggml_backend_cpu_buffer_type()->iface.get_alloc_size, ggml_backend_cpu_buffer_type()->iface.is_host }, nullptr };
    return &t;
}
GGML_API GGML_CALL void ggml_backend_cuda_get_device_description(int device, char * description, size_t n) {
    cudaDeviceProp p; if (cudaGetDeviceProperties(&p, device) == cudaSuccess) snprintf(description, n, "%s", p.name); else snprintf(description, n, "unknown");
}
GGML_API GGML_CALL void ggml_backend_cuda_get_device_memory(int device, size_t * free_, size_t * total) {
    cudaSetDevice(device); if (cudaMemGetInfo(free_, total) != cudaSuccess) { *free_ = 0; *total = 0; }
}
GGML_API GGML_CALL bool ggml_backend_cuda_register_host_buffer(void * buffer, size_t size) { return cudaHostRegister(buffer, size, cudaHostRegisterPortable | cudaHostRegisterReadOnly) == cudaSuccess; }
GGML_API GGML_CALL void ggml_backend_cuda_unregister_host_buffer(void * buffer) { cudaHostUnregister(buffer); }
GGML_API GGML_CALL void ggml_backend_cuda_log_set_callback(ggml_log_callback cb, void * ud) { g_log_cb = cb; g_log_ud = ud; }
GGML_API GGML_CALL void ggml_backend_cuda_invalidate_graphs(const void *) {}     // no cached CUDA graphs inside this backend
GGML_API GGML_CALL bool ggml_backend_is_cuda(ggml_backend_t backend) { return backend != nullptr && ggml_guid_matches(backend->guid, b200_guid()); }
GGML_API GGML_CALL ggml_backend_t ggml_backend_cuda_init(int device, const void * params, const void * model) {
    if (device < 0 || device >= ggml_backend_cuda_get_device_count()) { b200_log(GGML_LOG_LEVEL_ERROR, "%s: invalid device %d\n", __func__, device); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    if (params) {   // "k=v,k=v" like ggml_cuda_parse_params (ggml-cuda.cu:5339-5389); unknown keys are ignored like unknown features
        std::string s((const char *)params); size_t pos = 0;
        while (pos < s.size()) {
            size_t e = s.find(',', pos); if (e == std::string::npos) e = s.size();
            std::string kv = s.substr(pos, e - pos); size_t eq = kv.find('=');
            if (eq != std::string::npos) b200q_set_option(kv.substr(0, eq).c_str(), atoi(kv.c_str() + eq + 1));
            pos = e + 1;
        }
    }
    b200_backend_ctx * c = new b200_backend_ctx{device, "B200" + std::to_string(device)}; c->model = model;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
    return new ggml_backend{ b200_guid(), b200_backend_iface, c };
}
GGML_CALL static ggml_backend_t b200_reg_init(const char *, void * user_data) { return ggml_backend_cuda_init((int)(intptr_t)user_data, nullptr, nullptr); }
GGML_API GGML_CALL int ggml_backend_cuda_reg_devices(void) {
    const int n = ggml_backend_cuda_get_device_count();
    for (int i = 0; i < n; ++i) { char name[64]; snprintf(name, sizeof name, "B200%d", i); ggml_backend_register(name, b200_reg_init, ggml_backend_cuda_buffer_type(i), (void *)(intptr_t)i); }
    return n;
}
}
