// tests/backend_ops/test_moe_prefill_backend.cpp — MoE prefill through the ggml-backend API of the plug (libggml_b200.so):
// GGML_OP_MUL_MAT_ID and GGML_OP_MOE_FUSED_UP_GATE at prefill batch sizes, computed by ggml_backend_graph_compute of the plug (whose
// dispatcher b200q_mul_mat_id sends IQ4_NL / Q4_K to the grouped tcgen05 GEMM, and keeps the mat-vec kernel for Q6_K, which it does not
// cover) and compared with the reference CPU backend through ggml_backend_compare_graph_backend: NMSE <= 5e-4, the bar of test-backend-ops.
// Inputs are quantised with ggml_quantize_chunk from fixed seeds.  Same semantics as tests/backend_ops/test_mul_mat_backend.cpp.
#include "ggml.h"
#include "ggml-alloc.h"
#include "ggml-backend.h"
#include "ggml-cuda.h"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

static double nmse(const float * a, const float * b, size_t n) {
    double e = 0, s = 0; for (size_t i = 0; i < n; ++i) { e += ((double)a[i] - b[i]) * ((double)a[i] - b[i]); s += (double)b[i] * b[i]; } return e / (s > 0 ? s : 1e-300);
}
struct cb_data { double worst = 0; int n = 0; };
static bool cmp_cb(int, ggml_tensor * t1, ggml_tensor * t2, void * ud) {
    cb_data * d = (cb_data *)ud;
    std::vector<float> a(ggml_nelements(t1)), b(ggml_nelements(t2));
    ggml_backend_tensor_get(t1, a.data(), 0, ggml_nbytes(t1)); ggml_backend_tensor_get(t2, b.data(), 0, ggml_nbytes(t2));
    const double e = nmse(a.data(), b.data(), a.size()); if (e > d->worst) d->worst = e; d->n++;
    return true;
}
static void fill_uniform(std::vector<float> & v, std::mt19937 & rng) { std::uniform_real_distribution<float> u(-1.f, 1.f); for (auto & x : v) x = u(rng); }

// n_tokens tokens, each routed to n_used distinct experts of n_expert; shared_col: one activation column per token (up/gate), else one per slot (down)
static int run_moe_case(ggml_backend_t be, ggml_backend_t cpu, ggml_type type, int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tokens,
                        bool shared_col, bool up_gate, ggml_unary_op unary, unsigned seed) {
    ggml_init_params ip = { ggml_tensor_overhead() * 16 + ggml_graph_overhead(), nullptr, true };
    ggml_context * ctx = ggml_init(ip);
    ggml_tensor * w = ggml_new_tensor_3d(ctx, type, k, m, n_expert), * g = up_gate ? ggml_new_tensor_3d(ctx, type, k, m, n_expert) : nullptr;
    ggml_tensor * x = ggml_new_tensor_3d(ctx, GGML_TYPE_F32, k, shared_col ? 1 : n_used, n_tokens);
    ggml_tensor * ids = ggml_new_tensor_2d(ctx, GGML_TYPE_I32, n_used, n_tokens);
    ggml_tensor * y = up_gate ? ggml_moe_up_gate(ctx, w, g, x, ids, unary) : ggml_mul_mat_id(ctx, w, x, ids);
    ggml_cgraph * gf = ggml_new_graph(ctx); ggml_build_forward_expand(gf, y);
    ggml_backend_buffer_t buf = ggml_backend_alloc_ctx_tensors(ctx, be);
    if (!buf) { printf("  alloc failed\n"); ggml_free(ctx); return 1; }
    std::mt19937 rng(seed);
    for (ggml_tensor * t : {w, g}) {
        if (!t) continue;
        std::vector<float> wf(ggml_nelements(t)); fill_uniform(wf, rng);
        std::vector<uint8_t> wq(ggml_nbytes(t));
        ggml_quantize_chunk(type, wf.data(), wq.data(), 0, ggml_nrows(t), k, nullptr, nullptr);
        ggml_backend_tensor_set(t, wq.data(), 0, wq.size());
    }
    std::vector<float> xf(ggml_nelements(x)); fill_uniform(xf, rng); ggml_backend_tensor_set(x, xf.data(), 0, xf.size() * sizeof(float));
    std::vector<int32_t> idv(n_used * n_tokens), perm(n_expert);
    for (int64_t t = 0; t < n_tokens; ++t) {
        for (int64_t e = 0; e < n_expert; ++e) perm[e] = (int32_t)e;
        std::shuffle(perm.begin(), perm.end(), rng);
        if (t % 3 == 0) std::swap(perm[0], *std::find(perm.begin(), perm.end(), 0));     // a crowded expert 0: several token tiles
        for (int64_t s = 0; s < n_used; ++s) idv[t * n_used + s] = perm[s];
    }
    ggml_backend_tensor_set(ids, idv.data(), 0, idv.size() * sizeof(int32_t));
    int rc = 0;
    if (!ggml_backend_supports_op(be, y)) { printf("  %-8s %s not supported\n", ggml_type_name(type), ggml_op_name(y->op)); rc = 1; }
    else {
        cb_data d; ggml_backend_compare_graph_backend(be, cpu, gf, cmp_cb, &d);
        const bool ok = d.n > 0 && d.worst <= 5e-4;
        printf("  %-8s %-18s m=%lld k=%lld experts=%lld used=%lld tokens=%lld %s%s%s: NMSE vs CPU backend %.3g -> %s\n", ggml_type_name(type), ggml_op_name(y->op),
               (long long)m, (long long)k, (long long)n_expert, (long long)n_used, (long long)n_tokens, shared_col ? "(shared column)" : "(column per slot)",
               up_gate ? " " : "", up_gate ? ggml_unary_op_name(unary) : "", d.worst, ok ? "OK" : "FAIL");
        rc = ok ? 0 : 1;
    }
    ggml_backend_buffer_free(buf); ggml_free(ctx);
    return rc;
}

int main() {
    ggml_backend_t be = ggml_backend_cuda_init(0, "pdl=1", nullptr);
    if (!be) { printf("ggml_backend_cuda_init failed (no CUDA device?)\n"); return 2; }
    ggml_backend_t cpu = ggml_backend_cpu_init(); ggml_backend_cpu_set_n_threads(cpu, 4);
    int fails = 0; unsigned seed = 5000;
    for (ggml_type t : {GGML_TYPE_IQ4_NL, GGML_TYPE_Q4_K, GGML_TYPE_Q6_K})
        for (int64_t n : {64, 512})
            for (bool shared_col : {true, false})
                for (bool up_gate : {true, false})
                    fails += run_moe_case(be, cpu, t, 256, 1024, 8, 2, n, shared_col, up_gate, GGML_UNARY_OP_SILU, ++seed);
    // many small experts (ragged M, several slots per token) and the other activations of MOE_FUSED_UP_GATE
    fails += run_moe_case(be, cpu, GGML_TYPE_IQ4_NL, 200, 512, 32, 4, 128, true, true, GGML_UNARY_OP_GELU, ++seed);
    fails += run_moe_case(be, cpu, GGML_TYPE_Q4_K, 200, 512, 32, 4, 128, false, false, GGML_UNARY_OP_SILU, ++seed);
    fails += run_moe_case(be, cpu, GGML_TYPE_Q4_K, 256, 512, 16, 2, 96, true, true, GGML_UNARY_OP_RELU, ++seed);
    printf("%s: %d failures\n", fails ? "FAILED" : "PASSED", fails);
    ggml_backend_free(be); ggml_backend_free(cpu);
    return fails ? 1 : 0;
}
