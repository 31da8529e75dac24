// Host build of the MoE routing arithmetic (ik_llama_cpp_b200/csrc/b200q_moe.cuh), for tests/test_moe_routing_host.py.
#include "../../ik_llama_cpp_b200/csrc/b200q_moe.cuh"

extern "C" {
int emul_moe_route(const int32_t * ids, int n_tokens, int n_used, int nb1, int n_expert, int bn, int * counts, int * bounds, int * tile_off,
                   int * row_src, int * row_dst, int * tiles) {
    return b200q_moe_route_serial(ids, n_tokens, n_used, nb1, n_expert, bn, counts, bounds, tile_off, row_src, row_dst, (b200q_moe_tile *)tiles);
}
int emul_moe_tiles_bound(int n_rows, int n_expert, int bn) { return b200q_moe_tiles_bound(n_rows, n_expert, bn); }
int emul_moe_clamp(int id, int n_expert) { return b200q_moe_clamp(id, n_expert); }
}
