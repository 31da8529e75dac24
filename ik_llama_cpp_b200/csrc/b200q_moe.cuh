// b200q_moe.cuh — routing arithmetic of the grouped MoE prefill GEMM (GGML_OP_MUL_MAT_ID / GGML_OP_MOE_FUSED_UP_GATE).
//
// The n_tokens x n_used slots of a batch are sorted by expert (stable: slot order inside an expert) into n_rows = n_tokens * n_used rows:
//   counts[e]            rows routed to expert e (ids clamped into [0, n_expert), like the mat-vec kernel k_mmvq_id)
//   bounds[e .. e+1)     the sorted rows of expert e: bounds = exclusive scan of counts, bounds[n_expert] = n_rows
//   row_src[r]           activation column of sorted row r:  t * nb1 + (slot % nb1)
//   row_dst[r]           output row of sorted row r:         t * n_used + slot
//   tiles[i]             one {expert, col0, col_end} per BN-wide token tile of each expert (experts without rows have none)
// The GEMM walks the tile table with blockIdx.y; rows of a tile past col_end belong to the next expert (or lie beyond n_rows) and are masked.
//
// Everything here is plain arithmetic, compiled for the device (k_moe_route, b200q_moe.cu) and for the host (CPU tests: the serial
// b200q_moe_route_serial is the specification the parallel kernel reproduces).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B200Q_MOE_HD __host__ __device__ __forceinline__
#else
#define B200Q_MOE_HD inline
#endif

struct b200q_moe_tile { int expert, col0, col_end, pad; };     // 16 bytes: one int4 load in the GEMM

// a corrupt id must not address outside the expert tensor: clamp, exactly as k_mmvq_id does
B200Q_MOE_HD int b200q_moe_clamp(int id, int n_expert) { return id < 0 ? 0 : (id >= n_expert ? n_expert - 1 : id); }
B200Q_MOE_HD int b200q_moe_src_col(int t, int slot, int nb1) { return t * nb1 + slot % nb1; }
B200Q_MOE_HD int b200q_moe_dst_row(int t, int slot, int n_used) { return t * n_used + slot; }
B200Q_MOE_HD int b200q_moe_tiles_of(int count, int bn) { return (count + bn - 1) / bn; }
// host-known upper bound on the number of tiles: every expert with rows wastes less than one tile, and at most n_rows experts have rows
B200Q_MOE_HD int b200q_moe_tiles_bound(int n_rows, int n_expert, int bn) { return (n_rows + bn - 1) / bn + (n_expert < n_rows ? n_expert : n_rows); }

// bounds[0..n_expert] = exclusive scan of counts; tile_off[0..n_expert] = exclusive scan of the tile counts.  Returns the number of tiles.
B200Q_MOE_HD int b200q_moe_scan(const int * counts, int n_expert, int bn, int * bounds, int * tile_off) {
    int rows = 0, tiles = 0;
    for (int e = 0; e < n_expert; ++e) {
        bounds[e] = rows; tile_off[e] = tiles;
        rows += counts[e]; tiles += b200q_moe_tiles_of(counts[e], bn);
    }
    bounds[n_expert] = rows; tile_off[n_expert] = tiles;
    return tiles;
}
// the tile-table entries of expert e
B200Q_MOE_HD void b200q_moe_expert_tiles(int e, const int * bounds, const int * tile_off, int bn, b200q_moe_tile * tiles) {
    for (int i = tile_off[e], c = bounds[e]; i < tile_off[e + 1]; ++i, c += bn) {
        tiles[i].expert = e; tiles[i].col0 = c; tiles[i].col_end = bounds[e + 1]; tiles[i].pad = 0;
    }
}

// Serial routing: counts[n_expert], bounds[n_expert+1], tile_off[n_expert+1], row_src[n_rows], row_dst[n_rows],
// tiles[b200q_moe_tiles_bound(...)] (scratch cursor: counts is reused).  Returns the number of tiles.
B200Q_MOE_HD int b200q_moe_route_serial(const int32_t * ids, int n_tokens, int n_used, int nb1, int n_expert, int bn,
                                         int * counts, int * bounds, int * tile_off, int * row_src, int * row_dst, b200q_moe_tile * tiles) {
    const int n_rows = n_tokens * n_used;
    for (int e = 0; e < n_expert; ++e) counts[e] = 0;
    for (int s = 0; s < n_rows; ++s) ++counts[b200q_moe_clamp(ids[s], n_expert)];
    const int nt = b200q_moe_scan(counts, n_expert, bn, bounds, tile_off);
    for (int e = 0; e < n_expert; ++e) { b200q_moe_expert_tiles(e, bounds, tile_off, bn, tiles); counts[e] = 0; }
    for (int s = 0; s < n_rows; ++s) {
        const int e = b200q_moe_clamp(ids[s], n_expert), t = s / n_used, slot = s % n_used;
        const int r = bounds[e] + counts[e]++;
        row_src[r] = b200q_moe_src_col(t, slot, nb1); row_dst[r] = b200q_moe_dst_row(t, slot, n_used);
    }
    return nt;
}
