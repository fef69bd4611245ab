// zb_scan.cuh -- the fused leaf-tile scan (the bandwidth-critical kernel of the query path).
#pragma once
#include "zb_host.h"
#include "zb_kernels.cuh"

namespace zb {

struct ScanWorkspace {
    DBuf<u32> leaf_count, leaf_start, leaf_cursor, tile_per_leaf, tile_start, order, tile_leaf, tile_first, tile_cnt;
    DBuf<u32> counters, tile_prog;
    DBuf<u64> gthr;
    // dot-product filter for L2 / L2 squared (METRIC 3 of the third-generation kernel + refine_visits_kernel)
    DBuf<float> q_n2, cand_cut;
    DBuf<u64> cand;
    DBuf<u8> cand_flag;
    bool l2_filter = false;      // in: the caller allows the filter for this batch;  filtered: the last launch used it
    bool filtered = false;
    int long_list_warps = 8;     // in: math warps per team for n' > 32 (knob long_list_warps: 8 = default, 4 = the short-list shape)
    cudaEvent_t ev2 = nullptr;   // after the second pass
    DBuf<long long> pj_off;   // project3 / exact_scan3: first row of every row range
    // exact_scan3: visits (query-major: v = q * nranges + r), entry offsets, per-query visit offsets, the ranges' usable |row|^2
    // maximum, the visits' lists and the queries' reciprocal norms
    DBuf<u32> ex_leaf, ex_np, ex_q, ex_ent_off, ex_woff;
    DBuf<float> ex_n2max;
    DBuf<Entry> ex_entries;
    DBuf<double> ex_q_rinv;
    DBuf<u8> tmp, sort_tmp;
    DBuf<u32> sort_key[2], sort_val[2];   // tile order: leaves sorted by cost
    bool launched = false;
    bool seq_launched = false;   // seq_tile_scan (scalar metrics) ran for the last batch
    u32 launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // around the tile kernel alone
    const u32* ntiles_ptr = nullptr;           // device scalar: tiles of the last launch
};

// Device view of the bucket-major store: position p of the forest's member array holds a copy of row members[p],
// so every leaf is one contiguous [len][dimp] block (the on-device replacement of the reference's per-bucket
// storage on the search path).
struct BucketMajor {
    const float* rows = nullptr;    // [positions][dimp]
    const double* rinv = nullptr;   // [positions] 1/sqrt(|row|^2), f64 (cosine only)
    const u32* tomb = nullptr;      // bit per position
    const float* n2 = nullptr;      // [positions] canonical |row|^2, f32 (L2 / L2 squared: the dot-product filter)
    const float* leaf_n2max = nullptr;  // [leaves] largest usable n2 of the leaf
    const void* tmap = nullptr;     // host copy of the CUtensorMap (128 bytes) over `rows`, box = 48 floats x 128 rows
    const void* tmap3 = nullptr;    // the same tensor with a 48 floats x 64 rows box (third-generation scan)
    u64 positions = 0;
};

// Encodes the 2-D tensor map of the bucket-major store into out_map128 (128 bytes, 64-byte aligned).
void make_row_tile_map(void* out_map128, const float* bm_rows, u64 positions, int dimp, int box_rows, int box_floats);
int tile_scan_box_floats(int generation);   // K slice of a ring stage, in floats: second / third generation kernel
// True when the tile kernel can serve this shape (top_k <= 32, query block + ring fit in shared memory).
bool tile_scan_supported(int dimp, u32 top_k);
void launch_rinv(const float* d_x, u64 n, int dimp, double* d_out, cudaStream_t s);
void launch_n2(const float* d_x, u64 n, int dimp, float* d_out, cudaStream_t s);
void launch_leaf_n2max(u32 nleaves, const long long* d_leaf_off, const u32* d_leaf_len, const float* d_n2, float* d_out, cudaStream_t s);
// Largest top_k the dot-product filter serves (its 32-entry candidate lists need slack above n').
#define ZB_L2_FILTER_MAX_K 16

// Handles every visit whose leaf holds at least `min_rows` rows: groups those visits by leaf, and for each
// (leaf, tile of <= tile_queries queries) streams the leaf's rows once through shared memory, scores them
// against all queries of the tile in the canonical order and keeps each visit's top-n' on chip.  Handled
// visits get v_done = 1, v_pair_len = 0 and their entries written; the rest is left to the generic path.
// Asynchronous on `s`; tile_scan_stats reads the counters back (and synchronises).
void tile_scan(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
               u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, u64* v_pair_len,
               u8* v_done, Entry* entries, u32 top_k, u32 min_rows, u32 tile_queries, u32 nleaves, cudaStream_t s);
// Third generation (zb_scan3_kernel.cuh; the default): tiles of up to 16 queries, 64-row stages, one accumulator lane per
// thread, distances transposed through shared memory so that one warp owns a query's list.  Same contract as tile_scan.
bool tile_scan3_supported(int dimp, u32 top_k);
void tile_scan3(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
                u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, u64* v_pair_len,
                u8* v_done, Entry* entries, u32 top_k, u32 min_rows, u32 tile_queries, u32 nleaves, cudaStream_t s);
// Flat-table projection on the same kernel skeleton: sign[n][Hp] = point_is_above of every (row, plane) (lsh.rs:39-43).
bool project3_supported(int dimp);
void project3(ScanWorkspace& ws, const float* d_rows, u64 n, const float* d_coef, const float* d_cst, int H, int dimp, u8* d_sign, int Hp,
              cudaStream_t s);
// Exact mode of the third-generation scan (zb_index_search_exact): a plain [n][dimp] store (rows, ord, tomb of `store`, bm.rinv
// / bm.n2 per row) cut into ranges of `range_rows` rows; every (range, query) pair is a visit with n' = top_k, the query tiles
// of one range are handed out back to back so that they meet the range's rows in L2.  The visits' lists are merged into the
// per-query top_k (out_*: [nq][top_k] / [nq]).  n = 0 gives empty lists.  l2_filter: L2 / L2 squared with top_k <= 16 go
// through the dot-product filter and its exact second pass.
#define ZB_EXACT_MAX_K 128   // the fused kernel's longest list
struct ExactPlan {
    u32 range_rows = 0;   // rows per range (a multiple of the 64-row stage)
    u64 chunk = 0;        // queries per exact_scan3 call
};
// Range length and query chunk for n rows (the largest row count over all shards) and a batch of nq queries: enough tiles for
// every team, visit arrays + entries + candidate lists + per_query_bytes x chunk within budget_bytes (at least one query).
ExactPlan exact_plan(u64 n, u64 nq, int dimp, u32 top_k, bool l2_filter, u64 per_query_bytes, u64 budget_bytes);
void exact_scan3(ScanWorkspace& ws, const ForestView& store, const BucketMajor& bm, u64 n, u32 metric, const float* d_q, u32 nq,
                 u32 range_rows, u32 top_k, bool l2_filter, u64* out_ord, u64* out_bits, u32* out_counts, cudaStream_t s);
void tile_scan_stats(ScanWorkspace& ws, cudaStream_t s, u64* tile_visits, u64* tile_pairs, u64* moved_bytes, float* kernel_ms,
                     u32* tiles, u64* unique_bytes, u64* flagged_visits = nullptr, u64* refined_rows = nullptr, float* refine_ms = nullptr);

// The scalar metrics (zb_metric 3..11): every visit with pairs to score, grouped by leaf into (leaf, <= 8 queries) tiles;
// one thread folds a row against the tile's queries and writes the keys into the gather path's pair_key layout
// (pair_key[v_pair_off[v] + member]); select_visits_kernel then takes each visit's top-n'.  v_pair_off holds nv + 1 offsets.
bool seq_tile_scan_supported(int dimp);
void seq_tile_scan(ScanWorkspace& ws, const ForestView& f, u32 metric, int power, const float* d_q, u32 nv, const u32* v_leaf,
                   const u32* v_q, const u64* v_pair_off, u64* pair_key, u32 nleaves, int prefetch_lines, cudaStream_t s);
// Cosine / L2 visits the fused kernel does not take (n' > 32): the same grouping, a quad scores 4 rows x 4 queries in the
// canonical order (zb_quadtile.cuh), keys into pair_key.  Use a ScanWorkspace of its own (the fused kernel's statistics live
// in the other one until the end of the batch).  Statistics through seq_tile_scan_stats.
bool quad_tile_scan_supported(int dimp);
void quad_tile_scan(ScanWorkspace& ws, const ForestView& f, u32 metric, const float* d_q, u32 nv, const u32* v_leaf, const u32* v_q,
                    const u64* v_pair_off, u64* pair_key, u32 nleaves, cudaStream_t s);
void seq_tile_scan_stats(ScanWorkspace& ws, cudaStream_t s, u64* moved_bytes, float* kernel_ms, u32* tiles);

}  // namespace zb
