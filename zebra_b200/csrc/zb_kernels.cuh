// zb_kernels.cuh -- host-callable launchers of the sm_100a kernels (definitions in zb_kernels.cu, zb_scan.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "zb_device.cuh"
#include "zb_metrics.cuh"
#include "zb_project.cuh"
#include "zb_quadtile.cuh"

namespace zb {

#define ZB_MAX_DEPTH 96      // build never creates a node deeper than this; walkers keep a stack of this size
#define ZB_MAX_ATTEMPTS 4    // degenerate-split retries before a node is forced to be a leaf
#define ZB_MAX_TOPK 2048

// Device view of the forest + store, passed by value to kernels.
struct ForestView {
    const int4* nodes;        // {plane, left(below), right(above), leaf}
    const int* roots;         // [num_trees]
    const float* coef;        // [planes][dimp]
    const float* cst;         // [planes]
    const long long* leaf_off;  // [leaves] first member position
    const u32* leaf_len;      // [leaves] physical member count on this shard (tombstoned included)
    const u32* leaf_plan;     // [leaves] live member count over ALL shards (what tree_result sees as len)
    const u32* members;       // slots
    const float* rows;        // [slots][dimp]
    const u64* ord;           // [slots] global ordinal
    const float* row_norm;    // [slots] squared norm of the row in the canonical order (cosine)
    const u32* tomb;          // bitmask over slots
    int dimp, chunks, num_trees;
    int dim;                  // unpadded N (the scalar metrics must not fold the padding: Canberra would see 0/0)
};

struct SegDesc {      // one node under construction (build)
    long long off;    // first position in the work array (this shard)
    u32 len;          // positions on this shard
    u32 plane;        // plane slot to write
    u64 key;          // node key of the sampling spec
    u32 attempt;
    u32 pad;
};
struct Tile {         // 64 consecutive positions of one segment / leaf
    u32 seg;
    u32 count;
    long long start;
};

struct RecvSeg {      // rows of one (source rank, owned leaf) pair in the receive staging area (bucket-sharded store build)
    u64 start;
    u32 count;
    u32 leaf_seq;     // sequence number of the leaf among the leaves this rank owns in the tree being built
};

// ---- plan (tree_result control flow, lsh.rs:290-348) ----
void launch_plan(const ForestView& f, const float* d_queries, u32 nq, u32 top_k, u32 probes, u32 vpw, uint2* d_wvisits,
                 u32* d_wcounts, u32* d_overflow, u32* d_tail_list, cudaStream_t s);
// sharded plan exchange (compacted visit records, header first): pack -> ncclAllGather -> flags -> scan -> scatter -> offsets
void launch_pack_visits(u32 nwalkers, u32 vpw, const uint2* d_wvisits, const u32* d_wcounts, const u32* d_woff, u32 walker_base,
                        u32 cap, const u32* d_flag, uint4* d_out, cudaStream_t s);
void launch_own_flags(u32 G, u32 cap, size_t stride, const uint4* d_all, u32 rank, u32* d_flags, u32* d_summary, cudaStream_t s);
void launch_own_scatter(const ForestView& f, u32 G, u32 cap, size_t stride, const uint4* d_all, const u32* d_flags, const u32* d_pos, u32 vcap,
                        u32 tile_on, u32 min_rows, u32 kmax, u32* d_vleaf, u32* d_vnp, u32* d_vq, u32* d_vw, u64* d_pair_len,
                        u32* d_ent_len, u8* d_vdone, cudaStream_t s);
void launch_walker_offsets(u32 nwalkers, const u32* d_nv, u32 vcap, const u32* d_vw, u32* d_woff, cudaStream_t s);
void launch_compact_visits(const ForestView& f, u32 nwalkers, u32 vpw, const uint2* d_wvisits, const u32* d_wcounts,
                           const u32* d_woff, u32 G, u32 rank, u32 cap, u32 tile_on, u32 min_rows, u32 kmax, u32* d_vleaf,
                           u32* d_vnp, u32* d_vq, u64* d_pair_len, u32* d_ent_len, u8* d_vdone, cudaStream_t s);
void launch_plan_totals(const u32* d_flag, const u32* d_woff, u32 nwalkers, u32 cap, const u32* d_ent_off, const u64* d_pair_off,
                        const u32* d_maxcount, u64* d_out, cudaStream_t s);
// ---- scoring of (visit, member) pairs, generic path ----
void launch_score_pairs(const ForestView& f, int metric, int power, const float* d_queries, u32 nv, const u32* d_vleaf,
                        const u32* d_vq, const u64* d_pair_off, u64 total_pairs, u64* d_pair_key, cudaStream_t s);
// ---- per-visit top-n' (Q2) and per-query union/dedup/top-k (lsh.rs:557-564) ----
void launch_select_visits(const ForestView& f, u32 nv, const u32* d_vleaf, const u32* d_vnp, const u64* d_pair_off,
                          const u64* d_pair_key, const u32* d_ent_off, Entry* d_entries, const u8* d_vdone,
                          u32 top_k, int variant, cudaStream_t s);
void launch_merge_ranks(u32 nv, const u32* d_ent_off, u32 total_slots, u32 nranks, const Entry* d_gathered,
                        Entry* d_entries, u32 top_k, cudaStream_t s);
void launch_merge_queries(u32 nq, u32 num_trees, const u32* d_woff, const u32* d_ent_off, const Entry* d_entries,
                          u32 top_k, u64* d_out_ord, u64* d_out_bits, u32* d_out_counts, cudaStream_t s);
// ---- hashing / descent (lsh.rs:350-366) ----
void launch_hash(const ForestView& f, const float* d_rows, u64 n, u64* d_keys, u32* d_depths, int* d_leaves, int variant,
                 cudaStream_t s);
// ---- build (lsh.rs:192-267) ----
void launch_pick(int phase, const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work, const u64* d_ord,
                 const u64* d_exclude, u64* d_minh, u64* d_minord, int* d_slot, cudaStream_t s);
void launch_fetch_pair_rows(const SegDesc* d_segs, u32 nsegs, const int* d_slot_a, const int* d_slot_b,
                            const float* d_rows, int dimp, float* d_pair_rows, cudaStream_t s);
void launch_make_planes(const SegDesc* d_segs, u32 nsegs, const float* d_pair_rows, int dimp, float* d_coef,
                        float* d_cst, cudaStream_t s);
void launch_classify(const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work, const float* d_rows,
                     const float* d_coef, const float* d_cst, int dimp, u32* d_flags, int variant, cudaStream_t s);
void launch_seg_above(const SegDesc* d_segs, u32 nsegs, const u32* d_scan, u32* d_above, cudaStream_t s);
void launch_scatter(const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work_in, const u32* d_flags,
                    const u32* d_scan, u32* d_work_out, cudaStream_t s);
void launch_assign_leaf(const Tile* d_tiles, u32 ntiles, const u32* d_members, u32* d_slot_leaf_tree, cudaStream_t s);
// ---- mutation ----
void launch_tombstone(const u32* d_slots, u32 n, u32* d_tomb, const u32* d_slot_leaf, u64 slot_stride, int num_trees,
                      u32* d_leaf_live, u8* d_removed, cudaStream_t s);
void launch_bm_gather(u32 nleaves, const long long* d_leaf_off, const u32* d_leaf_len, const u32* d_leaf_tree, const u32* d_members,
                      const float* d_rows, const u32* d_tomb, int dimp, u64 slot_stride, float* d_bm_rows, u32* d_slot_pos,
                      u32* d_bm_tomb, cudaStream_t s);
void launch_bm_tombstone(const u32* d_slots, const u8* d_flags, u32 n, const u32* d_slot_pos, u64 slot_stride, int num_trees,
                         u32* d_bm_tomb, cudaStream_t s);
void launch_pad_rows(const float* d_src, u64 n, int dim, int dimp, float* d_dst, cudaStream_t s);
void launch_fill_u64(u64* d, u64 n, u64 v, cudaStream_t s);
void launch_iota_ord(u64* d, u64 n, u64 first, u64 stride, cudaStream_t s);
void launch_synth(float* d_out, u64 first_row, u64 row_stride, u64 n, u32 dim, u64 seed, u32 kind, cudaStream_t s);

void launch_sq_norms(const float* d_x, u64 n, int dimp, float* d_out, cudaStream_t s);
// Flat tables: sign[n][Hp] = point_is_above of every (row, plane); then the K bits of each of T tables -> key / depth / leaf.
void launch_project_flat(const float* d_rows, u64 n, const float* d_coef, const float* d_cst, int H, int dimp, u8* d_sign, int Hp,
                         cudaStream_t s);
void launch_pack_flat_keys(const u8* d_sign, u64 n, int Hp, int T, int K, u64* d_keys, u32* d_depths, int* d_leaves, cudaStream_t s);
void launch_pair_metric(int metric, int power, const float* d_a, const float* d_b, u64 n, int dim, int dimp, u64* d_out,
                        cudaStream_t s);
void launch_pair_above(const float* d_coef, const float* d_cst, const float* d_x, u64 n, int dimp, u8* d_out, cudaStream_t s);

// ---- bucket-sharded store (G > 1) ----
void launch_pack_rows(const u32* d_slots, u64 n, const float* d_rows, const u64* d_ord, const u32* d_tomb, int dimp,
                      float* d_out_rows, u64* d_out_key, cudaStream_t s);
void launch_seg_keys(const RecvSeg* d_segs, u32 nsegs, const u64* d_st_key, u64* d_sort_key, u32* d_sort_val, cudaStream_t s);
void launch_place_rows(const u32* d_perm, u64 n, const float* d_st_rows, const u64* d_st_key, int dimp, u64 base,
                       float* d_bm_rows, u64* d_bm_ord, u32* d_bm_tomb, cudaStream_t s);
void launch_iota_u32(u32* d, u64 n, u32 first, cudaStream_t s);
void launch_bm_tomb_lookup(const u64* d_ords, const u8* d_flags, u64 n, int num_trees, const u64* d_tree_base,
                           const u64* d_srt_ord, const u32* d_srt_pos, u32* d_bm_tomb, cudaStream_t s);
void launch_merge_gathered(u32 nq, u32 nslice, u32 top_k, u32 nranks, const u64* d_gathered, u64* d_out_ord, u64* d_out_bits,
                           u32* d_out_counts, cudaStream_t s);
void launch_unpack_results(const u64* d_res, u64 blk, u32 nq, u32 nslice, u32 top_k, u64* d_out_ord, u64* d_out_bits,
                           u32* d_out_counts, cudaStream_t s);
size_t sort_temp_bytes(size_t n);
void sort_pairs_u64_u32(void* d_temp, size_t temp_bytes, const u64* d_kin, u64* d_kout, const u32* d_vin, u32* d_vout, size_t n,
                        int end_bit, cudaStream_t s);

// ---- deduplicate (lsh.rs:270-288) ----
void launch_row_hash(const u32* d_slots, u64 n, const float* d_rows, int dimp, u64* d_h1, u64* d_h2, cudaStream_t s);
void launch_dup_mark(const u64* d_sorted_key, const u32* d_cand, u64 n, const u32* d_slots, const float* d_rows, int dimp,
                     u32* d_flag, u32* d_head, void* d_temp, size_t temp_bytes, u8* d_dup, cudaStream_t s);
size_t maxscan_temp_bytes(size_t n);

// cub wrappers (temp storage managed by caller)
size_t scan_temp_bytes(size_t n);
void exclusive_scan_u32(void* d_temp, size_t temp_bytes, const u32* d_in, u32* d_out, size_t n, cudaStream_t s);
void exclusive_scan_u64(void* d_temp, size_t temp_bytes, const u64* d_in, u64* d_out, size_t n, cudaStream_t s);

}  // namespace zb
