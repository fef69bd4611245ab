// zb_index.cu -- the index object behind the C ABI of include/zebra_b200.h.
//
// Host side of the hot path: owns the device-resident vector store and forest, drives the kernels of
// zb_kernels.cu / zb_scan.cu on one CUDA stream, and (when sharded) the NCCL exchanges.  It mirrors
// LSHIndex<N> of /root/reference/src/database/index/lsh.rs:145-566 (new :162, add :440, remove :473,
// clear :506, search :544, no_vectors :398, no_trees :407).  There is no CPU compute path in this file:
// every dot product, distance, sign test, partition and top-k runs in a CUDA kernel.
#include <algorithm>
#include <chrono>
#include <mutex>
#include <unordered_map>

#include "zb_host.h"
#include "zb_kernels.cuh"
#include "zb_scan.cuh"

namespace zb {
size_t g_device_bytes = 0;
thread_local std::string t_last_error;  // declared in zb_host.h (zb_interchange.cpp reports through it too)

struct Id16 {
    uint64_t hi, lo;
    bool operator==(const Id16& o) const { return hi == o.hi && lo == o.lo; }
};
struct Id16Hash {
    size_t operator()(const Id16& k) const { return (size_t)mix64(k.hi ^ mix64(k.lo)); }
};
static inline uint64_t load_be64(const uint8_t* p) {
    uint64_t v = 0;
    for (int i = 0; i < 8; ++i) v = (v << 8) | p[i];
    return v;
}
static inline void store_be64(uint8_t* p, uint64_t v) {
    for (int i = 7; i >= 0; --i) {
        p[i] = (uint8_t)v;
        v >>= 8;
    }
}

__global__ void remap_leaves_kernel(int* leaves, u64 n, const int* __restrict__ table) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) leaves[i] = table[leaves[i]];
}
__global__ void count_live_kernel(const u32* __restrict__ members, const long long* __restrict__ leaf_off,
                                  const u32* __restrict__ leaf_len, const u32* __restrict__ tomb, u32 nleaves,
                                  u32* __restrict__ leaf_live) {
    u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nleaves) return;
    u32 c = 0;
    const u32* m = members + leaf_off[l];
    for (u32 i = 0; i < leaf_len[l]; ++i) c += tomb_test(tomb, m[i]) ? 0u : 1u;
    leaf_live[l] = c;
}

struct BSeg {  // a node under construction
    u64 key;
    int depth, node, tree;
    long long off;
    u32 len;
    u64 glen;
    u32 attempt;
};

}  // namespace zb

using namespace zb;

struct zb_index {
    std::mutex mu;
    zb_options opt{};
    int dim = 0, dimp = 0, chunks = 0, T = 0, device = 0;
    u32 G = 1, rank = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8]{};
    Nccl nccl;
    bool comm_ready = false;
    u64 epoch_ms = 0;

    // ---- vector store (device resident, slot order) ----
    DBuf<float> rows;
    DBuf<u64> ord;
    DBuf<float> row_norm;
    DBuf<u32> tomb;
    DBuf<u32> slot_leaf;  // [T][slot_stride]
    u64 slot_stride = 0;
    u64 n_slots = 0, n_live = 0, total_rows = 0;
    std::vector<u64> h_ord;
    std::vector<uint8_t> h_tomb;
    int id_mode = 0;  // 0 unknown, 1 minted, 2 caller supplied
    std::vector<Id16> ids_by_ordinal;
    std::unordered_map<Id16, u64, Id16Hash> ordinal_by_id;

    // ---- forest: host mirror of the structure, device copies of everything ----
    std::vector<int4> h_nodes;
    std::vector<int> h_roots;
    u64 n_planes = 0;
    std::vector<long long> h_leaf_off;
    std::vector<u32> h_leaf_len, h_leaf_cap;
    std::vector<u64> h_leaf_key;
    std::vector<int> h_leaf_depth, h_leaf_node, h_leaf_tree;
    u64 members_used = 0;
    std::vector<u32> h_members;
    bool h_members_valid = false;
    bool built = false;
    // flat tables (zb_index_load_flat): every node at depth d of tree t uses plane t * flat_bits + d, so hashing is a dense
    // projection (zb_project.cuh).  Valid while the forest is the one that was loaded (a leaf split adds nodes).
    u32 flat_bits = 0;
    size_t flat_nodes = 0;
    DBuf<u8> pj_sign;
    DBuf<int4> d_nodes;
    DBuf<int> d_roots;
    DBuf<float> d_coef, d_cst;
    DBuf<long long> d_leaf_off;
    DBuf<u32> d_leaf_len, d_leaf_live, d_leaf_plan, d_members;
    DBuf<int> d_leaf_export;
    bool export_table_valid = false;

    // ---- bucket-major store (search path): position p of the member array holds a copy of row members[p] ----
    DBuf<float> bm_rows;
    DBuf<double> bm_rinv, q_rinv;
    DBuf<u32> w_tail;                   // plan walk: [0] count, then the walkers set aside for the tail kernel
    DBuf<float> bm_n2, bm_leaf_n2max;   // L2 / L2 squared: canonical |row|^2 per position, its usable maximum per leaf (the dot-product filter)
    int filter_backoff = 0;             // batches the filter sits out after one in which too many visits had to be rescanned exactly
    DBuf<u32> bm_tomb, slot_pos, d_leaf_tree;
    alignas(64) unsigned char bm_tmap[128];
    alignas(64) unsigned char bm_tmap3[128];
    bool bm_valid = false, bm_failed = false;
    u64 bm_positions = 0;
    // bucket-sharded layout (G > 1): leaf l lives, whole, on rank l % G; positions are tree-major, then leaf, then ordinal
    DBuf<long long> d_bm_off;   // [leaves] first position of the leaf here
    DBuf<u32> d_bm_len;         // [leaves] rows of the leaf here (0: another rank owns it)
    DBuf<u64> bm_ord;           // [positions] ordinal of the row at a position
    DBuf<u32> d_iota;           // [positions] identity "member" list: the scan view addresses rows by position
    DBuf<u64> srt_ord;          // per tree region: ordinals ascending ...
    DBuf<u32> srt_pos;          // ... and the position each one sits at (delete -> tombstone lookup)
    DBuf<u64> d_tree_base, rm_ords;
    std::vector<u64> h_tree_base;
    DBuf<u64> loc_results;      // this rank's per-query top-k over the leaves it owns: [ord nq*k | bits nq*k]
    DBuf<u64> res_all;          // finished query slices of all ranks

    // ---- workspaces ----
    DBuf<u8> cub_tmp;
    DBuf<u32> w_counts, w_off, w_flag, w_loc_off, v_w, x_flags, x_pos;
    DBuf<uint4> x_send, x_all;  // sharded plan exchange: [header | visit records] of this rank / of every rank
    u32 x_cap = 0;              // records per rank in an exchange block (grows on demand, kept between batches)
    DBuf<float> q_all;          // sliced search: the query slices of all ranks
    // Peer-memory exchange of the query slices (knob p2p_queries): every rank maps every other rank's batch buffer (CUDA IPC)
    // and PUSHES its slice into all of them with device-to-device copies over NVLink; the visit-record allgather that follows
    // is the barrier (a rank enters it only after its own pushes completed).  NCCL's allgather stays as the fallback.
    struct PeerQ {
        float* mine = nullptr;              // cudaMalloc'd (IPC needs a plain allocation, not the stream-ordered pool)
        u64 cap = 0;                        // floats
        std::vector<float*> peer;           // [G] mapped pointers (peer[rank] == mine)
        bool failed = false;
        static const int NS = 4;            // side streams: the pushes to different peers run on different copy engines
        cudaStream_t stream[NS] = {};
        cudaEvent_t fork = nullptr, done[NS] = {};
    } pq;
    DBuf<u64> plan_totals;
    DBuf<uint2> w_visits;
    u32 vpw = 32;  // slots per walker in the visit plan: 1 header + up to vpw - 1 visits (grows on demand)
    DBuf<u32> v_leaf, v_np, v_q, v_ent_len, v_ent_off;
    DBuf<u64> v_pair_len, v_pair_off, pair_key;
    DBuf<u8> v_done;
    DBuf<Entry> entries, gathered;
    DBuf<float> q_stage, r_stage, hash_in;
    // zb_index_search_prefetch: up to two announced uploads, staged on their own stream
    struct Prefetch {
        DBuf<float> buf;
        const float* host = nullptr;
        u64 rows = 0, seq = 0;
        cudaEvent_t done = nullptr;
    } pf[2];
    cudaStream_t copy_stream = nullptr;
    u64 pf_seq = 0;
    DBuf<u64> o_ord, o_bits, h_keys;
    DBuf<u32> o_counts, o_counts2, h_depths, rm_slots;
    DBuf<int> h_leaves;
    DBuf<u8> rm_flags;
    HBuf<u8> pin;
    // build workspaces
    DBuf<u32> b_work[2], b_flags, b_scan, b_above;
    DBuf<Tile> b_tiles;
    DBuf<SegDesc> b_segs;
    DBuf<u64> b_minh, b_minord, b_excl;
    DBuf<int> b_slot_a, b_slot_b;
    DBuf<float> b_pair_rows;
    ScanWorkspace scan_ws;
    ScanWorkspace pj_ws;  // flat-table projection (project3)
    ScanWorkspace qt_ws;  // keys-only tile scan of the visits the fused kernel leaves (cosine / L2, n' > 32)
    // exact search (zb_index_search_exact*): its own scan workspace; per-slot side arrays of the raw store, valid while
    // ex_gen == store_gen (every path that appends or replaces rows bumps store_gen); local / gathered lists of a sharded call
    ScanWorkspace ex_ws;
    u64 store_gen = 0, ex_gen = ~0ull;
    DBuf<u32> ex_iota, ex_counts;
    DBuf<double> ex_rinv;
    DBuf<float> ex_n2;
    DBuf<u64> ex_loc, ex_gath, ex_nmax;

    // ---- knobs / stats ----
    int64_t p_tile_min_rows = 64, p_tile_queries = 0, p_use_tile_scan = 1, p_hash_variant = 0, p_classify_variant = 0, p_seq_tile = 1, p_seq_prefetch = 0, p_flat_project = 1, p_quad_tile = 1, p_select_variant = 1, p_scan_gen = 3, p_bm_stage_mb = 2048, p_single_exchange = 1, p_p2p_queries = 1, p_l2_filter = 1, p_plan_tail = 1, p_exact_budget_mb = 256;
    zb_stats st{};

    ForestView view() const {
        ForestView f;
        f.nodes = d_nodes.p;
        f.roots = d_roots.p;
        f.coef = d_coef.p;
        f.cst = d_cst.p;
        f.leaf_off = d_leaf_off.p;
        f.leaf_len = d_leaf_len.p;
        f.leaf_plan = G > 1 ? d_leaf_plan.p : d_leaf_live.p;
        f.members = d_members.p;
        f.rows = rows.p;
        f.ord = ord.p;
        f.row_norm = row_norm.p;
        f.tomb = tomb.p;
        f.dimp = dimp;
        f.dim = dim;
        f.chunks = chunks;
        f.num_trees = T;
        return f;
    }
    // What the scoring kernels read leaves from.  Unsharded: the forest's own member lists.  Sharded: the bucket-major
    // store of the leaves this rank owns, addressed by position (members = identity, ordinals / tombstones per position).
    ForestView scan_view() const {
        ForestView f = view();
        if (G > 1) {
            f.leaf_off = d_bm_off.p;
            f.leaf_len = d_bm_len.p;
            f.members = d_iota.p;
            f.rows = bm_rows.p;
            f.ord = bm_ord.p;
            f.tomb = bm_tomb.p;
            f.row_norm = nullptr;
        }
        return f;
    }
    // ZB_TRACE=1: sub-phase times of every search call (CUDA events on the index's stream), printed by rank 0
    bool trace_on = getenv("ZB_TRACE") != nullptr;
    bool trace_all = getenv("ZB_TRACE") != nullptr && atoi(getenv("ZB_TRACE")) >= 2;   // every rank prints (one line per call: fprintf is atomic enough)
    std::vector<std::pair<const char*, cudaEvent_t>> trace_ev;
    size_t trace_n = 0;
    void trace_mark(const char* what) {
        if (!trace_on) return;
        if (trace_n == trace_ev.size()) {
            cudaEvent_t e;
            ZB_CUDA(cudaEventCreate(&e));
            trace_ev.push_back({what, e});
        }
        trace_ev[trace_n].first = what;
        ZB_CUDA(cudaEventRecord(trace_ev[trace_n++].second, stream));
    }
    void trace_dump() {
        if (!trace_on || trace_n < 2) { trace_n = 0; return; }
        sync();
        if (rank == 0 || trace_all) {  // one write per call, so the lines of concurrent ranks do not interleave
            std::string line = fmt("[zb trace r%u]", rank);
            for (size_t i = 1; i < trace_n; ++i) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, trace_ev[i - 1].second, trace_ev[i].second);
                line += fmt(" %s %.3f |", trace_ev[i].first, ms);
            }
            line += "\n";
            fputs(line.c_str(), stderr);
        }
        trace_n = 0;
    }
    void sync() { ZB_CUDA(cudaStreamSynchronize(stream)); }
    void use_device() { ZB_CUDA(cudaSetDevice(device)); }
    void scan_tmp(size_t n) {
        size_t need = scan_temp_bytes(n);
        cub_tmp.ensure(need);
    }
    bool owns(u64 ordinal) const { return G <= 1 || ordinal % G == rank; }
    u64 slot_of(u64 ordinal) const { return G <= 1 ? ordinal : ordinal / G; }

    // ---------------------------------------------------------------- ids
    Id16 mint(u64 ordinal) const {
        // UUIDv7 layout: 48-bit ms timestamp (the index epoch) | ver 7 | ordinal[63:52] | var 10 | ordinal[51:46]
        // | ordinal[45:0] << 10.  Byte order == ordinal order.
        uint64_t hi = (epoch_ms << 16) | 0x7000ull | ((ordinal >> 52) & 0xFFFull);
        uint64_t lo = (0x2ull << 62) | (((ordinal >> 46) & 0x3Full) << 56) | ((ordinal & ((1ull << 46) - 1)) << 10);
        return Id16{hi, lo};
    }
    bool unmint(const Id16& id, u64* ordinal) const {
        if ((id.hi >> 16) != (epoch_ms & 0xFFFFFFFFFFFFull) || ((id.hi >> 12) & 0xF) != 7 || (id.lo >> 62) != 2 ||
            (id.lo & 0x3FF))
            return false;
        *ordinal = ((id.hi & 0xFFFull) << 52) | (((id.lo >> 56) & 0x3Full) << 46) | ((id.lo >> 10) & ((1ull << 46) - 1));
        return true;
    }
    void id_of(u64 ordinal, uint8_t* out16) const {
        Id16 id = id_mode == 2 ? (ordinal < ids_by_ordinal.size() ? ids_by_ordinal[ordinal] : Id16{~0ull, ~0ull})
                               : mint(ordinal);
        store_be64(out16, id.hi);
        store_be64(out16 + 8, id.lo);
    }
    bool ordinal_of(const uint8_t* id16, u64* ordinal) const {
        Id16 id{load_be64(id16), load_be64(id16 + 8)};
        if (id_mode == 2) {
            auto it = ordinal_by_id.find(id);
            if (it == ordinal_by_id.end()) return false;
            *ordinal = it->second;
            return true;
        }
        return unmint(id, ordinal) && *ordinal < total_rows;
    }

    // ---------------------------------------------------------------- store
    void reserve_slots(u64 need) {
        if (need <= slot_stride) return;
        u64 ncap = slot_stride ? slot_stride + slot_stride / 2 : need;
        if (ncap < need) ncap = need;
        ncap = (ncap + 31) & ~31ull;
        rows.ensure(ncap * (u64)dimp, n_slots * (u64)dimp, stream, true);
        ord.ensure(ncap, n_slots, stream, true);
        row_norm.ensure(ncap, n_slots, stream, true);
        size_t old_words = tomb.cap;
        // + 3: the fused scan's exact mode reads three words from the first word of every 64-row block
        tomb.ensure(ncap / 32 + 3, (n_slots + 31) / 32, stream, true);
        (void)old_words;
        // slot_leaf is [T][stride]: re-stride
        DBuf<u32> nsl;
        nsl.ensure(ncap * (u64)T, 0, stream, true);
        if (slot_leaf.p && n_slots)
            ZB_CUDA(cudaMemcpy2DAsync(nsl.p, ncap * 4, slot_leaf.p, slot_stride * 4, n_slots * 4, T, cudaMemcpyDeviceToDevice,
                                      stream));
        sync();
        std::swap(nsl.p, slot_leaf.p);
        std::swap(nsl.cap, slot_leaf.cap);
        slot_stride = ncap;
    }
    // Append n_local rows already on the device (stride `src_stride` floats, dim floats used) with the given ordinals.
    void append_rows_device(const float* d_src, u64 src_stride, u64 n_local, const u64* ordinals) {
        if (!n_local) return;
        reserve_slots(n_slots + n_local);
        float* dst = rows.p + n_slots * (u64)dimp;
        if (dimp == dim) {
            ZB_CUDA(cudaMemcpy2DAsync(dst, (size_t)dimp * 4, d_src, src_stride * 4, (size_t)dim * 4, n_local,
                                      cudaMemcpyDeviceToDevice, stream));
        } else {
            ZB_REQUIRE(src_stride == (u64)dim, ZB_ERR_INVALID, "strided device rows need dim %% 16 == 0");
            launch_pad_rows(d_src, n_local, dim, dimp, dst, stream);
        }
        ZB_CUDA(cudaMemcpyAsync(ord.p + n_slots, ordinals, n_local * 8, cudaMemcpyHostToDevice, stream));
        if (opt.metric == ZB_METRIC_COSINE) launch_sq_norms(dst, n_local, dimp, row_norm.p + n_slots, stream);
        // clear tombstone bits of the new slots (word granular: new words zeroed, shared first word bits are already 0)
        u64 w0 = (n_slots + 31) / 32, w1 = (n_slots + n_local + 31) / 32;
        if (n_slots == 0) w0 = 0;
        if (w1 > w0) ZB_CUDA(cudaMemsetAsync(tomb.p + w0, 0, (w1 - w0) * 4, stream));
        sync();
        h_ord.insert(h_ord.end(), ordinals, ordinals + n_local);
        h_tomb.resize(h_tomb.size() + n_local, 0);
        n_slots += n_local;
        n_live += n_local;
        ++store_gen;
    }
    // exact search: identity member list, and per slot 1/sqrt(|row|^2) (cosine) or canonical |row|^2 (L2, L2 squared)
    void ensure_exact_side() {
        if (ex_gen == store_gen) return;
        const u64 n = n_slots ? n_slots : 1;
        ex_iota.ensure(n);
        launch_iota_u32(ex_iota.p, n_slots, 0u, stream);
        if (opt.metric == ZB_METRIC_COSINE) {
            ex_rinv.ensure(n);
            launch_rinv(rows.p, n_slots, dimp, ex_rinv.p, stream);
        } else {
            ex_n2.ensure(n);
            launch_n2(rows.p, n_slots, dimp, ex_n2.p, stream);
        }
        ex_gen = store_gen;
    }

    // ---------------------------------------------------------------- forest upload helpers
    void upload_structure() {
        size_t nn = h_nodes.size(), nl = h_leaf_off.size();
        d_nodes.ensure(nn ? nn : 1);
        d_roots.ensure(T);
        d_leaf_off.ensure(nl ? nl : 1);
        d_leaf_len.ensure(nl ? nl : 1);
        if (nn) ZB_CUDA(cudaMemcpyAsync(d_nodes.p, h_nodes.data(), nn * sizeof(int4), cudaMemcpyHostToDevice, stream));
        ZB_CUDA(cudaMemcpyAsync(d_roots.p, h_roots.data(), (size_t)T * 4, cudaMemcpyHostToDevice, stream));
        if (nl) {
            ZB_CUDA(cudaMemcpyAsync(d_leaf_off.p, h_leaf_off.data(), nl * 8, cudaMemcpyHostToDevice, stream));
            ZB_CUDA(cudaMemcpyAsync(d_leaf_len.p, h_leaf_len.data(), nl * 4, cudaMemcpyHostToDevice, stream));
        }
        sync();
        export_table_valid = false;
        bm_valid = false;
    }
    // (Re)build the bucket-major store after the forest or the row set changed.  Only forests whose leaves can reach
    // the tile kernel's minimum size get one; an allocation failure degrades to the generic gather path.
    // Whether the batch may use the fused leaf-tile kernel at all is the CALLER's decision (knobs use_tile_scan /
    // tile_min_rows are looked at per search call, search_device): this function only answers "is there a store".
    bool ensure_bucket_major() {
        if (bm_valid) return true;
        if (G > 1) return ensure_bucket_major_sharded();
        if (bm_failed || !built || !members_used) return false;
        const u32 nl = (u32)h_leaf_off.size();
        try {
            bm_rows.ensure(members_used * (u64)dimp, 0, stream, true);
            bm_tomb.ensure(members_used / 32 + 8);
            slot_pos.ensure(slot_stride * (u64)T);
            d_leaf_tree.ensure(nl);
            if (opt.metric == ZB_METRIC_COSINE) bm_rinv.ensure(members_used);
            if (opt.metric == ZB_METRIC_L2SQ || opt.metric == ZB_METRIC_L2) {
                bm_n2.ensure(members_used);
                bm_leaf_n2max.ensure(nl ? nl : 1);
            }
        } catch (const Error& e) {
            if (e.code != ZB_ERR_OOM) throw;
            bm_rows.release();
            bm_failed = true;
            return false;
        }
        std::vector<u32> lt(h_leaf_tree.begin(), h_leaf_tree.end());
        ZB_CUDA(cudaMemcpyAsync(d_leaf_tree.p, lt.data(), (size_t)nl * 4, cudaMemcpyHostToDevice, stream));
        ZB_CUDA(cudaMemsetAsync(bm_tomb.p, 0, (members_used / 32 + 8) * 4, stream));
        u64 used = 0;
        for (u32 l = 0; l < nl; ++l) used += h_leaf_len[l];
        if (used != members_used) ZB_CUDA(cudaMemsetAsync(bm_rows.p, 0, members_used * (u64)dimp * 4, stream));  // slack positions
        launch_bm_gather(nl, d_leaf_off.p, d_leaf_len.p, d_leaf_tree.p, d_members.p, rows.p, tomb.p, dimp, slot_stride, bm_rows.p,
                         slot_pos.p, bm_tomb.p, stream);
        if (opt.metric == ZB_METRIC_COSINE) launch_rinv(bm_rows.p, members_used, dimp, bm_rinv.p, stream);
        if (opt.metric == ZB_METRIC_L2SQ || opt.metric == ZB_METRIC_L2) {
            launch_n2(bm_rows.p, members_used, dimp, bm_n2.p, stream);
            launch_leaf_n2max(nl, d_leaf_off.p, d_leaf_len.p, bm_n2.p, bm_leaf_n2max.p, stream);
        }
        make_row_tile_map(bm_tmap, bm_rows.p, members_used, dimp, 128, tile_scan_box_floats(2));
        make_row_tile_map(bm_tmap3, bm_rows.p, members_used, dimp, 64, tile_scan_box_floats(3));
        sync();
        bm_positions = members_used;
        bm_valid = true;
        return true;
    }
    // Bucket-sharded store (north_star (c), SURVEY 8e): every leaf is moved, whole, to rank leaf % G -- each rank packs
    // the rows it holds of every leaf by destination, the ranks exchange them with grouped ncclSend / ncclRecv, and the
    // owner sorts what it received by (leaf, ordinal) into contiguous [len][dimp] blocks.  One tree at a time, so the
    // staging area is 1/T of the store.  Collective: every rank must call it at the same point.
    bool ensure_bucket_major_sharded() {
        ZB_REQUIRE(comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
        ZB_REQUIRE(total_rows < (1ull << 40), ZB_ERR_STATE, "bucket-sharded store supports up to 2^40 rows");
        const u32 nl = (u32)h_leaf_off.size();
        sync_host_members();
        // every rank's share of every leaf
        DBuf<u32> d_all;
        d_all.ensure((size_t)nl * G);
        nccl.allgather(d_leaf_len.p, d_all.p, (size_t)nl * 4, stream);
        std::vector<u32> all_len((size_t)nl * G);
        ZB_CUDA(cudaMemcpyAsync(all_len.data(), d_all.p, all_len.size() * 4, cudaMemcpyDeviceToHost, stream));
        sync();
        std::vector<std::vector<u32>> owned(T);
        for (u32 l = 0; l < nl; ++l)
            if (h_leaf_node[l] >= 0 && l % G == rank) owned[h_leaf_tree[l]].push_back(l);
        std::vector<long long> off(nl, 0);
        std::vector<u32> len(nl, 0);
        h_tree_base.assign(T + 1, 0);
        u64 P = 0;
        for (int t = 0; t < T; ++t) {
            h_tree_base[t] = P;
            for (u32 l : owned[t]) {
                u64 g = 0;
                for (u32 r = 0; r < G; ++r) g += all_len[(size_t)r * nl + l];
                off[l] = (long long)P;
                len[l] = (u32)g;
                P += g;
            }
        }
        h_tree_base[T] = P;
        ZB_REQUIRE(P < (1ull << 31), ZB_ERR_STATE, "more than 2^31 bucket-major positions on one rank");
        const u64 Pa = P ? P : 1;
        bm_rows.ensure(Pa * (u64)dimp, 0, stream, true);
        bm_ord.ensure(Pa);
        bm_tomb.ensure(Pa / 32 + 8);
        d_iota.ensure(Pa);
        srt_ord.ensure(Pa);
        srt_pos.ensure(Pa);
        d_bm_off.ensure(nl ? nl : 1);
        d_bm_len.ensure(nl ? nl : 1);
        d_tree_base.ensure(T + 1);
        if (opt.metric == ZB_METRIC_COSINE) bm_rinv.ensure(Pa);
        if (opt.metric == ZB_METRIC_L2SQ || opt.metric == ZB_METRIC_L2) {
            bm_n2.ensure(Pa);
            bm_leaf_n2max.ensure(nl ? nl : 1);
        }
        ZB_CUDA(cudaMemsetAsync(bm_tomb.p, 0, (Pa / 32 + 8) * 4, stream));
        if (nl) {
            ZB_CUDA(cudaMemcpyAsync(d_bm_off.p, off.data(), (size_t)nl * 8, cudaMemcpyHostToDevice, stream));
            ZB_CUDA(cudaMemcpyAsync(d_bm_len.p, len.data(), (size_t)nl * 4, cudaMemcpyHostToDevice, stream));
        }
        ZB_CUDA(cudaMemcpyAsync(d_tree_base.p, h_tree_base.data(), (size_t)(T + 1) * 8, cudaMemcpyHostToDevice, stream));
        launch_iota_u32(d_iota.p, P, 0u, stream);
        sync();
        DBuf<u32> d_slots, sort_val[2];
        DBuf<float> snd_rows, st_rows;
        DBuf<u64> snd_key, st_key, sort_key[2];
        DBuf<RecvSeg> d_segs;
        DBuf<u8> sort_tmp;
        std::vector<std::vector<u32>> by_tree(T);  // live leaves of each tree, ascending
        for (u32 l = 0; l < nl; ++l)
            if (h_leaf_node[l] >= 0) by_tree[h_leaf_tree[l]].push_back(l);
        // The leaves of a tree travel in GROUPS (ascending leaf ranges, the same cut on every rank: it is computed from the
        // allgathered leaf shares), so that neither the send nor the receive staging area of any rank exceeds
        // `stage_rows` rows: the store of a 100M x 768 index is built with ~4 GB of staging instead of 2/T of the store.
        const u64 stage_rows = std::max<u64>(4096, (u64)p_bm_stage_mb * (1ull << 20) / ((u64)dimp * 4));
        for (int t = 0; t < T; ++t) {
            const std::vector<u32>& tl = by_tree[t];
            size_t own_i = 0;  // next leaf of owned[t] not yet placed
            u64 tree_pos = h_tree_base[t];
            for (size_t g0 = 0; g0 < tl.size();) {
                // cut the group
                std::vector<u64> snd_r(G, 0), st_r(G, 0);
                size_t g1 = g0;
                for (; g1 < tl.size(); ++g1) {
                    const u32 l = tl[g1];
                    u64 gl = 0, worst = 0;
                    for (u32 r = 0; r < G; ++r) gl += all_len[(size_t)r * nl + l];
                    for (u32 r = 0; r < G; ++r)
                        worst = std::max(worst, std::max(snd_r[r] + all_len[(size_t)r * nl + l], st_r[r] + (l % G == r ? gl : 0)));
                    if (g1 > g0 && worst > stage_rows) break;
                    for (u32 r = 0; r < G; ++r) snd_r[r] += all_len[(size_t)r * nl + l];
                    st_r[l % G] += gl;
                }
                // send side: my rows of the group's leaves, grouped by destination, leaf ascending, member order
                std::vector<u32> slots;
                std::vector<u64> send_off(G + 1, 0);
                for (u32 d = 0; d < G; ++d) {
                    send_off[d] = slots.size();
                    for (size_t i = g0; i < g1; ++i) {
                        const u32 l = tl[i];
                        if (l % G == d)
                            slots.insert(slots.end(), h_members.begin() + h_leaf_off[l], h_members.begin() + h_leaf_off[l] + h_leaf_len[l]);
                    }
                }
                send_off[G] = slots.size();
                // receive side: for every source, the group's owned leaves in ascending order
                size_t own_j = own_i;
                while (own_j < owned[t].size() && owned[t][own_j] <= tl[g1 - 1]) ++own_j;
                std::vector<RecvSeg> segs;
                std::vector<u64> recv_off(G + 1, 0);
                u64 R = 0;
                for (u32 r = 0; r < G; ++r) {
                    recv_off[r] = R;
                    for (size_t i = own_i; i < own_j; ++i) {
                        const u32 c = all_len[(size_t)r * nl + owned[t][i]];
                        if (c) segs.push_back(RecvSeg{R, c, (u32)(i - own_i)});
                        R += c;
                    }
                }
                recv_off[G] = R;
                ZB_REQUIRE(R == st_r[rank], ZB_ERR_STATE, "bucket-sharded layout mismatch");
                ZB_REQUIRE(own_j - own_i < (1u << 24), ZB_ERR_STATE, "too many leaves in one exchange group");
                const u64 ns = slots.size();
                d_slots.ensure(ns ? ns : 1);
                snd_rows.ensure((ns ? ns : 1) * (u64)dimp);
                snd_key.ensure(ns ? ns : 1);
                st_rows.ensure((R ? R : 1) * (u64)dimp);
                st_key.ensure(R ? R : 1);
                for (int b = 0; b < 2; ++b) {
                    sort_key[b].ensure(R ? R : 1);
                    sort_val[b].ensure(R ? R : 1);
                }
                d_segs.ensure(segs.size() ? segs.size() : 1);
                sort_tmp.ensure(sort_temp_bytes(R ? R : 1));
                if (ns) ZB_CUDA(cudaMemcpyAsync(d_slots.p, slots.data(), ns * 4, cudaMemcpyHostToDevice, stream));
                if (!segs.empty()) ZB_CUDA(cudaMemcpyAsync(d_segs.p, segs.data(), segs.size() * sizeof(RecvSeg), cudaMemcpyHostToDevice, stream));
                launch_pack_rows(d_slots.p, ns, rows.p, ord.p, tomb.p, dimp, snd_rows.p, snd_key.p, stream);
                const size_t rb = (size_t)dimp * 4;
                nccl.group_start();
                for (u32 r = 0; r < G; ++r) {
                    if (r == rank) continue;
                    const u64 sc = send_off[r + 1] - send_off[r], rc = recv_off[r + 1] - recv_off[r];
                    nccl.send(snd_rows.p + send_off[r] * (u64)dimp, sc * rb, (int)r, stream);
                    nccl.send(snd_key.p + send_off[r], sc * 8, (int)r, stream);
                    nccl.recv(st_rows.p + recv_off[r] * (u64)dimp, rc * rb, (int)r, stream);
                    nccl.recv(st_key.p + recv_off[r], rc * 8, (int)r, stream);
                }
                nccl.group_end();
                {   // my own share never leaves the device
                    const u64 sc = send_off[rank + 1] - send_off[rank];
                    ZB_REQUIRE(sc == recv_off[rank + 1] - recv_off[rank], ZB_ERR_STATE, "bucket-sharded self share mismatch");
                    if (sc) {
                        ZB_CUDA(cudaMemcpyAsync(st_rows.p + recv_off[rank] * (u64)dimp, snd_rows.p + send_off[rank] * (u64)dimp, sc * rb,
                                                cudaMemcpyDeviceToDevice, stream));
                        ZB_CUDA(cudaMemcpyAsync(st_key.p + recv_off[rank], snd_key.p + send_off[rank], sc * 8, cudaMemcpyDeviceToDevice, stream));
                    }
                }
                launch_seg_keys(d_segs.p, (u32)segs.size(), st_key.p, sort_key[0].p, sort_val[0].p, stream);
                sort_pairs_u64_u32(sort_tmp.p, sort_tmp.bytes(), sort_key[0].p, sort_key[1].p, sort_val[0].p, sort_val[1].p, R, 64, stream);
                launch_place_rows(sort_val[1].p, R, st_rows.p, st_key.p, dimp, tree_pos, bm_rows.p, bm_ord.p, bm_tomb.p, stream);
                sync();  // the host vectors of this group (slots, segs) and the staging areas are reused by the next one
                tree_pos += R;
                own_i = own_j;
                g0 = g1;
            }
            ZB_REQUIRE(tree_pos == h_tree_base[t + 1] && own_i == owned[t].size(), ZB_ERR_STATE, "bucket-sharded layout mismatch");
            // ordinal -> position index of the tree's region
            const u64 Rt = h_tree_base[t + 1] - h_tree_base[t];
            sort_tmp.ensure(sort_temp_bytes(Rt ? Rt : 1));
            sort_pairs_u64_u32(sort_tmp.p, sort_tmp.bytes(), bm_ord.p + h_tree_base[t], srt_ord.p + h_tree_base[t],
                               d_iota.p + h_tree_base[t], srt_pos.p + h_tree_base[t], Rt, 40, stream);
            sync();
        }
        if (opt.metric == ZB_METRIC_COSINE) launch_rinv(bm_rows.p, P, dimp, bm_rinv.p, stream);
        if (opt.metric == ZB_METRIC_L2SQ || opt.metric == ZB_METRIC_L2) {   // leaves this rank does not own have length 0 here
            launch_n2(bm_rows.p, P, dimp, bm_n2.p, stream);
            launch_leaf_n2max(nl, d_bm_off.p, d_bm_len.p, bm_n2.p, bm_leaf_n2max.p, stream);
        }
        make_row_tile_map(bm_tmap, bm_rows.p, Pa, dimp, 128, tile_scan_box_floats(2));
        make_row_tile_map(bm_tmap3, bm_rows.p, Pa, dimp, 64, tile_scan_box_floats(3));
        sync();
        bm_positions = P;
        bm_valid = true;
        return true;
    }
    // Collective (every rank calls it with the same `need`): (re)allocates the batch buffer, exchanges the IPC handles through
    // the communicator and maps the peers.  Any rank failing makes every rank fall back to the NCCL allgather for good.
    bool ensure_peer_queries(u64 need) {
        if (pq.failed || !p_p2p_queries) return false;
        if (need <= pq.cap && !pq.peer.empty()) return true;
        release_peer_queries();
        const u64 ncap = need + need / 2;
        u32 ok = 1;
        if (cudaMalloc((void**)&pq.mine, ncap * 4) != cudaSuccess) { cudaGetLastError(); pq.mine = nullptr; ok = 0; }
        cudaIpcMemHandle_t h;
        memset(&h, 0, sizeof h);
        if (ok && cudaIpcGetMemHandle(&h, pq.mine) != cudaSuccess) { cudaGetLastError(); ok = 0; }
        // [handle (64 bytes) | ok flag] of every rank
        const size_t rec = 80;
        DBuf<u8> d_rec, d_all;
        d_rec.ensure(rec);
        d_all.ensure(rec * G);
        u8 hrec[80];
        memset(hrec, 0, sizeof hrec);
        memcpy(hrec, &h, sizeof h);
        memcpy(hrec + 64, &ok, 4);
        ZB_CUDA(cudaMemcpyAsync(d_rec.p, hrec, rec, cudaMemcpyHostToDevice, stream));
        nccl.allgather(d_rec.p, d_all.p, rec, stream);
        std::vector<u8> all(rec * G);
        ZB_CUDA(cudaMemcpyAsync(all.data(), d_all.p, rec * G, cudaMemcpyDeviceToHost, stream));
        sync();
        bool all_ok = true;
        for (u32 r = 0; r < G; ++r) {
            u32 f = 0;
            memcpy(&f, all.data() + r * rec + 64, 4);
            all_ok = all_ok && f;
        }
        pq.peer.assign(G, nullptr);
        u32 mapped = all_ok ? 1u : 0u;
        if (all_ok) {
            for (u32 r = 0; r < G && mapped; ++r) {
                if (r == rank) { pq.peer[r] = pq.mine; continue; }
                cudaIpcMemHandle_t ph;
                memcpy(&ph, all.data() + r * rec, sizeof ph);
                void* ptr = nullptr;
                if (cudaIpcOpenMemHandle(&ptr, ph, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); mapped = 0; }
                pq.peer[r] = (float*)ptr;
            }
        }
        // second round: did every rank map every peer?
        DBuf<u32> d_flag;
        d_flag.ensure(1);
        ZB_CUDA(cudaMemcpyAsync(d_flag.p, &mapped, 4, cudaMemcpyHostToDevice, stream));
        nccl.allreduce(d_flag.p, 1, Nccl::U32, Nccl::MIN, stream);
        ZB_CUDA(cudaMemcpyAsync(&mapped, d_flag.p, 4, cudaMemcpyDeviceToHost, stream));
        sync();
        if (!mapped) {
            release_peer_queries();
            pq.failed = true;
            return false;
        }
        if (!pq.fork) {
            ZB_CUDA(cudaEventCreateWithFlags(&pq.fork, cudaEventDisableTiming));
            for (int i = 0; i < PeerQ::NS; ++i) {
                ZB_CUDA(cudaStreamCreateWithFlags(&pq.stream[i], cudaStreamNonBlocking));
                ZB_CUDA(cudaEventCreateWithFlags(&pq.done[i], cudaEventDisableTiming));
            }
        }
        pq.cap = ncap;
        g_device_bytes += ncap * 4;
        return true;
    }
    void release_peer_queries() {
        cudaDeviceSynchronize();
        for (u32 r = 0; r < pq.peer.size(); ++r)
            if (r != rank && pq.peer[r]) cudaIpcCloseMemHandle(pq.peer[r]);
        pq.peer.clear();
        if (pq.mine) {
            cudaFree(pq.mine);
            if (pq.cap) g_device_bytes -= pq.cap * 4;
        }
        pq.mine = nullptr;
        pq.cap = 0;
    }
    BucketMajor bm_view() const {
        BucketMajor b;
        b.rows = bm_rows.p;
        b.rinv = bm_rinv.p;
        b.tomb = bm_tomb.p;
        if (opt.metric == ZB_METRIC_L2SQ || opt.metric == ZB_METRIC_L2) {
            b.n2 = bm_n2.p;
            b.leaf_n2max = bm_leaf_n2max.p;
        }
        b.tmap = bm_tmap;
        b.tmap3 = bm_tmap3;
        b.positions = bm_positions;
        return b;
    }
    void recount_live() {  // leaf_live from members + tombstones, then the global plan counts
        u32 nl = (u32)h_leaf_off.size();
        d_leaf_live.ensure(nl ? nl : 1);
        d_leaf_plan.ensure(nl ? nl : 1);
        if (nl) count_live_kernel<<<(nl + 127) / 128, 128, 0, stream>>>(d_members.p, d_leaf_off.p, d_leaf_len.p, tomb.p, nl, d_leaf_live.p);
        refresh_plan_counts();
    }
    void refresh_plan_counts() {
        u32 nl = (u32)h_leaf_off.size();
        if (G > 1 && nl) {
            ZB_REQUIRE(comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
            d_leaf_plan.ensure(nl);
            ZB_CUDA(cudaMemcpyAsync(d_leaf_plan.p, d_leaf_live.p, (size_t)nl * 4, cudaMemcpyDeviceToDevice, stream));
            nccl.allreduce(d_leaf_plan.p, nl, Nccl::U32, Nccl::SUM, stream);
        }
    }
    void sync_host_members() {
        if (h_members_valid) return;
        h_members.resize(members_used);
        if (members_used)
            ZB_CUDA(cudaMemcpyAsync(h_members.data(), d_members.p, members_used * 4, cudaMemcpyDeviceToHost, stream));
        sync();
        h_members_valid = true;
    }
    int new_leaf(int node, int tree, u64 key, int depth, long long off, u32 len, u32 cap) {
        int id = (int)h_leaf_off.size();
        h_leaf_off.push_back(off);
        h_leaf_len.push_back(len);
        h_leaf_cap.push_back(cap);
        h_leaf_key.push_back(key);
        h_leaf_depth.push_back(depth);
        h_leaf_node.push_back(node);
        h_leaf_tree.push_back(tree);
        return id;
    }

    void clear_forest() {
        h_nodes.clear();
        h_roots.assign(T, -1);
        n_planes = 0;
        h_leaf_off.clear(); h_leaf_len.clear(); h_leaf_cap.clear(); h_leaf_key.clear();
        h_leaf_depth.clear(); h_leaf_node.clear(); h_leaf_tree.clear();
        members_used = 0;
        h_members.clear();
        h_members_valid = false;
        built = false;
        export_table_valid = false;
        bm_valid = false;
        bm_failed = false;
    }

    // ---------------------------------------------------------------- build (lsh.rs:192-267, level synchronous)
    // `active`: nodes to build over the slots in b_work[0][0..total).  New leaves' members are appended to
    // d_members; nodes/planes/leaves are appended to the host mirror (uploaded by the caller).
    void build_subtrees(std::vector<BSeg> active, u64 total) {
        const u64 max_node = opt.max_node_size;
        auto t_start = std::chrono::steady_clock::now();
        int level = 0;
        std::vector<BSeg> leaves;
        int cur = 0;
        b_work[1].ensure(total ? total : 1);
        b_flags.ensure(total + 1);
        b_scan.ensure(total + 1);
        scan_tmp(total + 1);
        std::vector<SegDesc> hsegs;
        std::vector<Tile> htiles;
        std::vector<u32> habove, hgabove;
        while (true) {
            std::vector<BSeg> split, next;
            for (const BSeg& s : active) {
                if (s.glen < max_node || s.glen < 2 || s.depth >= ZB_MAX_DEPTH || s.attempt >= ZB_MAX_ATTEMPTS) leaves.push_back(s);
                else split.push_back(s);
            }
            if (split.empty()) break;
            const u32 ns = (u32)split.size();
            d_coef.ensure((n_planes + ns) * (u64)dimp, n_planes * (u64)dimp, stream);
            d_cst.ensure(n_planes + ns, n_planes, stream);
            hsegs.resize(ns);
            htiles.clear();
            for (u32 i = 0; i < ns; ++i) {
                const BSeg& s = split[i];
                hsegs[i] = SegDesc{s.off, s.len, (u32)(n_planes + i), s.key, s.attempt, 0};
                for (u32 b = 0; b < s.len; b += 64) htiles.push_back(Tile{i, std::min<u32>(64, s.len - b), s.off + b});
            }
            const u32 nt = (u32)htiles.size();
            b_segs.ensure(ns);
            b_tiles.ensure(nt ? nt : 1);
            b_minh.ensure(ns); b_minord.ensure(ns); b_excl.ensure(ns);
            b_slot_a.ensure(ns); b_slot_b.ensure(ns); b_above.ensure(2 * (size_t)ns);
            b_pair_rows.ensure((size_t)ns * 2 * dimp);
            ZB_CUDA(cudaMemcpyAsync(b_segs.p, hsegs.data(), ns * sizeof(SegDesc), cudaMemcpyHostToDevice, stream));
            if (nt) ZB_CUDA(cudaMemcpyAsync(b_tiles.p, htiles.data(), nt * sizeof(Tile), cudaMemcpyHostToDevice, stream));
            const u32* work = b_work[cur].p;
            for (int which = 0; which < 2; ++which) {  // a, then b (excluding a)
                int* slot_out = which ? b_slot_b.p : b_slot_a.p;
                const u64* excl = which ? b_excl.p : nullptr;
                ZB_CUDA(cudaMemsetAsync(b_minh.p, 0xFF, ns * 8, stream));
                ZB_CUDA(cudaMemsetAsync(b_minord.p, 0xFF, ns * 8, stream));
                ZB_CUDA(cudaMemsetAsync(slot_out, 0xFF, ns * 4, stream));
                launch_pick(0, b_tiles.p, nt, b_segs.p, work, ord.p, excl, b_minh.p, b_minord.p, slot_out, stream);
                if (G > 1) nccl.allreduce(b_minh.p, ns, Nccl::U64, Nccl::MIN, stream);
                launch_pick(1, b_tiles.p, nt, b_segs.p, work, ord.p, excl, b_minh.p, b_minord.p, slot_out, stream);
                if (G > 1) nccl.allreduce(b_minord.p, ns, Nccl::U64, Nccl::MIN, stream);
                launch_pick(2, b_tiles.p, nt, b_segs.p, work, ord.p, excl, b_minh.p, b_minord.p, slot_out, stream);
                if (!which) ZB_CUDA(cudaMemcpyAsync(b_excl.p, b_minord.p, ns * 8, cudaMemcpyDeviceToDevice, stream));
            }
            launch_fetch_pair_rows(b_segs.p, ns, b_slot_a.p, b_slot_b.p, rows.p, dimp, b_pair_rows.p, stream);
            if (G > 1) nccl.allreduce(b_pair_rows.p, (size_t)ns * 2 * dimp, Nccl::I32, Nccl::SUM, stream);
            launch_make_planes(b_segs.p, ns, b_pair_rows.p, dimp, d_coef.p, d_cst.p, stream);
            ZB_CUDA(cudaMemsetAsync(b_flags.p, 0, (total + 1) * 4, stream));
            launch_classify(b_tiles.p, nt, b_segs.p, work, rows.p, d_coef.p, d_cst.p, dimp, b_flags.p, (int)p_classify_variant, stream);
            exclusive_scan_u32(cub_tmp.p, cub_tmp.bytes(), b_flags.p, b_scan.p, total + 1, stream);
            launch_seg_above(b_segs.p, ns, b_scan.p, b_above.p, stream);
            habove.resize(ns);
            hgabove.resize(ns);
            ZB_CUDA(cudaMemcpyAsync(habove.data(), b_above.p, ns * 4, cudaMemcpyDeviceToHost, stream));
            if (G > 1) {
                ZB_CUDA(cudaMemcpyAsync(b_above.p + ns, b_above.p, ns * 4, cudaMemcpyDeviceToDevice, stream));
                nccl.allreduce(b_above.p + ns, ns, Nccl::U32, Nccl::SUM, stream);
                ZB_CUDA(cudaMemcpyAsync(hgabove.data(), b_above.p + ns, ns * 4, cudaMemcpyDeviceToHost, stream));
            }
            if (total) ZB_CUDA(cudaMemcpyAsync(b_work[cur ^ 1].p, work, total * 4, cudaMemcpyDeviceToDevice, stream));
            launch_scatter(b_tiles.p, nt, b_segs.p, work, b_flags.p, b_scan.p, b_work[cur ^ 1].p, stream);
            sync();
            cur ^= 1;
            if (G <= 1) hgabove = habove;
            for (u32 i = 0; i < ns; ++i) {
                BSeg s = split[i];
                const u64 ga = hgabove[i], gb = s.glen - ga;
                if (ga == 0 || gb == 0) {  // degenerate split: retry with the next sample (D2)
                    s.attempt++;
                    next.push_back(s);
                    continue;
                }
                const u32 la = habove[i], lb = s.len - la;
                const int nl = (int)h_nodes.size(), nr = nl + 1;
                h_nodes.push_back(make_int4(-1, -1, -1, -1));
                h_nodes.push_back(make_int4(-1, -1, -1, -1));
                h_nodes[s.node] = make_int4((int)(n_planes + i), nl, nr, -1);
                next.push_back(BSeg{child_key(s.key, 0), s.depth + 1, nl, s.tree, s.off, lb, gb, 0});
                next.push_back(BSeg{child_key(s.key, 1), s.depth + 1, nr, s.tree, s.off + lb, la, ga, 0});
            }
            n_planes += ns;
            active.swap(next);
            if (trace_on && rank == 0) {
                auto now = std::chrono::steady_clock::now();
                fprintf(stderr, "[zb trace] build level %d: %u nodes, %u tiles, %.3f ms\n", level, ns, nt,
                        std::chrono::duration<double, std::milli>(now - t_start).count());
                t_start = now;
            }
            ++level;
        }
        // finalize leaves: members of leaf = b_work[cur][off, off+len)
        d_members.ensure(members_used + total, members_used, stream);
        if (total) ZB_CUDA(cudaMemcpyAsync(d_members.p + members_used, b_work[cur].p, total * 4, cudaMemcpyDeviceToDevice, stream));
        std::vector<std::vector<Tile>> tiles_by_tree(T);
        for (const BSeg& s : leaves) {
            int leaf = new_leaf(s.node, s.tree, s.key, s.depth, (long long)members_used + s.off, s.len, s.len);
            h_nodes[s.node] = make_int4(-1, -1, -1, leaf);
            for (u32 b = 0; b < s.len; b += 64)
                tiles_by_tree[s.tree].push_back(Tile{(u32)leaf, std::min<u32>(64, s.len - b), (long long)members_used + s.off + b});
        }
        for (int t = 0; t < T; ++t) {
            u32 nt = (u32)tiles_by_tree[t].size();
            if (!nt) continue;
            b_tiles.ensure(nt);
            ZB_CUDA(cudaMemcpyAsync(b_tiles.p, tiles_by_tree[t].data(), nt * sizeof(Tile), cudaMemcpyHostToDevice, stream));
            launch_assign_leaf(b_tiles.p, nt, d_members.p, slot_leaf.p + (u64)t * slot_stride, stream);
            sync();
        }
        members_used += total;
        h_members_valid = false;
        if (trace_on && rank == 0)
            fprintf(stderr, "[zb trace] build finalize: %.3f ms\n",
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    }

    u64 allreduce_sum_u64(u64 v) {
        if (G <= 1) return v;
        b_minh.ensure(1);
        ZB_CUDA(cudaMemcpyAsync(b_minh.p, &v, 8, cudaMemcpyHostToDevice, stream));
        nccl.allreduce(b_minh.p, 1, Nccl::U64, Nccl::SUM, stream);
        ZB_CUDA(cudaMemcpyAsync(&v, b_minh.p, 8, cudaMemcpyDeviceToHost, stream));
        sync();
        return v;
    }

    // build_index, lsh.rs:411-429: every tree over every live row.
    void bulk_build() {
        clear_forest();
        std::vector<u32> live;
        live.reserve(n_slots);
        for (u64 s = 0; s < n_slots; ++s)
            if (!h_tomb[s]) live.push_back((u32)s);
        const u64 nl = live.size();
        const u64 gl = allreduce_sum_u64(nl);
        const u64 total = nl * (u64)T;
        b_work[0].ensure(total ? total : 1);
        std::vector<BSeg> segs;
        for (int t = 0; t < T; ++t) {
            if (nl) ZB_CUDA(cudaMemcpyAsync(b_work[0].p + (u64)t * nl, live.data(), nl * 4, cudaMemcpyHostToDevice, stream));
            h_nodes.push_back(make_int4(-1, -1, -1, -1));
            h_roots[t] = t;
            segs.push_back(BSeg{root_key(opt.seed, t), 0, t, t, (long long)((u64)t * nl), (u32)nl, gl, 0});
        }
        sync();
        build_subtrees(segs, total);
        upload_structure();
        recount_live();
        built = true;
    }

    // add on an existing forest (lsh.rs:445-462 per D4): descend, append to leaves, rebuild overfull leaves.
    void incremental_insert(u64 first_slot, u64 n_new) {
        if (!n_new && G <= 1) return;
        ForestView f = view();
        std::vector<int> leaf_of((size_t)n_new * T);
        if (n_new) {
            h_leaves.ensure(n_new * (u64)T);
            launch_hash(f, rows.p + first_slot * (u64)dimp, n_new, nullptr, nullptr, h_leaves.p, (int)p_hash_variant, stream);
            ZB_CUDA(cudaMemcpyAsync(leaf_of.data(), h_leaves.p, leaf_of.size() * 4, cudaMemcpyDeviceToHost, stream));
        }
        sync_host_members();
        for (u64 i = 0; i < n_new; ++i) {
            for (int t = 0; t < T; ++t) {
                const int l = leaf_of[i * T + t];
                if (h_leaf_len[l] == h_leaf_cap[l]) {  // relocate the leaf to the end of the member array with slack
                    u32 ncap = std::max<u32>(8, h_leaf_cap[l] * 2);
                    size_t noff = h_members.size();
                    h_members.resize(noff + ncap, 0);
                    std::copy(h_members.begin() + h_leaf_off[l], h_members.begin() + h_leaf_off[l] + h_leaf_len[l],
                              h_members.begin() + noff);
                    h_leaf_off[l] = (long long)noff;
                    h_leaf_cap[l] = ncap;
                }
                h_members[h_leaf_off[l] + h_leaf_len[l]++] = (u32)(first_slot + i);
            }
        }
        members_used = h_members.size();
        d_members.ensure(members_used ? members_used : 1);
        if (members_used) ZB_CUDA(cudaMemcpyAsync(d_members.p, h_members.data(), members_used * 4, cudaMemcpyHostToDevice, stream));
        if (n_new) {  // slot_leaf of the new rows
            std::vector<u32> col(n_new);
            for (int t = 0; t < T; ++t) {
                for (u64 i = 0; i < n_new; ++i) col[i] = (u32)leaf_of[i * T + t];
                ZB_CUDA(cudaMemcpyAsync(slot_leaf.p + (u64)t * slot_stride + first_slot, col.data(), n_new * 4, cudaMemcpyHostToDevice, stream));
                sync();
            }
        }
        upload_structure();
        recount_live();
        // overfull leaves (global live count > max_node_size) are rebuilt: lsh.rs:367-378
        const u32 nl = (u32)h_leaf_off.size();
        std::vector<u32> plan(nl);
        ZB_CUDA(cudaMemcpyAsync(plan.data(), view().leaf_plan, (size_t)nl * 4, cudaMemcpyDeviceToHost, stream));
        sync();
        std::vector<BSeg> segs;
        std::vector<u32> work;
        for (u32 l = 0; l < nl; ++l) {
            if (h_leaf_node[l] < 0 || plan[l] <= opt.max_node_size) continue;
            long long off = (long long)work.size();
            for (u32 i = 0; i < h_leaf_len[l]; ++i) {
                u32 s = h_members[h_leaf_off[l] + i];
                if (!h_tomb[s]) work.push_back(s);
            }
            segs.push_back(BSeg{h_leaf_key[l], h_leaf_depth[l], h_leaf_node[l], h_leaf_tree[l], off,
                                (u32)(work.size() - off), plan[l], 0});
            h_leaf_node[l] = -1;  // retired: no node references it any more
            h_leaf_len[l] = 0;
        }
        if (!segs.empty()) {
            b_work[0].ensure(work.size() ? work.size() : 1);
            if (!work.empty()) ZB_CUDA(cudaMemcpyAsync(b_work[0].p, work.data(), work.size() * 4, cudaMemcpyHostToDevice, stream));
            sync();
            build_subtrees(segs, work.size());
            upload_structure();
            recount_live();
        }
    }
};

// =====================================================================================================
// search
// =====================================================================================================
namespace zb {

// nq = queries of the whole batch.  Unsharded, or sharded with sliced == false: d_q holds all of them and the outputs hold
// all nq results (on every rank).  Sharded with sliced == true (the scalable form): d_q holds only the slice this rank
// fronts, queries [rank * nqp, (rank + 1) * nqp) with nqp = ceil(nq / G); the slices are allgathered over NVLink into
// q_all, and the outputs receive the results of the rank's own slice only (no result allgather).
// probes > 0: multi-probe walk (DESIGN 3.9); the visits it appends go through the same compaction, scan and merge.
static void search_device(zb_index* ix, u64 nq, const float* d_q, u64 top_k, u32 probes, u64* d_out_ord, u64* d_out_bits,
                          u32* d_out_counts, bool sliced) {
    cudaStream_t s = ix->stream;
    const u32 T = ix->T;
    ix->st.last_queries = nq;
    ix->st.last_visits = ix->st.last_pairs = ix->st.last_tile_visits = ix->st.last_tile_pairs = 0;
    ix->st.last_moved_bytes = 0;
    ix->st.last_scan_launches = ix->st.last_total_launches = 0;
    if (!nq) return;
    const bool sharded = ix->G > 1;
    const u32 G = ix->G;
    const u64 nqp = sharded ? (nq + G - 1) / G : nq;
    const u64 q0 = sharded ? std::min<u64>(nq, (u64)ix->rank * nqp) : 0;
    const u64 qn = sharded ? std::min<u64>(nqp, nq - q0) : nq;
    sliced = sliced && sharded;
    const u64 n_out = sliced ? qn : nq;
    if (!ix->built || top_k == 0) {
        launch_fill_u64(d_out_ord, n_out * top_k, ZB_SENTINEL, s);
        launch_fill_u64(d_out_bits, n_out * top_k, ZB_SENTINEL, s);
        if (n_out) ZB_CUDA(cudaMemsetAsync(d_out_counts, 0, n_out * 4, s));
        return;
    }
    if (sharded) ix->ensure_bucket_major();  // collective (rebuilds the bucket-sharded store after a forest change)
    ForestView f = ix->view();              // the plan walks the replicated forest with GLOBAL live leaf counts
    const ForestView fs = ix->scan_view();  // scoring reads the leaves this rank holds
    const u64 nw = nqp * (sharded ? G : 1) * T;  // walkers, padded to G equal slices
    const u64 nwl = nqp * T;                     // walkers this rank plans
    ZB_REQUIRE(nw < (1ull << 31), ZB_ERR_INVALID, "batch too large: %llu walkers", (unsigned long long)nw);
    ZB_CUDA(cudaEventRecord(ix->ev[0], s));
    ix->trace_mark("start");
    const float* d_q_mine = d_q + (sliced ? 0 : q0 * (u64)ix->dimp);  // the queries this rank plans
    // knob single_exchange (default 1): the query slices travel in the SAME allgather as the visit records, after the plan walk
    // (which needs only the rank's own slice) -- one collective before the scan instead of two
    const bool p2p = sliced && ix->ensure_peer_queries(nqp * G * (u64)ix->dimp);
    const bool one_exchange = sliced && !p2p && ix->p_single_exchange;
    if (p2p) {
        // my slice goes to every rank's batch buffer on a side stream (copy engines over NVLink), overlapped with the plan
        // walk; the main stream joins before the visit-record allgather, which is then also the barrier for the pushes
        const u64 slice = nqp * (u64)ix->dimp;
        ZB_CUDA(cudaEventRecord(ix->pq.fork, s));
        for (int i = 0; i < zb_index::PeerQ::NS; ++i) ZB_CUDA(cudaStreamWaitEvent(ix->pq.stream[i], ix->pq.fork, 0));
        for (u32 i = 0; i < G; ++i) {
            const u32 r = (ix->rank + i) % G;   // start with myself, then round the ring: the ranks do not all hit the same target first
            cudaStream_t ps = ix->pq.stream[i % zb_index::PeerQ::NS];
            float* dst = ix->pq.peer[r] + (u64)ix->rank * slice;
            if (qn) ZB_CUDA(cudaMemcpyAsync(dst, d_q, qn * (u64)ix->dimp * 4, cudaMemcpyDeviceToDevice, ps));
            if (qn < nqp) ZB_CUDA(cudaMemsetAsync(dst + qn * (u64)ix->dimp, 0, (nqp - qn) * (u64)ix->dimp * 4, ps));
        }
        for (int i = 0; i < zb_index::PeerQ::NS; ++i) ZB_CUDA(cudaEventRecord(ix->pq.done[i], ix->pq.stream[i]));
        d_q = ix->pq.mine;
    } else if (one_exchange) {
        ix->q_all.ensure(nqp * G * (u64)ix->dimp);
        d_q = ix->q_all.p;   // filled from the exchanged blocks below
    } else if (sliced) {  // every rank needs every query for the scan of the leaves it owns: allgather of the slices (in place)
        ix->q_all.ensure(nqp * G * (u64)ix->dimp);
        float* mine = ix->q_all.p + (u64)ix->rank * nqp * ix->dimp;
        if (qn) ZB_CUDA(cudaMemcpyAsync(mine, d_q, qn * (u64)ix->dimp * 4, cudaMemcpyDeviceToDevice, s));
        if (qn < nqp) ZB_CUDA(cudaMemsetAsync(mine + qn * (u64)ix->dimp, 0, (nqp - qn) * (u64)ix->dimp * 4, s));
        ix->nccl.allgather(mine, ix->q_all.p, nqp * (u64)ix->dimp * 4, s);
        d_q = ix->q_all.p;
        ix->trace_mark("allgather of queries");
    }
    ix->w_counts.ensure(nw + 1);
    ix->w_off.ensure(nw + 1);
    ix->w_flag.ensure(4);
    ix->scan_tmp(nw + 1);
    u32 nv = 0, total_slots = 0;
    u64 total_pairs = 0;
    // the fused tile kernel takes every visit of a leaf with >= tile_min_rows rows (here) and n' <= 32; known up front, so
    // the compaction can already set those visits aside and the host reads ONE record {flag, visits, slots, pairs} per batch
    // (the scalar metrics 3..11 are a sequential fold per pair: gather path only)
    const bool gen3 = ix->p_scan_gen != 2 && tile_scan3_supported(ix->dimp, (u32)top_k);
    const bool tile_on = ix->opt.metric <= ZB_METRIC_L2 && ix->p_use_tile_scan && ix->opt.max_node_size >= (u64)ix->p_tile_min_rows &&
                         (gen3 || tile_scan_supported(ix->dimp, (u32)top_k)) && ix->ensure_bucket_major();
    u64 v_cap = std::max<u64>(ix->v_leaf.cap ? ix->v_leaf.cap - 1 : 0, nw * (1 + (u64)probes) + nw / 2 + 1024);
    // a walker's region holds its cascade (31 visits by default) plus its probe visits, so the first probe batch needs no replan
    if (probes) ix->vpw = std::max<u32>(ix->vpw, 32 + probes);
    if (sharded && !ix->x_cap) ix->x_cap = (u32)std::min<u64>(nwl + nwl / 2 + 64, 0x7FFFFFFFull);
    ix->plan_totals.ensure(8);
    // Three nested retries, each decided from data every rank sees identically or from purely local state:
    //   replan   (a walker produced more visits than its region holds): flag travels in the exchanged headers;
    //   re-exchange (a rank packed more records than the exchange block holds): counts travel in the headers;
    //   re-compact  (more visits land here than the local arrays hold): local arrays only, no collective is repeated.
    bool need_plan = true, need_exchange = true;
    for (;;) {
        ix->v_leaf.ensure(v_cap + 1); ix->v_np.ensure(v_cap + 1); ix->v_q.ensure(v_cap + 1);
        ix->v_pair_len.ensure(v_cap + 1); ix->v_pair_off.ensure(v_cap + 1);
        ix->v_ent_len.ensure(v_cap + 1); ix->v_ent_off.ensure(v_cap + 1);
        ix->v_done.ensure(v_cap + 1);
        if (sharded) ix->v_w.ensure(v_cap + 1);
        ix->scan_tmp(std::max<u64>(std::max<u64>(nw, v_cap), sharded ? (u64)G * ix->x_cap : 0) + 1);
        if (need_plan) {
            ix->w_visits.ensure(nwl * ix->vpw);
            ZB_CUDA(cudaMemsetAsync(ix->w_flag.p, 0, 16, s));
            ZB_CUDA(cudaMemsetAsync(ix->w_counts.p + nwl, 0, 4, s));
            // padding walkers of my slice (queries beyond nq) carry an empty header
            if (sharded && qn < nqp) {
                ZB_CUDA(cudaMemsetAsync(ix->w_visits.p + qn * T * ix->vpw, 0, (nqp - qn) * T * ix->vpw * sizeof(uint2), s));
                ZB_CUDA(cudaMemsetAsync(ix->w_counts.p + qn * T, 0, (nqp - qn) * T * 4, s));
            }
            // walkers whose first leaf cannot fill the budget (the count cascade goes on: few, but each a long chain of dependent
            // nodes) go to the latency-optimised tail kernel -- unless the leaves are so small that every walker cascades
            u32* tail = nullptr;
            if (ix->p_plan_tail && ix->opt.max_node_size >= 4 * top_k) {
                ix->w_tail.ensure(nwl + 2);
                tail = ix->w_tail.p;
            }
            launch_plan(f, d_q_mine, (u32)qn, (u32)top_k, probes, ix->vpw, ix->w_visits.p, ix->w_counts.p, ix->w_flag.p, tail, s);
            if (tail) ix->st.last_total_launches += 1;
            ix->trace_mark("plan walk");
            if (sharded) {
                ix->w_loc_off.ensure(nwl + 1);
                exclusive_scan_u32(ix->cub_tmp.p, ix->cub_tmp.bytes(), ix->w_counts.p, ix->w_loc_off.p, nwl + 1, s);
            }
            need_plan = false;
            need_exchange = true;
            ix->st.last_total_launches += 1;
        }
        // a rank's block of the exchange: [header | C visit records | (one_exchange) its query slice, nqp rows], in uint4 units
        const size_t q4 = one_exchange ? (size_t)nqp * ix->dimp / 4 : 0;
        if (sharded && need_exchange) {
            const u32 C = ix->x_cap;
            const size_t B4 = (size_t)C + 1 + q4;
            ix->x_send.ensure(B4);
            ix->x_all.ensure(B4 * G);
            ix->x_flags.ensure((size_t)C * G + 1);
            ix->x_pos.ensure((size_t)C * G + 1);
            launch_pack_visits((u32)nwl, ix->vpw, ix->w_visits.p, ix->w_counts.p, ix->w_loc_off.p, (u32)((u64)ix->rank * nwl), C,
                               ix->w_flag.p, ix->x_send.p, s);
            if (one_exchange) {
                float* qdst = reinterpret_cast<float*>(ix->x_send.p + (size_t)C + 1);
                if (qn) ZB_CUDA(cudaMemcpyAsync(qdst, d_q_mine, qn * (u64)ix->dimp * 4, cudaMemcpyDeviceToDevice, s));
                if (qn < nqp) ZB_CUDA(cudaMemsetAsync(qdst + qn * (u64)ix->dimp, 0, (nqp - qn) * (u64)ix->dimp * 4, s));
            }
            if (p2p)  // my pushes are complete before I enter the collective
                for (int i = 0; i < zb_index::PeerQ::NS; ++i) ZB_CUDA(cudaStreamWaitEvent(s, ix->pq.done[i], 0));
            ix->nccl.allgather(ix->x_send.p, ix->x_all.p, B4 * sizeof(uint4), s);
            ix->trace_mark(p2p ? "push of queries + allgather of visits" : one_exchange ? "allgather of visits + queries" : "allgather of visits");
            if (one_exchange)  // the G slices, one per block, into the contiguous batch the scoring kernels index by query number
                ZB_CUDA(cudaMemcpy2DAsync(ix->q_all.p, (size_t)nqp * ix->dimp * 4, ix->x_all.p + (size_t)C + 1, B4 * sizeof(uint4),
                                          (size_t)nqp * ix->dimp * 4, G, cudaMemcpyDeviceToDevice, s));
            launch_own_flags(G, C, B4, ix->x_all.p, ix->rank, ix->x_flags.p, ix->w_flag.p + 2, s);
            exclusive_scan_u32(ix->cub_tmp.p, ix->cub_tmp.bytes(), ix->x_flags.p, ix->x_pos.p, (size_t)C * G + 1, s);
            need_exchange = false;
            ix->st.last_total_launches += 3;
        }
        ZB_CUDA(cudaMemsetAsync(ix->v_pair_len.p, 0, (v_cap + 1) * 8, s));
        ZB_CUDA(cudaMemsetAsync(ix->v_ent_len.p, 0, (v_cap + 1) * 4, s));
        if (sharded) {
            const u32 C = ix->x_cap;
            launch_own_scatter(fs, G, C, (size_t)C + 1 + q4, ix->x_all.p, ix->x_flags.p, ix->x_pos.p, (u32)v_cap, tile_on ? 1u : 0u, (u32)ix->p_tile_min_rows,
                               (u32)top_k, ix->v_leaf.p, ix->v_np.p, ix->v_q.p, ix->v_w.p, ix->v_pair_len.p, ix->v_ent_len.p,
                               ix->v_done.p, s);
            launch_walker_offsets((u32)nw, ix->x_pos.p + (size_t)C * G, (u32)v_cap, ix->v_w.p, ix->w_off.p, s);
        } else {
            exclusive_scan_u32(ix->cub_tmp.p, ix->cub_tmp.bytes(), ix->w_counts.p, ix->w_off.p, nw + 1, s);
            launch_compact_visits(fs, (u32)nw, ix->vpw, ix->w_visits.p, ix->w_counts.p, ix->w_off.p, 1, 0, (u32)v_cap,
                                  tile_on ? 1u : 0u, (u32)ix->p_tile_min_rows, (u32)top_k, ix->v_leaf.p, ix->v_np.p, ix->v_q.p,
                                  ix->v_pair_len.p, ix->v_ent_len.p, ix->v_done.p, s);
        }
        exclusive_scan_u32(ix->cub_tmp.p, ix->cub_tmp.bytes(), ix->v_ent_len.p, ix->v_ent_off.p, v_cap + 1, s);
        exclusive_scan_u64(ix->cub_tmp.p, ix->cub_tmp.bytes(), ix->v_pair_len.p, ix->v_pair_off.p, v_cap + 1, s);
        launch_plan_totals(sharded ? ix->w_flag.p + 2 : ix->w_flag.p, ix->w_off.p, (u32)nw, (u32)v_cap, ix->v_ent_off.p, ix->v_pair_off.p,
                           sharded ? ix->w_flag.p + 3 : nullptr, ix->plan_totals.p, s);
        u64 h_tot[5] = {0, 0, 0, 0, 0};
        ZB_CUDA(cudaMemcpyAsync(h_tot, ix->plan_totals.p, 40, cudaMemcpyDeviceToHost, s));
        ix->sync();
        ix->st.last_total_launches += 6;
        if (h_tot[0]) {
            ZB_REQUIRE(h_tot[0] == 1, ZB_ERR_STATE, "forest deeper than %d levels", ZB_MAX_DEPTH);
            ix->vpw *= 2;  // a walker produced more visits than its region holds: grow and replan
            ZB_REQUIRE(ix->vpw <= (1u << 16), ZB_ERR_STATE, "visit plan does not converge");
            need_plan = true;
            continue;
        }
        if (sharded && h_tot[4] > ix->x_cap) {  // some rank packed more records than a block holds: every rank sees it
            ix->x_cap = (u32)std::min<u64>(h_tot[4] + h_tot[4] / 4 + 64, 0x7FFFFFFFull);
            need_exchange = true;
            continue;
        }
        nv = (u32)h_tot[1];
        if (nv > v_cap) {  // more visits than the local arrays hold: grow and compact again (no collective involved)
            v_cap = (u64)nv + nv / 4;
            continue;
        }
        total_slots = (u32)h_tot[2];
        total_pairs = h_tot[3];
        break;
    }
    ZB_CUDA(cudaEventRecord(ix->ev[1], s));
    ix->trace_mark("compact");

    // ---- fused leaf-tile scan for visits of large leaves (zb_scan.cu) ----
    ix->entries.ensure(total_slots ? total_slots : 1);
    ix->pair_key.ensure(total_pairs ? total_pairs : 1);
    u64 tile_pairs = 0, tile_visits = 0, moved = 0;
    u32 scan_launches = 0;
    ix->scan_ws.launched = false;
    if (nv && tile_on) {
        if (ix->opt.metric == ZB_METRIC_COSINE) {
            ix->q_rinv.ensure(nq);
            launch_rinv(d_q, nq, ix->dimp, ix->q_rinv.p, s);
        }
        // L2 / L2 squared, top_k <= 16, rows of 128 floats or more: the fused kernel scores through the dot product and a second
        // pass evaluates the exact distance of the few rows that can reach a visit's list (knob l2_filter: 0 off, 1 unless the
        // last batches had to rescan too many visits exactly, 2 always)
        ix->scan_ws.l2_filter = gen3 && ix->dimp >= 128 && (ix->p_l2_filter == 2 || (ix->p_l2_filter == 1 && ix->filter_backoff == 0));
        if (ix->filter_backoff > 0) --ix->filter_backoff;
        (gen3 ? tile_scan3 : tile_scan)(ix->scan_ws, fs, ix->bm_view(), ix->opt.metric, d_q, ix->q_rinv.p, (u32)nq, nv, ix->v_leaf.p,
                                        ix->v_np.p, ix->v_q.p, ix->v_ent_off.p, ix->v_pair_len.p, ix->v_done.p, ix->entries.p,
                                        (u32)top_k, (u32)ix->p_tile_min_rows, (u32)ix->p_tile_queries,
                                        (u32)ix->h_leaf_off.size(), s);
        ZB_REQUIRE(ix->scan_ws.launched, ZB_ERR_STATE, "tile scan did not launch for visits set aside for it");
        scan_launches = ix->scan_ws.launches + (ix->opt.metric == ZB_METRIC_COSINE ? 1 : 0);
    }

    // ---- generic path for the remaining visits (pair offsets were scanned with the plan) ----
    // scalar metrics (sequential fold per pair): visits grouped by leaf, one thread folds a row against the <= 8 queries of a
    // tile, keys land in the same pair_key layout (zb_scan.cu, seq_tile_scan); knob seq_tile = 0 keeps one thread per pair
    ix->scan_ws.seq_launched = false;
    if (ix->opt.metric > ZB_METRIC_L2 && ix->p_seq_tile && total_pairs && seq_tile_scan_supported(ix->dimp))
        seq_tile_scan(ix->scan_ws, fs, ix->opt.metric, (int)ix->opt.metric_power, d_q, nv, ix->v_leaf.p, ix->v_q.p, ix->v_pair_off.p,
                      ix->pair_key.p, (u32)ix->h_leaf_off.size(), (int)ix->p_seq_prefetch, s);
    ix->qt_ws.seq_launched = false;
    if (ix->opt.metric <= ZB_METRIC_L2 && ix->p_quad_tile && total_pairs && quad_tile_scan_supported(ix->dimp))
        quad_tile_scan(ix->qt_ws, fs, ix->opt.metric, d_q, nv, ix->v_leaf.p, ix->v_q.p, ix->v_pair_off.p, ix->pair_key.p,
                       (u32)ix->h_leaf_off.size(), s);
    if (!ix->scan_ws.seq_launched && !ix->qt_ws.seq_launched)
        launch_score_pairs(fs, (int)ix->opt.metric, (int)ix->opt.metric_power, d_q, nv, ix->v_leaf.p, ix->v_q.p, ix->v_pair_off.p,
                           total_pairs, ix->pair_key.p, s);
    ZB_CUDA(cudaEventRecord(ix->ev[2], s));
    ix->trace_mark("scan");
    if (total_pairs)
        launch_select_visits(fs, nv, ix->v_leaf.p, ix->v_np.p, ix->v_pair_off.p, ix->pair_key.p, ix->v_ent_off.p,
                             ix->entries.p, ix->v_done.p, (u32)top_k, (int)ix->p_select_variant, s);
    ZB_CUDA(cudaEventRecord(ix->ev[3], s));
    ix->trace_mark("select");
    if (sharded) {
        // every visit was scored, whole, by the rank that owns its leaf (Q2's per-visit top-n' is already global): reduce my
        // visits to a per-query local top-k; all-to-all: the lists of query slice r go to rank r, which merges the G lists of
        // each of its queries; the finished slices are allgathered.
        const u64 nsk = nqp * top_k;          // u64 per (rank, array) slice
        const u64 nqP = nqp * G;
        u64* loc_ord = nullptr;
        u64* loc_bits = nullptr;
        ix->loc_results.ensure(2 * nqP * top_k + 1);
        loc_ord = ix->loc_results.p;
        loc_bits = loc_ord + nqP * top_k;
        if (nqP > nq) {  // padding queries of the last slice: empty lists
            ZB_CUDA(cudaMemsetAsync(loc_ord + nq * top_k, 0xFF, (nqP - nq) * top_k * 8, s));
            ZB_CUDA(cudaMemsetAsync(loc_bits + nq * top_k, 0xFF, (nqP - nq) * top_k * 8, s));
        }
        ix->o_counts.ensure(nq);
        launch_merge_queries((u32)nq, T, ix->w_off.p, ix->v_ent_off.p, ix->entries.p, (u32)top_k, loc_ord, loc_bits, ix->o_counts.p, s);
        ix->trace_mark("local merge");
        u64* gath = reinterpret_cast<u64*>((ix->gathered.ensure((size_t)nsk * G + 1), ix->gathered.p));  // [G][ord nsk | bits nsk]
        ix->nccl.group_start();
        for (u32 r = 0; r < G; ++r) {
            if (r == ix->rank) continue;
            ix->nccl.send(loc_ord + (u64)r * nsk, nsk * 8, (int)r, s);
            ix->nccl.send(loc_bits + (u64)r * nsk, nsk * 8, (int)r, s);
            ix->nccl.recv(gath + (u64)r * 2 * nsk, nsk * 8, (int)r, s);
            ix->nccl.recv(gath + (u64)r * 2 * nsk + nsk, nsk * 8, (int)r, s);
        }
        ix->nccl.group_end();
        ZB_CUDA(cudaMemcpyAsync(gath + (u64)ix->rank * 2 * nsk, loc_ord + (u64)ix->rank * nsk, nsk * 8, cudaMemcpyDeviceToDevice, s));
        ZB_CUDA(cudaMemcpyAsync(gath + (u64)ix->rank * 2 * nsk + nsk, loc_bits + (u64)ix->rank * nsk, nsk * 8, cudaMemcpyDeviceToDevice, s));
        ix->trace_mark("all-to-all of local top-k");
        if (sliced) {  // the finished slice is this rank's answer: nothing else to exchange
            launch_merge_gathered((u32)qn, (u32)nqp, (u32)top_k, G, gath, d_out_ord, d_out_bits, d_out_counts, s);
            ix->trace_mark("final merge of my slice");
        } else {
            const u64 blk = 2 * nsk + (nqp + 1) / 2;  // [ord nsk | bits nsk | counts nqp u32]
            ix->res_all.ensure(blk * G + 1);
            u64* mine = ix->res_all.p + (u64)ix->rank * blk;
            launch_merge_gathered((u32)qn, (u32)nqp, (u32)top_k, G, gath, mine, mine + nsk, reinterpret_cast<u32*>(mine + 2 * nsk), s);
            ix->trace_mark("final merge of my slice");
            ix->nccl.allgather(mine, ix->res_all.p, blk * 8, s);
            launch_unpack_results(ix->res_all.p, blk, (u32)nq, (u32)nqp, (u32)top_k, d_out_ord, d_out_bits, d_out_counts, s);
        }
    } else {
        launch_merge_queries((u32)nq, T, ix->w_off.p, ix->v_ent_off.p, ix->entries.p, (u32)top_k, d_out_ord, d_out_bits,
                             d_out_counts, s);
    }
    ZB_CUDA(cudaEventRecord(ix->ev[4], s));
    ix->trace_mark(sharded ? "allgather of results" : "merge");
    float tile_ms = 0.f;
    u32 tiles = 0;
    u64 unique_bytes = 0;
    u64 flagged = 0, refined = 0;
    float refine_ms = 0.f;
    tile_scan_stats(ix->scan_ws, s, &tile_visits, &tile_pairs, &moved, &tile_ms, &tiles, &unique_bytes, &flagged, &refined, &refine_ms);
    ix->st.last_unique_bytes = unique_bytes;
    ix->st.last_filter_flagged = (u32)std::min<u64>(flagged, 0xFFFFFFFFull);
    ix->st.last_filter_rows = (u32)std::min<u64>(refined, 0xFFFFFFFFull);
    ix->st.last_ms_refine = refine_ms;
    ix->st.last_filter_used = ix->scan_ws.launched && ix->scan_ws.filtered ? 1u : 0u;
    if (ix->scan_ws.launched && ix->scan_ws.filtered && flagged * 16 > tile_visits) ix->filter_backoff = 32;  // crowded keys: the exact kernel is cheaper
    u64 seq_moved = 0;
    if (ix->scan_ws.seq_launched) seq_tile_scan_stats(ix->scan_ws, s, &seq_moved, &tile_ms, &tiles);
    u64 qt_moved = 0;
    if (ix->qt_ws.seq_launched) {  // next to the fused kernel (if it ran too): times and tiles add up
        float qt_ms = 0.f;
        u32 qt_tiles = 0;
        seq_tile_scan_stats(ix->qt_ws, s, &qt_moved, &qt_ms, &qt_tiles);
        tile_ms += qt_ms;
        tiles += qt_tiles;
    }
    ix->st.last_ms_tile_kernel = tile_ms;
    ix->st.last_tiles = tiles;
    ix->sync();
    float ms;
    ix->trace_dump();
    cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]); ix->st.last_ms_plan = ms;
    cudaEventElapsedTime(&ms, ix->ev[1], ix->ev[2]); ix->st.last_ms_scan = ms;
    cudaEventElapsedTime(&ms, ix->ev[2], ix->ev[3]); ix->st.last_ms_select = ms;
    cudaEventElapsedTime(&ms, ix->ev[3], ix->ev[4]); ix->st.last_ms_merge = ms;
    cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[4]); ix->st.last_ms_total = ms;
    ix->st.last_visits = nv;
    ix->st.last_pairs = total_pairs + tile_pairs;
    ix->st.last_tile_visits = tile_visits;
    ix->st.last_tile_pairs = tile_pairs;
    ix->st.last_moved_bytes = ix->scan_ws.seq_launched ? seq_moved
                              : (ix->qt_ws.seq_launched ? moved + qt_moved : moved + total_pairs * (u64)ix->dim * 4);
    ix->st.last_scan_launches = scan_launches + (total_pairs ? (ix->scan_ws.seq_launched ? 7 : 1) : 0);
    // generic-path launches: the score kernel (or the 7 of seq_tile_scan: count, scan, scatter, tile count, scan, fill, scan
    // kernel) + select; then the merge
    ix->st.last_total_launches += scan_launches + 5 + (sharded ? 1 : 0) + ((ix->scan_ws.seq_launched || ix->qt_ws.seq_launched) ? 6 : 0);
}

// Exact search (zb_index_search_exact*): the top_k smallest (bits, ordinal) over every live row of the raw store.  Each rank
// scans the rows it owns; a sharded call allgathers the ranks' per-query lists and merges them (the same exchange as the
// unsliced search).  Queries go in chunks that keep the workspace within the exact_budget_mb knob; the plan comes from the
// largest row count of all ranks, so every rank runs the same sequence of collectives.
static void exact_device(zb_index* ix, u64 nq, const float* d_q, u64 top_k, u64* d_out_ord, u64* d_out_bits, u32* d_out_counts) {
    cudaStream_t s = ix->stream;
    if (!nq) return;
    if (!top_k) {
        ZB_CUDA(cudaMemsetAsync(d_out_counts, 0, nq * 4, s));
        return;
    }
    const u32 G = ix->G;
    const bool sharded = G > 1;
    u64 n_max = ix->n_slots;
    if (sharded) {
        ix->ex_nmax.ensure(1);
        ZB_CUDA(cudaMemcpyAsync(ix->ex_nmax.p, &n_max, 8, cudaMemcpyHostToDevice, s));
        ix->nccl.allreduce(ix->ex_nmax.p, 1, Nccl::U64, Nccl::MAX, s);
        ZB_CUDA(cudaMemcpyAsync(&n_max, ix->ex_nmax.p, 8, cudaMemcpyDeviceToHost, s));
        ix->sync();
    }
    const u32 metric = ix->opt.metric;
    // L2 / L2 squared with short lists go through the dot-product filter, as in the LSH search (DESIGN 3.8: measured on config 2)
    const bool filt = (metric == ZB_METRIC_L2SQ || metric == ZB_METRIC_L2) && top_k <= ZB_L2_FILTER_MAX_K && ix->dimp >= 128;
    ix->ensure_exact_side();
    // per query: q_rinv / q_n2 / shared bound, and (sharded) its local lists plus the G gathered ones
    const u64 per_query = 24 + (sharded ? 16 * top_k * (G + 1) + 4 : 0);
    const ExactPlan p = exact_plan(n_max, nq, ix->dimp, (u32)top_k, filt, per_query, (u64)ix->p_exact_budget_mb << 20);
    ForestView store = ix->view();
    store.members = ix->ex_iota.p;
    BucketMajor bm;
    bm.rows = ix->rows.p;
    bm.tomb = ix->tomb.p;
    bm.rinv = metric == ZB_METRIC_COSINE ? ix->ex_rinv.p : nullptr;
    bm.n2 = filt ? ix->ex_n2.p : nullptr;
    alignas(64) unsigned char tmap[128];
    if (ix->n_slots) make_row_tile_map(tmap, ix->rows.p, ix->n_slots, ix->dimp, 64, tile_scan_box_floats(3));
    bm.tmap3 = tmap;
    bm.positions = ix->n_slots;
    for (u64 c0 = 0; c0 < nq; c0 += p.chunk) {
        const u64 c = std::min<u64>(p.chunk, nq - c0);
        const float* q = d_q + c0 * (u64)ix->dimp;
        if (!sharded) {
            exact_scan3(ix->ex_ws, store, bm, ix->n_slots, metric, q, (u32)c, p.range_rows, (u32)top_k, filt, d_out_ord + c0 * top_k,
                        d_out_bits + c0 * top_k, d_out_counts + c0, s);
            continue;
        }
        const u64 nsk = c * top_k;   // [ord nsk | bits nsk] per rank, the layout merge_gathered reads
        ix->ex_loc.ensure(2 * p.chunk * top_k);
        ix->ex_gath.ensure(2 * p.chunk * top_k * G);
        ix->ex_counts.ensure(p.chunk);
        exact_scan3(ix->ex_ws, store, bm, ix->n_slots, metric, q, (u32)c, p.range_rows, (u32)top_k, filt, ix->ex_loc.p,
                    ix->ex_loc.p + nsk, ix->ex_counts.p, s);
        ix->nccl.allgather(ix->ex_loc.p, ix->ex_gath.p, 2 * nsk * 8, s);
        launch_merge_gathered((u32)c, (u32)c, (u32)top_k, G, ix->ex_gath.p, d_out_ord + c0 * top_k, d_out_bits + c0 * top_k,
                              d_out_counts + c0, s);
    }
    ix->sync();
}

static const float* stage_queries_device(zb_index* ix, const float* d_q, u64 nq) {
    if (ix->dim == ix->dimp && ((uintptr_t)d_q & 15) == 0) return d_q;
    ix->q_stage.ensure(nq * (u64)ix->dimp);
    launch_pad_rows(d_q, nq, ix->dim, ix->dimp, ix->q_stage.p, ix->stream);
    return ix->q_stage.p;
}

static void build_export_table(zb_index* ix, std::vector<int>* order_nodes, std::vector<int>* leaf_export) {
    // preorder numbering (node, left subtree, right subtree), trees in order -- the oracle's numbering
    leaf_export->assign(ix->h_leaf_off.size(), -1);
    int next_leaf = 0;
    std::vector<int> stack;
    for (int t = 0; t < ix->T && ix->built; ++t) {
        stack.push_back(ix->h_roots[t]);
        while (!stack.empty()) {
            int n = stack.back();
            stack.pop_back();
            if (order_nodes) order_nodes->push_back(n);
            int4 nd = ix->h_nodes[n];
            if (nd.x < 0) (*leaf_export)[nd.w] = next_leaf++;
            else {
                stack.push_back(nd.z);
                stack.push_back(nd.y);
            }
        }
    }
}

}  // namespace zb

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

const char* zb_last_error(void) { return zb::t_last_error.c_str(); }
int zb_abi_version(void) { return ZB_ABI_VERSION; }

int zb_device_count(int* out_count) {
    ZB_API_BEGIN
    ZB_REQUIRE(out_count, ZB_ERR_INVALID, "out_count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    *out_count = n;
    ZB_API_END
}

int zb_index_create(const zb_options* o, zb_index** out) {
    ZB_API_BEGIN
    ZB_REQUIRE(o && out, ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(o->dim >= 1 && o->dim <= 65536, ZB_ERR_INVALID, "dim %u out of range", o->dim);
    ZB_REQUIRE(o->metric < ZB_METRIC_COUNT, ZB_ERR_INVALID, "metric %u is not a zb_metric", o->metric);
    ZB_REQUIRE((o->metric != ZB_METRIC_MINKOWSKI && o->metric != ZB_METRIC_PNORM) ||
                   (o->metric_power >= 0 && o->metric_power <= ZB_METRIC_MAX_POWER),
               ZB_ERR_INVALID, "metric_power %d out of range 0..%d", o->metric_power, ZB_METRIC_MAX_POWER);
    ZB_REQUIRE(o->num_trees >= 1 && o->num_trees <= 4096, ZB_ERR_INVALID, "num_trees %u out of range", o->num_trees);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        throw zb::Error(ZB_ERR_NO_DEVICE, "no CUDA device: libzebra_b200 has no CPU fallback");
    }
    ZB_REQUIRE(o->device >= 0 && o->device < ndev, ZB_ERR_INVALID, "device %d out of range (%d devices)", o->device, ndev);
    cudaDeviceProp prop;
    ZB_CUDA(cudaGetDeviceProperties(&prop, o->device));
    ZB_REQUIRE(prop.major == 10, ZB_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
               o->device, prop.major, prop.minor);
    zb_index* ix = new zb_index();
    ix->opt = *o;
    ix->dim = (int)o->dim;
    ix->dimp = (ix->dim + 15) / 16 * 16;
    ix->chunks = ix->dimp / 16;
    ix->T = (int)o->num_trees;
    ix->device = o->device;
    ix->G = o->shard_count > 1 ? o->shard_count : 1;
    ix->rank = ix->G > 1 ? o->shard_rank : 0;
    ZB_REQUIRE(ix->rank < ix->G, ZB_ERR_INVALID, "shard_rank %u >= shard_count %u", ix->rank, ix->G);
    ix->use_device();
    ZB_CUDA(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    for (auto& ev : ix->ev) ZB_CUDA(cudaEventCreate(&ev));
    ix->epoch_ms = (u64)std::chrono::duration_cast<std::chrono::milliseconds>(
                       std::chrono::system_clock::now().time_since_epoch()).count() & 0xFFFFFFFFFFFFull;
    ix->h_roots.assign(ix->T, -1);
    *out = ix;
    ZB_API_END
}

int zb_index_destroy(zb_index* ix) {
    ZB_API_BEGIN
    if (!ix) return ZB_OK;
    cudaSetDevice(ix->device);
    cudaStreamSynchronize(ix->stream);
    ix->release_peer_queries();
    if (ix->pq.fork) {
        cudaEventDestroy(ix->pq.fork);
        for (int i = 0; i < zb_index::PeerQ::NS; ++i) {
            cudaStreamDestroy(ix->pq.stream[i]);
            cudaEventDestroy(ix->pq.done[i]);
        }
    }
    ix->nccl.destroy();
    for (auto& ev : ix->ev) cudaEventDestroy(ev);
    if (ix->copy_stream) {
        cudaStreamSynchronize(ix->copy_stream);
        cudaStreamDestroy(ix->copy_stream);
    }
    for (auto& p : ix->pf)
        if (p.done) cudaEventDestroy(p.done);
    cudaStreamDestroy(ix->stream);
    delete ix;
    ZB_API_END
}

static void add_common(zb_index* ix, u64 n, const float* src, bool src_on_device, const uint8_t* ids16, uint8_t* out_ids16,
                       u64* out_ordinals) {
    auto t0 = std::chrono::steady_clock::now();
    ix->use_device();
    if (ix->G > 1) ZB_REQUIRE(ix->comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
    // Ids: an index holds either library-minted ids (mode 1: id <-> ordinal is arithmetic) or registered ids (mode 2: a map).
    // Rows without ids may be added to a mode-2 index (one reopened from a store, Database::open -> insert_records): their
    // ids are minted and registered like the caller's.  The whole batch is validated before anything is committed.
    const bool registered = ids16 || (ix->id_mode == 2 && n);
    const u64 first = ix->total_rows;
    std::vector<Id16> new_ids;
    if (n) {
        ZB_REQUIRE(ix->id_mode == 0 || ix->id_mode == (registered ? 2 : 1), ZB_ERR_INVALID,
                   "ids must be supplied for every row of an index or for none");
        if (registered) {
            new_ids.resize(n);
            std::unordered_map<Id16, u64, Id16Hash> batch;
            batch.reserve(n);
            for (u64 i = 0; i < n; ++i) {
                const Id16 id = ids16 ? Id16{load_be64(ids16 + 16 * i), load_be64(ids16 + 16 * i + 8)} : ix->mint(first + i);
                ZB_REQUIRE(ix->ordinal_by_id.find(id) == ix->ordinal_by_id.end() && batch.emplace(id, i).second, ZB_ERR_INVALID,
                           "duplicate id at row %llu", (unsigned long long)i);
                new_ids[i] = id;
            }
        }
    }
    // rows this shard owns
    std::vector<u64> ordinals;
    u64 i0 = 0;
    if (ix->G > 1) {
        i0 = (ix->rank + ix->G - first % ix->G) % ix->G;
        for (u64 i = i0; i < n; i += ix->G) ordinals.push_back(first + i);
    } else {
        ordinals.resize(n);
        for (u64 i = 0; i < n; ++i) ordinals[i] = first + i;
    }
    const u64 nloc = ordinals.size();
    const u64 first_slot = ix->n_slots;
    if (nloc) {
        const u64 stride = (u64)ix->dim * ix->G;
        if (src_on_device) {
            ix->append_rows_device(src + i0 * (u64)ix->dim, stride, nloc, ordinals.data());
        } else {
            ix->r_stage.ensure(nloc * (u64)ix->dim);
            ZB_CUDA(cudaMemcpy2DAsync(ix->r_stage.p, (size_t)ix->dim * 4, src + i0 * (u64)ix->dim, stride * 4,
                                      (size_t)ix->dim * 4, nloc, cudaMemcpyHostToDevice, ix->stream));
            ix->append_rows_device(ix->r_stage.p, ix->dim, nloc, ordinals.data());
        }
    }
    if (n) ix->id_mode = registered ? 2 : 1;
    for (u64 i = 0; i < new_ids.size(); ++i) {
        ix->ordinal_by_id.emplace(new_ids[i], first + i);
        ix->ids_by_ordinal.push_back(new_ids[i]);
    }
    ix->total_rows += n;
    for (u64 i = 0; i < n; ++i) {
        if (out_ordinals) out_ordinals[i] = first + i;
        if (out_ids16) ix->id_of(first + i, out_ids16 + 16 * i);
    }
    auto t1 = std::chrono::steady_clock::now();
    if (!ix->built) {
        if (ix->total_rows > 0) ix->bulk_build();
    } else {
        ix->incremental_insert(first_slot, nloc);
    }
    if (ix->trace_on && ix->rank == 0)
        fprintf(stderr, "[zb trace] add: store %.3f ms, build/insert %.3f ms\n", std::chrono::duration<double, std::milli>(t1 - t0).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count());
}

int zb_index_add(zb_index* ix, uint64_t n, const float* rows, const uint8_t* ids16, uint8_t* out_ids16, uint64_t* out_ordinals) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (rows || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    add_common(ix, n, rows, false, ids16, out_ids16, (u64*)out_ordinals);
    ZB_API_END
}
int zb_index_add_device(zb_index* ix, uint64_t n, const float* d_rows, const uint8_t* ids16, uint8_t* out_ids16,
                        uint64_t* out_ordinals) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_rows || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    add_common(ix, n, d_rows, true, ids16, out_ids16, (u64*)out_ordinals);
    ZB_API_END
}
int zb_index_add_owned_device(zb_index* ix, uint64_t n_local, const float* d_rows, const uint64_t* ordinals, uint64_t total_n) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_rows || !n_local) && (ordinals || !n_local), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->use_device();
    if (ix->G > 1) ZB_REQUIRE(ix->comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
    ZB_REQUIRE(ix->id_mode != 2, ZB_ERR_INVALID, "owned-row loading needs library-minted ids");
    if (total_n) ix->id_mode = 1;
    for (u64 i = 0; i < n_local; ++i)
        ZB_REQUIRE(ix->owns(ordinals[i]) && ordinals[i] >= ix->total_rows && ordinals[i] < ix->total_rows + total_n &&
                       ix->slot_of(ordinals[i]) == ix->n_slots + i,
                   ZB_ERR_INVALID, "ordinal %llu is not the next row this shard owns", (unsigned long long)ordinals[i]);
    const u64 first_slot = ix->n_slots;
    ix->append_rows_device(d_rows, ix->dim, n_local, (const u64*)ordinals);
    ix->total_rows += total_n;
    if (!ix->built) {
        if (ix->total_rows > 0) ix->bulk_build();
    } else {
        ix->incremental_insert(first_slot, n_local);
    }
    ZB_API_END
}

static void remove_ordinals(zb_index* ix, u64 n, const u64* ordinals, const u8* valid, uint8_t* out_removed) {
    ix->use_device();
    std::vector<u32> slots(n);
    for (u64 i = 0; i < n; ++i) {
        bool ok = (!valid || valid[i]) && ordinals[i] < ix->total_rows && ix->owns(ordinals[i]) &&
                  ix->slot_of(ordinals[i]) < ix->n_slots;
        slots[i] = ok ? (u32)ix->slot_of(ordinals[i]) : 0xFFFFFFFFu;
    }
    std::vector<u8> flags(n, 0);
    if (n) {
        ix->rm_slots.ensure(n);
        ix->rm_flags.ensure(n);
        ZB_CUDA(cudaMemcpyAsync(ix->rm_slots.p, slots.data(), n * 4, cudaMemcpyHostToDevice, ix->stream));
        if (ix->built) {
            launch_tombstone(ix->rm_slots.p, (u32)n, ix->tomb.p, ix->slot_leaf.p, ix->slot_stride, ix->T, ix->d_leaf_live.p,
                             ix->rm_flags.p, ix->stream);
        } else {
            ZB_CUDA(cudaMemsetAsync(ix->rm_flags.p, 0, n, ix->stream));
        }
        if (ix->built && ix->bm_valid && ix->G <= 1)
            launch_bm_tombstone(ix->rm_slots.p, ix->rm_flags.p, (u32)n, ix->slot_pos.p, ix->slot_stride, ix->T, ix->bm_tomb.p, ix->stream);
        if (ix->G > 1) {
            ix->nccl.allreduce(ix->rm_flags.p, n, Nccl::U8, Nccl::MAX, ix->stream);
            if (ix->built && ix->bm_valid) {  // the copies of a removed row sit on the ranks that own its T leaves
                ix->rm_ords.ensure(n);
                ZB_CUDA(cudaMemcpyAsync(ix->rm_ords.p, ordinals, n * 8, cudaMemcpyHostToDevice, ix->stream));
                launch_bm_tomb_lookup(ix->rm_ords.p, ix->rm_flags.p, n, ix->T, ix->d_tree_base.p, ix->srt_ord.p, ix->srt_pos.p,
                                      ix->bm_tomb.p, ix->stream);
            }
        }
        ZB_CUDA(cudaMemcpyAsync(flags.data(), ix->rm_flags.p, n, cudaMemcpyDeviceToHost, ix->stream));
    }
    ix->refresh_plan_counts();
    ix->sync();
    for (u64 i = 0; i < n; ++i) {
        if (flags[i] && slots[i] != 0xFFFFFFFFu && !ix->h_tomb[slots[i]]) {
            ix->h_tomb[slots[i]] = 1;
            ix->n_live--;
        }
        if (out_removed) out_removed[i] = flags[i];
    }
}

int zb_index_remove_ordinals(zb_index* ix, uint64_t n, const uint64_t* ordinals, uint8_t* out_removed) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (ordinals || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    remove_ordinals(ix, n, (const u64*)ordinals, nullptr, out_removed);
    ZB_API_END
}
int zb_index_remove(zb_index* ix, uint64_t n, const uint8_t* ids16, uint8_t* out_removed) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (ids16 || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    std::vector<u64> ords(n, 0);
    std::vector<u8> valid(n, 0);
    for (u64 i = 0; i < n; ++i) valid[i] = ix->ordinal_of(ids16 + 16 * i, &ords[i]) ? 1 : 0;
    remove_ordinals(ix, n, ords.data(), valid.data(), out_removed);
    ZB_API_END
}

// LSHIndex::deduplicate (lsh.rs:270-288).  Unsharded: exact on the device (hash, sort, bitwise compare inside hash runs).
// Sharded: every rank hashes its rows (128 bits), the (hash, ordinal) records are allgathered and grouped on the host;
// rows with equal 128-bit hashes are taken as equal (no cross-rank row compare).  Either way the first row in id order of
// every group stays and the others go through the ordinary remove path (tombstones, live counts, bucket-major store).
static void deduplicate_impl(zb_index* ix, std::vector<u64>* removed) {
    ix->use_device();
    cudaStream_t s = ix->stream;
    removed->clear();
    // live slots in id order: minted ids order like ordinals (= slot order); caller-supplied ids order by their bytes
    std::vector<u32> live;
    live.reserve(ix->n_slots);
    for (u64 sl = 0; sl < ix->n_slots; ++sl)
        if (!ix->h_tomb[sl]) live.push_back((u32)sl);
    auto id_less = [&](u64 oa, u64 ob) {
        if (ix->id_mode != 2) return oa < ob;
        const Id16 &a = ix->ids_by_ordinal[oa], &b = ix->ids_by_ordinal[ob];
        return a.hi != b.hi ? a.hi < b.hi : (a.lo != b.lo ? a.lo < b.lo : oa < ob);
    };
    if (ix->id_mode == 2)
        std::stable_sort(live.begin(), live.end(), [&](u32 x, u32 y) { return id_less(ix->h_ord[x], ix->h_ord[y]); });
    const u64 n = live.size();
    DBuf<u32> d_slots, d_val[2], d_flag, d_head;
    DBuf<u64> d_h1[2], d_h2;
    DBuf<u8> d_dup, d_tmp;
    d_slots.ensure(n ? n : 1);
    d_h1[0].ensure(n ? n : 1);
    d_h2.ensure(n ? n : 1);
    if (n) ZB_CUDA(cudaMemcpyAsync(d_slots.p, live.data(), n * 4, cudaMemcpyHostToDevice, s));
    launch_row_hash(d_slots.p, n, ix->rows.p, ix->dimp, d_h1[0].p, d_h2.p, s);
    std::vector<u64> dups;
    if (ix->G <= 1) {
        d_h1[1].ensure(n ? n : 1);
        for (int b = 0; b < 2; ++b) d_val[b].ensure(n ? n : 1);
        d_flag.ensure(n ? n : 1);
        d_head.ensure(n ? n : 1);
        d_dup.ensure(n ? n : 1);
        d_tmp.ensure(std::max(sort_temp_bytes(n ? n : 1), maxscan_temp_bytes(n ? n : 1)));
        launch_iota_u32(d_val[0].p, n, 0u, s);
        sort_pairs_u64_u32(d_tmp.p, d_tmp.bytes(), d_h1[0].p, d_h1[1].p, d_val[0].p, d_val[1].p, n, 64, s);
        launch_dup_mark(d_h1[1].p, d_val[1].p, n, d_slots.p, ix->rows.p, ix->dimp, d_flag.p, d_head.p, d_tmp.p, d_tmp.bytes(), d_dup.p, s);
        std::vector<u8> h_dup(n);
        std::vector<u32> h_cand(n);
        if (n) {
            ZB_CUDA(cudaMemcpyAsync(h_dup.data(), d_dup.p, n, cudaMemcpyDeviceToHost, s));
            ZB_CUDA(cudaMemcpyAsync(h_cand.data(), d_val[1].p, n * 4, cudaMemcpyDeviceToHost, s));
        }
        ix->sync();
        for (u64 i = 0; i < n; ++i)
            if (h_dup[i]) dups.push_back(ix->h_ord[live[h_cand[i]]]);
    } else {
        ZB_REQUIRE(ix->comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
        // records (h1, h2, ordinal), padded to the largest shard
        u64 nmax = n;
        {
            ix->b_minh.ensure(1);
            ZB_CUDA(cudaMemcpyAsync(ix->b_minh.p, &nmax, 8, cudaMemcpyHostToDevice, s));
            ix->nccl.allreduce(ix->b_minh.p, 1, Nccl::U64, Nccl::MAX, s);
            ZB_CUDA(cudaMemcpyAsync(&nmax, ix->b_minh.p, 8, cudaMemcpyDeviceToHost, s));
            ix->sync();
        }
        std::vector<u64> rec(3 * (nmax ? nmax : 1), ZB_SENTINEL), h1(n), h2(n);
        if (n) {
            ZB_CUDA(cudaMemcpyAsync(h1.data(), d_h1[0].p, n * 8, cudaMemcpyDeviceToHost, s));
            ZB_CUDA(cudaMemcpyAsync(h2.data(), d_h2.p, n * 8, cudaMemcpyDeviceToHost, s));
        }
        ix->sync();
        for (u64 i = 0; i < n; ++i) {
            rec[3 * i] = h1[i];
            rec[3 * i + 1] = h2[i];
            rec[3 * i + 2] = ix->h_ord[live[i]];
        }
        DBuf<u64> d_rec, d_all;
        const size_t per = 3 * (nmax ? nmax : 1);
        d_rec.ensure(per);
        d_all.ensure(per * ix->G);
        ZB_CUDA(cudaMemcpyAsync(d_rec.p, rec.data(), per * 8, cudaMemcpyHostToDevice, s));
        ix->nccl.allgather(d_rec.p, d_all.p, per * 8, s);
        std::vector<u64> all(per * ix->G);
        ZB_CUDA(cudaMemcpyAsync(all.data(), d_all.p, all.size() * 8, cudaMemcpyDeviceToHost, s));
        ix->sync();
        struct Rec { u64 h1, h2, ord; };
        std::vector<Rec> v;
        for (size_t i = 0; i + 2 < all.size(); i += 3)
            if (all[i + 2] != ZB_SENTINEL) v.push_back(Rec{all[i], all[i + 1], all[i + 2]});
        std::sort(v.begin(), v.end(), [&](const Rec& a, const Rec& b) {
            return a.h1 != b.h1 ? a.h1 < b.h1 : (a.h2 != b.h2 ? a.h2 < b.h2 : id_less(a.ord, b.ord));
        });
        for (size_t i = 1; i < v.size(); ++i)
            if (v[i].h1 == v[i - 1].h1 && v[i].h2 == v[i - 1].h2) dups.push_back(v[i].ord);
    }
    std::sort(dups.begin(), dups.end());
    if (!dups.empty() || ix->G > 1) {
        std::vector<u8> flags(dups.size() ? dups.size() : 1, 0);
        remove_ordinals(ix, dups.size(), dups.data(), nullptr, flags.data());
    }
    *removed = dups;
}

int zb_index_deduplicate(zb_index* ix, uint64_t* out_count, uint64_t* out_ordinals, uint8_t* out_ids16, uint64_t cap) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out_count, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    std::vector<u64> removed;
    deduplicate_impl(ix, &removed);
    *out_count = removed.size();
    for (u64 i = 0; i < removed.size() && i < cap; ++i) {
        if (out_ordinals) out_ordinals[i] = removed[i];
        if (out_ids16) ix->id_of(removed[i], out_ids16 + 16 * i);
    }
    ZB_API_END
}

static void clear_locked(zb_index* ix);
int zb_index_clear(zb_index* ix) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    clear_locked(ix);
    ZB_API_END
}

int zb_index_no_vectors(zb_index* ix, int* out) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    u64 live = ix->n_live;
    if (ix->G > 1) {
        ix->use_device();
        live = ix->allreduce_sum_u64(live);
    }
    *out = live == 0;
    ZB_API_END
}
int zb_index_no_trees(zb_index* ix, int* out) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    *out = !ix->built;
    ZB_API_END
}

// Batches beyond 131072 queries are cut into chunks (walker count < 2^31, bounded workspaces).  sliced: see search_device;
// the chunks of a sliced call are chunks of the whole batch, so every rank sees the same sequence of collectives.
static void search_entry_device(zb_index* ix, u64 nq, const float* d_q, u64 top_k, u32 probes, u64* d_out_ord, u64* d_out_bits,
                                u32* d_out_counts, bool sliced, bool exact = false) {
    ix->use_device();
    const u64 G = ix->G;
    sliced = sliced && G > 1;
    const u64 chunk = sliced ? 131072 / G * G : 131072;
    u64 in_off = 0;  // queries consumed from d_q / results written so far (sliced: of this rank's slices)
    for (u64 c0 = 0; c0 < nq; c0 += chunk) {
        const u64 c = std::min<u64>(chunk, nq - c0);
        u64 mine = c;
        if (sliced) {
            const u64 nqp = (c + G - 1) / G, lo = std::min<u64>(c, ix->rank * nqp);
            mine = std::min<u64>(nqp, c - lo);
        }
        const float* q = stage_queries_device(ix, d_q + in_off * (u64)ix->dim, mine);
        if (exact) exact_device(ix, c, q, top_k, d_out_ord + in_off * top_k, d_out_bits + in_off * top_k, d_out_counts + in_off);
        else search_device(ix, c, q, top_k, probes, d_out_ord + in_off * top_k, d_out_bits + in_off * top_k, d_out_counts + in_off, sliced);
        in_off += mine;
    }
    ix->sync();
}

int zb_index_search_batch_device(zb_index* ix, uint64_t nq, const float* d_q, uint64_t top_k, uint64_t* d_out_ord,
                                 uint64_t* d_out_bits, uint32_t* d_out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_q || !nq) && ((d_out_ord && d_out_bits && d_out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(top_k <= ZB_MAX_TOPK, ZB_ERR_INVALID, "top_k %llu exceeds %d", (unsigned long long)top_k, ZB_MAX_TOPK);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_device(ix, nq, d_q, top_k, 0, (u64*)d_out_ord, (u64*)d_out_bits, d_out_counts, false);
    ZB_API_END
}
int zb_index_search_slice_device(zb_index* ix, uint64_t nq_total, const float* d_q, uint64_t top_k, uint64_t* d_out_ord,
                                 uint64_t* d_out_bits, uint32_t* d_out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(top_k <= ZB_MAX_TOPK, ZB_ERR_INVALID, "top_k %llu exceeds %d", (unsigned long long)top_k, ZB_MAX_TOPK);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_device(ix, nq_total, d_q, top_k, 0, (u64*)d_out_ord, (u64*)d_out_bits, d_out_counts, true);
    ZB_API_END
}

// Host buffers in, host buffers out.  sliced: `queries` and the outputs hold this rank's slices only.
static void search_entry_host(zb_index* ix, u64 nq, const float* queries, u64 top_k, u32 probes, uint8_t* out_ids16,
                              u64* out_ordinals, u64* out_bits, u32* out_counts, bool sliced, bool exact = false) {
    ix->use_device();
    cudaStream_t s = ix->stream;
    const u64 G = ix->G;
    sliced = sliced && G > 1;
    const u64 chunk = sliced ? 131072 / G * G : 131072;
    std::vector<u64> ord_tmp;
    u64 in_off = 0;
    for (u64 c0 = 0; c0 < nq; c0 += chunk) {
        const u64 c = std::min<u64>(chunk, nq - c0);
        u64 mine = c;
        if (sliced) {
            const u64 nqp = (c + G - 1) / G, lo = std::min<u64>(c, ix->rank * nqp);
            mine = std::min<u64>(nqp, c - lo);
        }
        bool staged = false;
        if (c0 == 0 && mine && !exact) {  // announced by zb_index_search_prefetch: the rows are (being) copied on the copy stream
            for (auto& p : ix->pf)
                if (p.host == queries && p.rows >= mine && nq <= chunk) {
                    ZB_CUDA(cudaStreamWaitEvent(s, p.done, 0));
                    std::swap(ix->q_stage.p, p.buf.p);
                    std::swap(ix->q_stage.cap, p.buf.cap);
                    p.host = nullptr;
                    staged = true;
                    break;
                }
        }
        ix->q_stage.ensure(std::max<u64>(1, mine * (u64)ix->dimp));
        if (mine && !staged) {
            if (ix->dim == ix->dimp) {
                ZB_CUDA(cudaMemcpyAsync(ix->q_stage.p, queries + in_off * (u64)ix->dim, mine * (u64)ix->dim * 4, cudaMemcpyHostToDevice, s));
            } else {
                ZB_CUDA(cudaMemsetAsync(ix->q_stage.p, 0, mine * (u64)ix->dimp * 4, s));
                ZB_CUDA(cudaMemcpy2DAsync(ix->q_stage.p, (size_t)ix->dimp * 4, queries + in_off * (u64)ix->dim, (size_t)ix->dim * 4,
                                          (size_t)ix->dim * 4, mine, cudaMemcpyHostToDevice, s));
            }
        }
        ix->o_ord.ensure(mine * top_k + 1);
        ix->o_bits.ensure(mine * top_k + 1);
        ix->o_counts2.ensure(mine + 1);
        if (exact) exact_device(ix, c, ix->q_stage.p, top_k, ix->o_ord.p, ix->o_bits.p, ix->o_counts2.p);
        else search_device(ix, c, ix->q_stage.p, top_k, probes, ix->o_ord.p, ix->o_bits.p, ix->o_counts2.p, sliced);
        if (!out_ordinals && out_ids16) ord_tmp.resize(mine * top_k);
        u64* ords = out_ordinals ? out_ordinals + in_off * top_k : ord_tmp.data();
        if (top_k && mine) {
            if (out_ordinals || out_ids16) ZB_CUDA(cudaMemcpyAsync(ords, ix->o_ord.p, mine * top_k * 8, cudaMemcpyDeviceToHost, s));
            ZB_CUDA(cudaMemcpyAsync(out_bits + in_off * top_k, ix->o_bits.p, mine * top_k * 8, cudaMemcpyDeviceToHost, s));
        }
        if (mine) ZB_CUDA(cudaMemcpyAsync(out_counts + in_off, ix->o_counts2.p, mine * 4, cudaMemcpyDeviceToHost, s));
        ix->sync();
        if (out_ids16) {
            for (u64 i = 0; i < mine * top_k; ++i) {
                uint8_t* dst = out_ids16 + (in_off * top_k + i) * 16;
                if (ords[i] == ZB_SENTINEL) memset(dst, 0xFF, 16);
                else ix->id_of(ords[i], dst);
            }
        }
        in_off += mine;
    }
}

int zb_index_search_batch(zb_index* ix, uint64_t nq, const float* queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_bits, uint32_t* out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (queries || !nq) && ((out_bits && out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(top_k <= ZB_MAX_TOPK, ZB_ERR_INVALID, "top_k %llu exceeds %d", (unsigned long long)top_k, ZB_MAX_TOPK);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_host(ix, nq, queries, top_k, 0, out_ids16, (u64*)out_ordinals, (u64*)out_bits, out_counts, false);
    ZB_API_END
}
static void exact_check(zb_index* ix, u64 top_k) {
    ZB_REQUIRE(ix->opt.metric <= ZB_METRIC_L2, ZB_ERR_INVALID, "exact search serves cosine, L2 squared and L2, not metric %u",
               ix->opt.metric);
    ZB_REQUIRE(top_k <= ZB_EXACT_MAX_K, ZB_ERR_INVALID, "exact search: top_k %llu exceeds %d", (unsigned long long)top_k,
               ZB_EXACT_MAX_K);
    ix->use_device();
    ZB_REQUIRE(tile_scan3_supported(ix->dimp, top_k ? (u32)top_k : 1u), ZB_ERR_INVALID,
               "exact search: %d dimensions exceed the fused scan's limit for top_k %llu", ix->dim, (unsigned long long)top_k);
    if (ix->G > 1) ZB_REQUIRE(ix->comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
}
int zb_index_search_exact(zb_index* ix, uint64_t nq, const float* queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_bits, uint32_t* out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (queries || !nq) && ((out_bits && out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    exact_check(ix, top_k);
    search_entry_host(ix, nq, queries, top_k, 0, out_ids16, (u64*)out_ordinals, (u64*)out_bits, out_counts, false, true);
    ZB_API_END
}
int zb_index_search_exact_device(zb_index* ix, uint64_t nq, const float* d_q, uint64_t top_k, uint64_t* d_out_ord,
                                 uint64_t* d_out_bits, uint32_t* d_out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_q || !nq) && ((d_out_ord && d_out_bits && d_out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    exact_check(ix, top_k);
    search_entry_device(ix, nq, d_q, top_k, 0, (u64*)d_out_ord, (u64*)d_out_bits, d_out_counts, false, true);
    ZB_API_END
}
int zb_index_search_prefetch(zb_index* ix, uint64_t n, const float* queries) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (queries || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!n) return ZB_OK;
    ix->use_device();
    if (!ix->copy_stream) {  // highest priority: the upload must not queue behind the scan's own memsets / device copies
        int lo = 0, hi = 0;
        ZB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        ZB_CUDA(cudaStreamCreateWithPriority(&ix->copy_stream, cudaStreamNonBlocking, hi));
    }
    zb_index::Prefetch* slot = nullptr;
    for (auto& p : ix->pf)
        if (p.host == queries) slot = &p;            // announced again: refresh
    if (!slot)
        for (auto& p : ix->pf)
            if (!p.host) { slot = &p; break; }       // a free slot
    if (!slot) slot = ix->pf[0].seq < ix->pf[1].seq ? &ix->pf[0] : &ix->pf[1];  // both pending: the older announcement goes
    if (!slot->done) ZB_CUDA(cudaEventCreateWithFlags(&slot->done, cudaEventDisableTiming));
    // the slot's buffer may still be read by a search in flight on the main stream only if it was swapped in: it is not (a
    // swapped-in buffer belongs to q_stage); searches are synchronous, so whatever used this buffer before has completed
    slot->buf.ensure(n * (u64)ix->dimp);
    if (ix->dim == ix->dimp) {
        ZB_CUDA(cudaMemcpyAsync(slot->buf.p, queries, n * (u64)ix->dim * 4, cudaMemcpyHostToDevice, ix->copy_stream));
    } else {
        ZB_CUDA(cudaMemsetAsync(slot->buf.p, 0, n * (u64)ix->dimp * 4, ix->copy_stream));
        ZB_CUDA(cudaMemcpy2DAsync(slot->buf.p, (size_t)ix->dimp * 4, queries, (size_t)ix->dim * 4, (size_t)ix->dim * 4, n,
                                  cudaMemcpyHostToDevice, ix->copy_stream));
    }
    ZB_CUDA(cudaEventRecord(slot->done, ix->copy_stream));
    slot->host = queries;
    slot->rows = n;
    slot->seq = ++ix->pf_seq;
    ZB_API_END
}
int zb_index_search_slice(zb_index* ix, uint64_t nq_total, const float* queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_bits, uint32_t* out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(top_k <= ZB_MAX_TOPK, ZB_ERR_INVALID, "top_k %llu exceeds %d", (unsigned long long)top_k, ZB_MAX_TOPK);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_host(ix, nq_total, queries, top_k, 0, out_ids16, (u64*)out_ordinals, (u64*)out_bits, out_counts, true);
    ZB_API_END
}

// Multi-probe forms of the four search calls (DESIGN 3.9); probes = 0 is the plain call.
static void probe_check(u64 top_k, u32 probes) {
    ZB_REQUIRE(top_k <= ZB_MAX_TOPK, ZB_ERR_INVALID, "top_k %llu exceeds %d", (unsigned long long)top_k, ZB_MAX_TOPK);
    ZB_REQUIRE(probes <= ZB_MAX_PROBES, ZB_ERR_INVALID, "probes %u exceeds %d", probes, ZB_MAX_PROBES);
}
int zb_index_search_probe(zb_index* ix, uint64_t nq, const float* queries, uint64_t top_k, uint32_t probes, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_bits, uint32_t* out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (queries || !nq) && ((out_bits && out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    probe_check(top_k, probes);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_host(ix, nq, queries, top_k, probes, out_ids16, (u64*)out_ordinals, (u64*)out_bits, out_counts, false);
    ZB_API_END
}
int zb_index_search_probe_device(zb_index* ix, uint64_t nq, const float* d_q, uint64_t top_k, uint32_t probes, uint64_t* d_out_ord,
                                 uint64_t* d_out_bits, uint32_t* d_out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_q || !nq) && ((d_out_ord && d_out_bits && d_out_counts) || !nq), ZB_ERR_INVALID, "NULL argument");
    probe_check(top_k, probes);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_device(ix, nq, d_q, top_k, probes, (u64*)d_out_ord, (u64*)d_out_bits, d_out_counts, false);
    ZB_API_END
}
int zb_index_search_slice_probe(zb_index* ix, uint64_t nq_total, const float* queries, uint64_t top_k, uint32_t probes,
                                uint8_t* out_ids16, uint64_t* out_ordinals, uint64_t* out_bits, uint32_t* out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    probe_check(top_k, probes);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_host(ix, nq_total, queries, top_k, probes, out_ids16, (u64*)out_ordinals, (u64*)out_bits, out_counts, true);
    ZB_API_END
}
int zb_index_search_slice_probe_device(zb_index* ix, uint64_t nq_total, const float* d_q, uint64_t top_k, uint32_t probes,
                                       uint64_t* d_out_ord, uint64_t* d_out_bits, uint32_t* d_out_counts) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    probe_check(top_k, probes);
    std::lock_guard<std::mutex> lk(ix->mu);
    search_entry_device(ix, nq_total, d_q, top_k, probes, (u64*)d_out_ord, (u64*)d_out_bits, d_out_counts, true);
    ZB_API_END
}

// caller holds ix->mu
static void hash_device_impl(zb_index* ix, uint64_t n, const float* d_rows, uint64_t* d_keys, uint32_t* d_depths, int32_t* d_leaves) {
    ix->use_device();
    ZB_REQUIRE(ix->built, ZB_ERR_STATE, "hash on an index without trees");
    const float* x = d_rows;
    if (!(ix->dim == ix->dimp && ((uintptr_t)d_rows & 15) == 0)) {
        ix->r_stage.ensure(n * (u64)ix->dimp);
        launch_pad_rows(d_rows, n, ix->dim, ix->dimp, ix->r_stage.p, ix->stream);
        x = ix->r_stage.p;
    }
    const bool flat = ix->flat_bits && ix->p_flat_project && ix->h_nodes.size() == ix->flat_nodes &&
                      ix->n_planes == (u64)ix->T * ix->flat_bits;
    if (flat) {  // every row asks the same T x K planes: one dense pass, sign bits packed into the keys
        const int H = ix->T * (int)ix->flat_bits, Hp = (H + 15) / 16 * 16;
        ix->pj_sign.ensure(std::max<u64>(1, n * (u64)Hp));
        if (ix->p_flat_project == 1 && project3_supported(ix->dimp))   // knob flat_project: 1 = TMA-staged tile kernel, 2 = the first kernel (rows and planes through L1)
            project3(ix->pj_ws, x, n, ix->d_coef.p, ix->d_cst.p, H, ix->dimp, ix->pj_sign.p, Hp, ix->stream);
        else
            launch_project_flat(x, n, ix->d_coef.p, ix->d_cst.p, H, ix->dimp, ix->pj_sign.p, Hp, ix->stream);
        launch_pack_flat_keys(ix->pj_sign.p, n, Hp, ix->T, (int)ix->flat_bits, (u64*)d_keys, d_depths, d_leaves, ix->stream);
    } else {
        launch_hash(ix->view(), x, n, (u64*)d_keys, d_depths, d_leaves, (int)ix->p_hash_variant, ix->stream);
    }
    if (d_leaves) {
        if (!ix->export_table_valid) {
            std::vector<int> table;
            build_export_table(ix, nullptr, &table);
            ix->d_leaf_export.ensure(table.size() ? table.size() : 1);
            if (!table.empty())
                ZB_CUDA(cudaMemcpyAsync(ix->d_leaf_export.p, table.data(), table.size() * 4, cudaMemcpyHostToDevice, ix->stream));
            ix->sync();
            ix->export_table_valid = true;
        }
        u64 tot = n * (u64)ix->T;
        if (tot) remap_leaves_kernel<<<(u32)((tot + 255) / 256), 256, 0, ix->stream>>>(d_leaves, tot, ix->d_leaf_export.p);
    }
    ix->sync();
}

int zb_index_hash_device(zb_index* ix, uint64_t n, const float* d_rows, uint64_t* d_keys, uint32_t* d_depths, int32_t* d_leaves) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (d_rows || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    hash_device_impl(ix, n, d_rows, d_keys, d_depths, d_leaves);
    ZB_API_END
}

// The handle stays locked for the whole call: the staging and result buffers are the index's own.
int zb_index_hash(zb_index* ix, uint64_t n, const float* rows, uint64_t* out_keys, uint32_t* out_depths, int32_t* out_leaves) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (rows || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->use_device();
    ZB_REQUIRE(ix->built, ZB_ERR_STATE, "hash on an index without trees");
    ix->h_keys.ensure(n * (u64)ix->T + 1);
    ix->h_depths.ensure(n * (u64)ix->T + 1);
    ix->h_leaves.ensure(n * (u64)ix->T + 1);
    ix->hash_in.ensure(n * (u64)ix->dim + 4);
    // on the index's stream: a pageable cudaMemcpy on the legacy stream may return before its DMA has landed, and the
    // index's stream is non-blocking, so the hash kernel could otherwise read rows that are not there yet
    ZB_CUDA(cudaMemcpyAsync(ix->hash_in.p, rows, n * (u64)ix->dim * 4, cudaMemcpyHostToDevice, ix->stream));
    hash_device_impl(ix, n, ix->hash_in.p, (uint64_t*)ix->h_keys.p, ix->h_depths.p, ix->h_leaves.p);
    const u64 tot = n * (u64)ix->T;
    if (out_keys) ZB_CUDA(cudaMemcpyAsync(out_keys, ix->h_keys.p, tot * 8, cudaMemcpyDeviceToHost, ix->stream));
    if (out_depths) ZB_CUDA(cudaMemcpyAsync(out_depths, ix->h_depths.p, tot * 4, cudaMemcpyDeviceToHost, ix->stream));
    if (out_leaves) ZB_CUDA(cudaMemcpyAsync(out_leaves, ix->h_leaves.p, tot * 4, cudaMemcpyDeviceToHost, ix->stream));
    ix->sync();
    ZB_API_END
}

int zb_index_forest_sizes(zb_index* ix, int64_t* sizes4) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && sizes4, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    std::vector<int> order, leaf_export;
    build_export_table(ix, &order, &leaf_export);
    int64_t planes = 0, leaves = 0, members = 0;
    for (int n : order) {
        int4 nd = ix->h_nodes[n];
        if (nd.x >= 0) planes++;
        else {
            leaves++;
            members += ix->h_leaf_len[nd.w];
        }
    }
    sizes4[0] = (int64_t)order.size(); sizes4[1] = planes; sizes4[2] = leaves; sizes4[3] = members;
    ZB_API_END
}

int zb_index_export_forest(zb_index* ix, int32_t* nodes, int32_t* roots, float* coef, float* cst, int64_t* leaf_off,
                           uint64_t* members) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->use_device();
    if (!ix->built) return ZB_OK;
    ix->sync_host_members();
    std::vector<int> order, leaf_export;
    build_export_table(ix, &order, &leaf_export);
    std::vector<int> newid(ix->h_nodes.size(), -1);
    for (size_t i = 0; i < order.size(); ++i) newid[order[i]] = (int)i;
    int64_t np = 0, nl = 0, nm = 0;
    leaf_off[0] = 0;
    std::vector<int64_t> plane_pos(order.size(), -1);  // where inner node i's plane goes in the output
    for (size_t i = 0; i < order.size(); ++i) {
        int4 nd = ix->h_nodes[order[i]];
        if (nd.x >= 0) {
            ZB_REQUIRE((u64)nd.x < ix->n_planes, ZB_ERR_STATE, "plane %d out of range", nd.x);
            plane_pos[i] = np;
            nodes[4 * i + 0] = (int)np++; nodes[4 * i + 1] = newid[nd.y]; nodes[4 * i + 2] = newid[nd.z]; nodes[4 * i + 3] = -1;
        } else {
            const int l = nd.w;
            for (u32 j = 0; j < ix->h_leaf_len[l]; ++j) members[nm++] = ix->h_ord[ix->h_members[ix->h_leaf_off[l] + j]];
            leaf_off[++nl] = nm;
            nodes[4 * i + 0] = -1; nodes[4 * i + 1] = -1; nodes[4 * i + 2] = -1; nodes[4 * i + 3] = (int)(nl - 1);
        }
    }
    // planes: the device array comes over in chunks of <= 256 MB and every inner node picks its plane out of the chunk
    // (one copy per inner node cost ~10 us each: minutes for a default forest over 1M rows)
    const u64 chunk = std::max<u64>(1, (256ull << 20) / ((u64)ix->dim * 4));
    std::vector<float> h_coef, h_cst;
    for (u64 p0 = 0; p0 < ix->n_planes; p0 += chunk) {
        const u64 cnt = std::min<u64>(chunk, ix->n_planes - p0);
        h_coef.resize((size_t)cnt * ix->dim);
        h_cst.resize((size_t)cnt);
        ZB_CUDA(cudaMemcpy2D(h_coef.data(), (size_t)ix->dim * 4, ix->d_coef.p + p0 * (u64)ix->dimp, (size_t)ix->dimp * 4,
                             (size_t)ix->dim * 4, cnt, cudaMemcpyDeviceToHost));
        ZB_CUDA(cudaMemcpy(h_cst.data(), ix->d_cst.p + p0, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < order.size(); ++i) {
            if (plane_pos[i] < 0) continue;
            const u64 pl = (u64)ix->h_nodes[order[i]].x;
            if (pl < p0 || pl >= p0 + cnt) continue;
            memcpy(coef + plane_pos[i] * ix->dim, h_coef.data() + (size_t)(pl - p0) * ix->dim, (size_t)ix->dim * 4);
            cst[plane_pos[i]] = h_cst[(size_t)(pl - p0)];
        }
    }
    for (int t = 0; t < ix->T; ++t) roots[t] = newid[ix->h_roots[t]];
    ZB_API_END
}

static void clear_locked(zb_index* ix) {
    ix->use_device();
    ix->sync();
    ix->clear_forest();
    ix->n_slots = ix->n_live = ix->total_rows = 0;
    ++ix->store_gen;
    ix->h_ord.clear();
    ix->h_tomb.clear();
    ix->flat_bits = 0;
    ix->flat_nodes = 0;
    ix->ids_by_ordinal.clear();
    ix->ordinal_by_id.clear();
    ix->id_mode = 0;
}

// Everything is validated against the caller's arrays BEFORE the index is touched (a rejected forest leaves the index as
// it was), and the replace happens under one lock: node ranges, leaf_off monotone, every leaf referenced by exactly one
// node reachable from a root, depth <= ZB_MAX_DEPTH, no cycle, every row exactly once in every tree, ids distinct.
int zb_index_load_forest(zb_index* ix, uint64_t n, const float* rows, const uint8_t* ids16, const int64_t* sizes4,
                         const int32_t* nodes, const int32_t* roots, const float* coef, const float* cst,
                         const int64_t* leaf_off, const uint64_t* members) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && sizes4 && nodes && roots && leaf_off && (rows || !n), ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->use_device();
    if (ix->G > 1) ZB_REQUIRE(ix->comm_ready, ZB_ERR_STATE, "sharded index used before zb_index_comm_init");
    const int64_t nn = sizes4[0], npl = sizes4[1], nl = sizes4[2], nm = sizes4[3];
    ZB_REQUIRE(nn >= ix->T && npl >= 0 && nl >= 1 && nm >= 0, ZB_ERR_INVALID, "bad forest sizes");
    ZB_REQUIRE((members && coef && cst) || (!nm && !npl), ZB_ERR_INVALID, "NULL argument");
    const int T = ix->T;
    // ---- validation pass (no index state is modified) ----
    std::vector<int4> v_nodes((size_t)nn);
    for (int64_t i = 0; i < nn; ++i) {
        const int32_t* nd = nodes + 4 * i;
        if (nd[0] >= 0) {
            ZB_REQUIRE(nd[0] < npl && nd[1] >= 0 && nd[1] < nn && nd[2] >= 0 && nd[2] < nn, ZB_ERR_INVALID, "node %lld malformed", (long long)i);
        } else {
            ZB_REQUIRE(nd[3] >= 0 && nd[3] < nl, ZB_ERR_INVALID, "leaf node %lld malformed", (long long)i);
        }
        v_nodes[i] = make_int4(nd[0], nd[1], nd[2], nd[3]);
    }
    ZB_REQUIRE(leaf_off[0] == 0, ZB_ERR_INVALID, "leaf_off must start at 0");
    for (int64_t l = 0; l < nl; ++l)
        ZB_REQUIRE(leaf_off[l] <= leaf_off[l + 1] && leaf_off[l + 1] <= nm, ZB_ERR_INVALID, "leaf_off not monotone");
    for (int64_t j = 0; j < leaf_off[nl]; ++j) ZB_REQUIRE(members[j] < n, ZB_ERR_INVALID, "member ordinal out of range");
    std::vector<u64> v_key((size_t)nl, 0);
    std::vector<int> v_depth((size_t)nl, 0), v_node((size_t)nl, -1), v_tree((size_t)nl, 0);
    {
        struct Fr { int node; u64 key; int depth; };
        std::vector<Fr> stack;
        std::vector<u8> in_tree((size_t)n);
        size_t visited = 0;
        for (int t = 0; t < T; ++t) {
            ZB_REQUIRE(roots[t] >= 0 && roots[t] < nn, ZB_ERR_INVALID, "root %d out of range", t);
            std::fill(in_tree.begin(), in_tree.end(), 0);
            u64 rows_in_tree = 0;
            stack.push_back(Fr{roots[t], root_key(ix->opt.seed, t), 0});
            while (!stack.empty()) {
                Fr fr = stack.back();
                stack.pop_back();
                ZB_REQUIRE(++visited <= (size_t)nn, ZB_ERR_INVALID, "forest has a cycle or shares nodes between trees");
                ZB_REQUIRE(fr.depth <= ZB_MAX_DEPTH, ZB_ERR_INVALID, "tree %d deeper than %d levels", t, ZB_MAX_DEPTH);
                const int4 nd = v_nodes[fr.node];
                if (nd.x >= 0) {
                    stack.push_back(Fr{nd.z, child_key(fr.key, 1), fr.depth + 1});
                    stack.push_back(Fr{nd.y, child_key(fr.key, 0), fr.depth + 1});
                } else {
                    ZB_REQUIRE(v_node[nd.w] < 0, ZB_ERR_INVALID, "leaf %d referenced twice", nd.w);
                    v_node[nd.w] = fr.node;
                    v_key[nd.w] = fr.key;
                    v_depth[nd.w] = fr.depth;
                    v_tree[nd.w] = t;
                    for (int64_t j = leaf_off[nd.w]; j < leaf_off[nd.w + 1]; ++j) {
                        ZB_REQUIRE(!in_tree[members[j]], ZB_ERR_INVALID, "row %llu is in two leaves of tree %d",
                                   (unsigned long long)members[j], t);
                        in_tree[members[j]] = 1;
                        ++rows_in_tree;
                    }
                }
            }
            ZB_REQUIRE(rows_in_tree == n, ZB_ERR_INVALID, "tree %d holds %llu of the %llu rows", t,
                       (unsigned long long)rows_in_tree, (unsigned long long)n);
        }
        for (int64_t l = 0; l < nl; ++l)
            ZB_REQUIRE(v_node[l] >= 0, ZB_ERR_INVALID, "leaf %lld is not reachable from any root", (long long)l);
    }
    std::vector<Id16> v_ids;
    std::unordered_map<Id16, u64, Id16Hash> v_map;
    if (ids16) {
        v_ids.resize((size_t)n);
        v_map.reserve((size_t)n);
        for (u64 i = 0; i < n; ++i) {
            v_ids[i] = Id16{load_be64(ids16 + 16 * i), load_be64(ids16 + 16 * i + 8)};
            ZB_REQUIRE(v_map.emplace(v_ids[i], i).second, ZB_ERR_INVALID, "duplicate id at row %llu", (unsigned long long)i);
        }
    }
    // ---- commit ----
    clear_locked(ix);
    ix->id_mode = n ? (ids16 ? 2 : 1) : 0;
    ix->ids_by_ordinal.swap(v_ids);
    ix->ordinal_by_id.swap(v_map);
    std::vector<u64> ordinals;
    for (u64 i = ix->rank; i < n; i += ix->G) ordinals.push_back(i);
    if (!ordinals.empty()) {
        ix->r_stage.ensure(ordinals.size() * (u64)ix->dim);
        ZB_CUDA(cudaMemcpy2DAsync(ix->r_stage.p, (size_t)ix->dim * 4, rows + (u64)ix->rank * ix->dim, (size_t)ix->dim * ix->G * 4,
                                  (size_t)ix->dim * 4, ordinals.size(), cudaMemcpyHostToDevice, ix->stream));
        ix->append_rows_device(ix->r_stage.p, ix->dim, ordinals.size(), ordinals.data());
    }
    ix->total_rows = n;
    ix->h_nodes.swap(v_nodes);
    ix->h_leaf_off.assign(nl, 0); ix->h_leaf_len.assign(nl, 0); ix->h_leaf_cap.assign(nl, 0);
    ix->h_leaf_key.swap(v_key); ix->h_leaf_depth.swap(v_depth); ix->h_leaf_node.swap(v_node); ix->h_leaf_tree.swap(v_tree);
    // local member lists (owned rows only), leaf-major
    ix->h_members.clear();
    std::vector<u32> slot_leaf_h((size_t)T * std::max<u64>(ix->n_slots, 1), 0);
    for (int64_t l = 0; l < nl; ++l) {
        ix->h_leaf_off[l] = (long long)ix->h_members.size();
        for (int64_t j = leaf_off[l]; j < leaf_off[l + 1]; ++j)
            if (ix->owns(members[j])) ix->h_members.push_back((u32)ix->slot_of(members[j]));
        ix->h_leaf_len[l] = ix->h_leaf_cap[l] = (u32)(ix->h_members.size() - ix->h_leaf_off[l]);
        // invariant of the bucket-major store: inside a leaf, position order == ordinal order (ties by id, D3)
        std::sort(ix->h_members.begin() + ix->h_leaf_off[l], ix->h_members.end());
        const size_t t = (size_t)ix->h_leaf_tree[l];
        for (u32 j = 0; j < ix->h_leaf_len[l]; ++j) slot_leaf_h[t * ix->n_slots + ix->h_members[ix->h_leaf_off[l] + j]] = (u32)l;
    }
    for (int t = 0; t < T; ++t) ix->h_roots[t] = roots[t];
    ix->n_planes = (u64)npl;
    ix->d_coef.ensure(std::max<u64>(1, (u64)npl * ix->dimp));
    ix->d_cst.ensure(std::max<u64>(1, (u64)npl));
    if (npl) {
        ZB_CUDA(cudaMemsetAsync(ix->d_coef.p, 0, (u64)npl * ix->dimp * 4, ix->stream));
        ZB_CUDA(cudaMemcpy2DAsync(ix->d_coef.p, (size_t)ix->dimp * 4, coef, (size_t)ix->dim * 4, (size_t)ix->dim * 4, npl,
                                  cudaMemcpyHostToDevice, ix->stream));
        ZB_CUDA(cudaMemcpyAsync(ix->d_cst.p, cst, (u64)npl * 4, cudaMemcpyHostToDevice, ix->stream));
    }
    ix->members_used = ix->h_members.size();
    ix->h_members_valid = true;
    ix->d_members.ensure(std::max<u64>(1, ix->members_used));
    if (ix->members_used)
        ZB_CUDA(cudaMemcpyAsync(ix->d_members.p, ix->h_members.data(), ix->members_used * 4, cudaMemcpyHostToDevice, ix->stream));
    if (ix->n_slots)
        ZB_CUDA(cudaMemcpy2DAsync(ix->slot_leaf.p, ix->slot_stride * 4, slot_leaf_h.data(), ix->n_slots * 4, ix->n_slots * 4, T,
                                  cudaMemcpyHostToDevice, ix->stream));
    ix->sync();
    ix->built = true;
    ix->upload_structure();
    ix->recount_live();
    ix->sync();
    ZB_API_END
}

static void pad_to_device(int device, const float* h, u64 n, u32 dim, int dimp, DBuf<float>& d);

// Flat tables.  coef = T * bits planes of dim f32 (table t, bit d at index t * bits + d), cst = their constants.
int zb_index_load_flat(zb_index* ix, uint64_t n, const float* rows, const uint8_t* ids16, uint32_t bits, const float* coef,
                       const float* cst) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && (rows || !n) && coef && cst, ZB_ERR_INVALID, "NULL argument");
    ZB_REQUIRE(bits >= 1 && bits <= 16, ZB_ERR_INVALID, "bits %u out of range 1..16", bits);
    ZB_REQUIRE(n < (1ull << 32), ZB_ERR_INVALID, "too many rows for one load");
    int T, dim, dimp;
    {
        std::lock_guard<std::mutex> lk(ix->mu);
        ix->use_device();
        T = ix->T; dim = ix->dim; dimp = ix->dimp;
    }
    const int K = (int)bits, H = T * K, Hp = (H + 15) / 16 * 16;
    // ---- bucket keys of every row: the dense projection (legacy stream: ordered after the staging copies) ----
    std::vector<u64> keys((size_t)n * T + 1);
    {
        DBuf<float> d_rows, d_coef, d_cst;
        DBuf<u8> d_sign;
        DBuf<u64> d_keys;
        pad_to_device(ix->device, rows, n, (u32)dim, dimp, d_rows);
        pad_to_device(ix->device, coef, (u64)H, (u32)dim, dimp, d_coef);
        d_cst.ensure((size_t)H);
        ZB_CUDA(cudaMemcpy(d_cst.p, cst, (size_t)H * 4, cudaMemcpyHostToDevice));
        d_sign.ensure(std::max<u64>(1, n * (u64)Hp));
        d_keys.ensure((size_t)n * T + 1);
        launch_project_flat(d_rows.p, n, d_coef.p, d_cst.p, H, dimp, d_sign.p, Hp, 0);
        launch_pack_flat_keys(d_sign.p, n, Hp, T, K, d_keys.p, nullptr, nullptr, 0);
        ZB_CUDA(cudaGetLastError());
        if (n) ZB_CUDA(cudaMemcpy(keys.data(), d_keys.p, (size_t)n * T * 8, cudaMemcpyDeviceToHost));
    }
    // ---- the equivalent forest: T complete trees of depth K in preorder (node, left = below = bit 0, right = above) ----
    const int64_t per_tree = ((int64_t)2 << K) - 1, leaves_per_tree = (int64_t)1 << K;
    int64_t sizes4[4] = {per_tree * T, (int64_t)H, leaves_per_tree * T, (int64_t)n * T};
    std::vector<int32_t> nodes((size_t)sizes4[0] * 4), roots((size_t)T);
    for (int t = 0; t < T; ++t) {
        int32_t idx = (int32_t)(per_tree * t);
        roots[t] = idx;
        struct Fr { int depth; u32 prefix; int32_t parent; int side; };
        std::vector<Fr> stack{{0, 0u, -1, 0}};
        while (!stack.empty()) {
            const Fr fr = stack.back();
            stack.pop_back();
            const int32_t me = idx++;
            if (fr.parent >= 0) nodes[4 * (size_t)fr.parent + 1 + fr.side] = me;
            int32_t* nd = nodes.data() + 4 * (size_t)me;
            if (fr.depth == K) {
                nd[0] = -1; nd[1] = -1; nd[2] = -1; nd[3] = (int32_t)(leaves_per_tree * t + fr.prefix);
            } else {
                nd[0] = t * K + fr.depth; nd[1] = -1; nd[2] = -1; nd[3] = -1;
                stack.push_back({fr.depth + 1, (fr.prefix << 1) | 1u, me, 1});  // right subtree after ...
                stack.push_back({fr.depth + 1, fr.prefix << 1, me, 0});         // ... the left one (preorder)
            }
        }
    }
    std::vector<int64_t> leaf_off((size_t)sizes4[2] + 1, 0);
    for (u64 o = 0; o < n; ++o)
        for (int t = 0; t < T; ++t) leaf_off[(size_t)(leaves_per_tree * t + (int64_t)keys[o * T + t]) + 1]++;
    for (size_t l = 0; l < (size_t)sizes4[2]; ++l) leaf_off[l + 1] += leaf_off[l];
    std::vector<int64_t> cursor(leaf_off.begin(), leaf_off.end() - 1);
    std::vector<uint64_t> members((size_t)n * T + 1);
    for (u64 o = 0; o < n; ++o)  // ascending ordinal inside a leaf
        for (int t = 0; t < T; ++t) members[(size_t)cursor[(size_t)(leaves_per_tree * t + (int64_t)keys[o * T + t])]++] = o;
    int rc = zb_index_load_forest(ix, n, rows, ids16, sizes4, nodes.data(), roots.data(), coef, cst, leaf_off.data(), members.data());
    if (rc != ZB_OK) return rc;
    {
        std::lock_guard<std::mutex> lk(ix->mu);
        ix->flat_bits = bits;
        ix->flat_nodes = ix->h_nodes.size();
    }
    ZB_API_END
}

int zb_index_options(zb_index* ix, zb_options* out) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    *out = ix->opt;
    ZB_API_END
}

int zb_index_export_rows(zb_index* ix, uint64_t first_ordinal, uint64_t n, float* out_rows, uint8_t* out_ids16,
                         uint8_t* out_live) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->use_device();
    ZB_REQUIRE(ix->G <= 1, ZB_ERR_STATE, "zb_index_export_rows needs an unsharded index (a shard holds 1/G of the rows)");
    ZB_REQUIRE(first_ordinal <= ix->total_rows && n <= ix->total_rows - first_ordinal, ZB_ERR_INVALID,
               "rows [%llu, +%llu) out of range (%llu rows)", (unsigned long long)first_ordinal, (unsigned long long)n,
               (unsigned long long)ix->total_rows);
    if (out_rows && n) {  // unsharded: slot == ordinal
        ZB_CUDA(cudaMemcpy2DAsync(out_rows, (size_t)ix->dim * 4, ix->rows.p + first_ordinal * (u64)ix->dimp, (size_t)ix->dimp * 4,
                                  (size_t)ix->dim * 4, n, cudaMemcpyDeviceToHost, ix->stream));
        ix->sync();
    }
    for (u64 i = 0; i < n; ++i) {
        if (out_ids16) ix->id_of(first_ordinal + i, out_ids16 + 16 * i);
        if (out_live) out_live[i] = ix->h_tomb[first_ordinal + i] ? 0 : 1;
    }
    ZB_API_END
}

int zb_index_stats(zb_index* ix, zb_stats* out) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->st.rows = ix->n_slots;
    ix->st.live_rows = ix->n_live;
    ix->st.total_rows = ix->total_rows;
    ix->st.nodes = ix->h_nodes.size();
    ix->st.planes = ix->n_planes;
    ix->st.leaves = ix->h_leaf_off.size();
    ix->st.device_bytes = zb::g_device_bytes;
    *out = ix->st;
    ZB_API_END
}

int zb_index_stream(zb_index* ix, void** out_stream) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && out_stream, ZB_ERR_INVALID, "NULL argument");
    *out_stream = (void*)ix->stream;
    ZB_API_END
}

int zb_index_set_param(zb_index* ix, const char* key, int64_t value) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && key, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    std::string k(key);
    if (k == "tile_min_rows") ix->p_tile_min_rows = value;
    else if (k == "tile_queries") ix->p_tile_queries = value;
    else if (k == "use_tile_scan") ix->p_use_tile_scan = value;
    else if (k == "scan_gen") ix->p_scan_gen = value;  // fused leaf-tile scan: 3 = third generation (default), 2 = second (8-query tiles, 128-row stages)
    else if (k == "classify_variant") ix->p_classify_variant = value;  // 0: rows gathered through L1; 1: rows staged by TMA bulk copies
    else if (k == "seq_prefetch") ix->p_seq_prefetch = value;  // scalar metrics: L2 prefetch distance of the row stream in 128-byte lines (0 = off, the default: measured slower)
    else if (k == "select_variant") ix->p_select_variant = value;  // per-visit top-n' of the gather path: 0 = block bitonic, 1 = one warp per visit, list in registers (default: 4.9 -> 0.38 ms on 2047-row visits, profiles/r02a_bench_manhattan_select*.json)
    else if (k == "quad_tile") ix->p_quad_tile = value;  // cosine / L2 visits outside the fused kernel (n' > 32): 1 = keys-only leaf-tile scan (default: 2.4x the gather path on top-100, profiles/r02a_bench_top100_quad*.json), 0 = one quad per pair
    else if (k == "flat_project") ix->p_flat_project = value;  // flat tables: 1 = dense projection + ballot packing (default), 0 = the generic tree walk
    else if (k == "l2_filter") { ix->p_l2_filter = value; ix->filter_backoff = 0; }  // L2 / L2 squared through the dot-product filter + exact second pass: 0 off, 1 adaptive (default), 2 always
    else if (k == "long_list_warps") { ZB_REQUIRE(value == 4 || value == 8, ZB_ERR_INVALID, "long_list_warps is 4 or 8"); ix->scan_ws.long_list_warps = (int)value; }  // fused scan with n' > 32: math warps per team
    else if (k == "exact_budget_mb") {  // exact search: workspace of one query chunk, MiB (default 256)
        ZB_REQUIRE(value >= 1 && value <= (1 << 20), ZB_ERR_INVALID, "exact_budget_mb out of range");
        ix->p_exact_budget_mb = value;
    }
    else if (k == "plan_tail") ix->p_plan_tail = value;  // plan walk: 1 = cascade walkers go to the latency-optimised tail kernel (default), 0 = one kernel
    else if (k == "p2p_queries") ix->p_p2p_queries = value;  // sliced search: 1 = query slices pushed into the peers' buffers over NVLink (CUDA IPC; default), 0 = NCCL
    else if (k == "single_exchange") ix->p_single_exchange = value;  // sliced search: 1 = query slices ride in the visit-record allgather (default), 0 = their own allgather first
    else if (k == "bm_stage_mb") ix->p_bm_stage_mb = value > 0 ? value : 1;  // bucket-sharded store build: staging area per direction, MiB (default 2048)
    else if (k == "seq_tile") ix->p_seq_tile = value;          // scalar metrics: 1 = leaf-tile scan (default), 0 = one thread per pair
    else if (k == "hash_variant") ix->p_hash_variant = value;  // 0: quad per (row, tree), rows through L1; 1: row staged in shared memory
    else if (k == "visit_slots") {  // initial per-walker capacity of the visit plan (tests force the grow-and-replan path)
        ZB_REQUIRE(value >= 2 && value <= 65536, ZB_ERR_INVALID, "visit_slots out of range");
        ix->vpw = (u32)value;
    }
    else throw zb::Error(ZB_ERR_INVALID, "unknown parameter " + k);
    ZB_API_END
}

int zb_comm_unique_id(uint8_t* out_id128) {
    ZB_API_BEGIN
    ZB_REQUIRE(out_id128, ZB_ERR_INVALID, "NULL argument");
    Nccl::unique_id(out_id128);
    ZB_API_END
}

int zb_index_comm_init(zb_index* ix, const uint8_t* id128) {
    ZB_API_BEGIN
    ZB_REQUIRE(ix && id128, ZB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    ZB_REQUIRE(ix->G > 1, ZB_ERR_STATE, "index is not sharded");
    ZB_REQUIRE(!ix->comm_ready, ZB_ERR_STATE, "communicator already initialised");
    ix->nccl.init(id128, (int)ix->rank, (int)ix->G, ix->device);
    ix->comm_ready = true;
    // agree on the id epoch (minted ids must be identical on every rank)
    ix->b_minh.ensure(1);
    ZB_CUDA(cudaMemcpyAsync(ix->b_minh.p, &ix->epoch_ms, 8, cudaMemcpyHostToDevice, ix->stream));
    ix->nccl.allreduce(ix->b_minh.p, 1, Nccl::U64, Nccl::MIN, ix->stream);
    ZB_CUDA(cudaMemcpyAsync(&ix->epoch_ms, ix->b_minh.p, 8, cudaMemcpyDeviceToHost, ix->stream));
    ix->sync();
    ZB_API_END
}

static void pad_to_device(int device, const float* h, u64 n, u32 dim, int dimp, DBuf<float>& d) {
    d.ensure(std::max<u64>(1, n * (u64)dimp));
    if (!n) return;
    ZB_CUDA(cudaMemset(d.p, 0, n * (u64)dimp * 4));
    ZB_CUDA(cudaMemcpy2D(d.p, (size_t)dimp * 4, h, (size_t)dim * 4, (size_t)dim * 4, n, cudaMemcpyHostToDevice));
}

int zb_metric_distance_batch(int device, uint32_t metric, int32_t power, uint64_t n, uint32_t dim, const float* a, const float* b,
                             uint64_t* out_bits) {
    ZB_API_BEGIN
    ZB_REQUIRE(metric < ZB_METRIC_COUNT && dim >= 1 && ((a && b && out_bits) || !n), ZB_ERR_INVALID, "bad argument");
    ZB_REQUIRE((metric != ZB_METRIC_MINKOWSKI && metric != ZB_METRIC_PNORM) || (power >= 0 && power <= ZB_METRIC_MAX_POWER),
               ZB_ERR_INVALID, "power %d out of range 0..%d", power, ZB_METRIC_MAX_POWER);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || !ndev) {
        cudaGetLastError();
        throw zb::Error(ZB_ERR_NO_DEVICE, "no CUDA device: libzebra_b200 has no CPU fallback");
    }
    ZB_CUDA(cudaSetDevice(device));
    const int dimp = ((int)dim + 15) / 16 * 16;
    DBuf<float> da, db;
    DBuf<u64> dout;
    pad_to_device(device, a, n, dim, dimp, da);
    pad_to_device(device, b, n, dim, dimp, db);
    dout.ensure(std::max<u64>(1, n));
    launch_pair_metric((int)metric, (int)power, da.p, db.p, n, (int)dim, dimp, dout.p, 0);
    ZB_CUDA(cudaMemcpy(out_bits, dout.p, n * 8, cudaMemcpyDeviceToHost));
    ZB_API_END
}

int zb_point_is_above_batch(int device, uint64_t n, uint32_t dim, const float* coef, const float* cst, const float* x,
                            uint8_t* out) {
    ZB_API_BEGIN
    ZB_REQUIRE(dim >= 1 && ((coef && cst && x && out) || !n), ZB_ERR_INVALID, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || !ndev) {
        cudaGetLastError();
        throw zb::Error(ZB_ERR_NO_DEVICE, "no CUDA device: libzebra_b200 has no CPU fallback");
    }
    ZB_CUDA(cudaSetDevice(device));
    const int dimp = ((int)dim + 15) / 16 * 16;
    DBuf<float> dc, dx, dk;
    DBuf<u8> dout;
    pad_to_device(device, coef, n, dim, dimp, dc);
    pad_to_device(device, x, n, dim, dimp, dx);
    dk.ensure(std::max<u64>(1, n));
    dout.ensure(std::max<u64>(1, n));
    if (n) ZB_CUDA(cudaMemcpy(dk.p, cst, n * 4, cudaMemcpyHostToDevice));
    launch_pair_above(dc.p, dk.p, dx.p, n, dimp, dout.p, 0);
    if (n) ZB_CUDA(cudaMemcpy(out, dout.p, n, cudaMemcpyDeviceToHost));
    ZB_API_END
}

int zb_synth_fill_device(int device, float* d_out, uint64_t first_row, uint64_t row_stride, uint64_t n, uint32_t dim,
                         uint64_t seed, uint32_t kind) {
    ZB_API_BEGIN
    ZB_REQUIRE(d_out || !n, ZB_ERR_INVALID, "NULL argument");
    ZB_CUDA(cudaSetDevice(device));
    launch_synth(d_out, first_row, row_stride, n, dim, seed, kind, 0);
    ZB_CUDA(cudaStreamSynchronize(0));
    ZB_API_END
}

}  // extern "C"
