// zb_scan.cu -- the fused leaf-tile scan: bucket-major row tiles + distance scoring + per-visit top-n' in one kernel.
//
// Replaces, for visits of large leaves, the leaf branch of tree_result
// (/root/reference/src/database/index/lsh.rs:299-331: fetch every member, metric.distance, sort, take n) and
// the rescoring of search (:557-563).  Work unit ("tile") = (leaf, <= 16 queries that visit it).
//
//   * The rows of a leaf are CONTIGUOUS in the bucket-major store (zb_index.cu: bm_rows[position][dimp], position =
//     index into the forest's member array), so a K slice of a 128-row block is one 2-D TMA box
//     (cp.async.bulk.tensor.2d, SASS UTMALDG): one instruction per 24 KB stage, issued by a dedicated producer warp
//     that runs up to TS ring stages ahead of the math warps -- across row blocks AND across tiles.
//   * 8 consumer warps score stage rows x tile queries with 8x4 register tiles per quad in the canonical
//     skylake-16 accumulation order (zb_device.cuh); the tile's queries stay resident in shared memory.
//   * Top-n' is warp-private and register resident: lane l of a warp holds the l-th best (key, position) of a
//     (query, row half); a finished distance is first filtered against the list's n'-th key, survivors are inserted
//     with a ballot + shuffle-up.  No block-wide barrier anywhere in the steady state.  The two row halves of a
//     query are merged once per tile with a shuffle bitonic network, tombstoned rows are masked at insertion.
// The kernel is persistent (one CTA per SM, tiles handed out by an atomic counter).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda.h>

#include "zb_scan.cuh"

namespace zb {

#define TS_TEAMS 2          // independent teams per CTA: each streams its own tiles through its own ring
#define TS_TWARPS 4         // math warps per team (one per SM sub-partition)
#define TS_QT 8             // queries per tile (2 query groups of 4)
#define TS_RB 128           // rows per row block (16 row groups of 8, interleaved: row = i * 16 + group)
#define TS_KC 3             // 16-float chunks per K slice: 192 B row pitch puts adjacent rows in different bank halves
#define TS_SLICE_FLOATS (TS_KC * 16)
#define TS_STAGE_BYTES (TS_RB * TS_SLICE_FLOATS * 4)   // 24576
#define TS_CWARPS (TS_TEAMS * TS_TWARPS)   // consumer (math) warps
#define TS_THREADS 384      // 2 math warpgroups (= teams) + 1 producer warpgroup (one TMA-driving warp per team; its registers go to the math warps)
#define TS_MAX_STAGES 8
#define TS_KL 32            // list length of the register top-n' (one entry per lane)
#define TS_NOPOS 0xFFFFFFFFu
#define TS_PACE_WINDOW 8    // a tile may run at most this many stages ahead of a sibling tile (same leaf, other queries)
#define TS_PACE_EVERY 4

// Phase timing of the math warps (debug builds only: make EXTRA=-DZB_SCAN_TIMING): cycles spent waiting for the
// tile info / queries, waiting for row stages, in the FP32 loop, in the fold + key epilogue, in list insertion and in
// the end-of-tile merge, summed over the ACTIVE math warps (slot 7 counts idle-warp time), written to stats[8..].
#ifdef ZB_SCAN_TIMING
#define TS_T(var) const long long var = clock64()
#define TS_ACC(slot, t0, t1) tacc[slot] += (t1) - (t0)
#else
#define TS_T(var)
#define TS_ACC(slot, t0, t1)
#endif

struct TileInfo {
    u32 tile, leaf, first, nqt, L, pad;
    long long moff;
};

struct TileParams {
    const u32* tile_leaf;
    const u32* tile_first;
    const u32* tile_count;
    const u32* ntiles;   // device scalar
    u32* tile_counter;   // device scalar, zeroed before launch
    const u32* order;    // visits grouped by leaf
    const u32* v_np;
    const u32* v_q;
    const u32* v_ent_off;
    Entry* entries;
    const float* queries;
    const double* q_rinv;   // [nq] 1/sqrt(|q|^2) in f64 (cosine)
    const double* bm_rinv;  // [positions] 1/sqrt(|row|^2) in f64 (cosine)
    const u32* bm_tomb;     // bit per position
    u64* stats;             // [0] visits, [1] pairs, [2] moved bytes
    u32 pace_window;        // 0 = no pacing
    u32* tile_prog;         // [ntiles] stages issued so far per tile (0xFFFFFFFF = finished): sibling tiles of a leaf pace each other
    u64* gthr;              // [nq] per-query bound shared by all of the query's visits: min over full lists of their n'-th key
    u32 top_k;
    int nst;                // ring depth
};

// ---- PTX helpers (mbarrier, 1-D bulk copy: zb_device.cuh); 2-D tensor copy (TMA) ----
__device__ __forceinline__ void tma_2d_g2s(u32 dst, const CUtensorMap* map, int c0, int c1, u32 bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void pair_sync(int g) { asm volatile("bar.sync %0, 64;" ::"r"(g + 1) : "memory"); }

__device__ __forceinline__ u64 shfl64(u64 v, int src) {
    u32 lo = __shfl_sync(0xffffffffu, (u32)v, src), hi = __shfl_sync(0xffffffffu, (u32)(v >> 32), src);
    return ((u64)hi << 32) | lo;
}
__device__ __forceinline__ u64 shfl_up64(u64 v) {
    u32 lo = __shfl_up_sync(0xffffffffu, (u32)v, 1), hi = __shfl_up_sync(0xffffffffu, (u32)(v >> 32), 1);
    return ((u64)hi << 32) | lo;
}
__device__ __forceinline__ u64 shfl_xor64(u64 v, int m) {
    u32 lo = __shfl_xor_sync(0xffffffffu, (u32)v, m), hi = __shfl_xor_sync(0xffffffffu, (u32)(v >> 32), m);
    return ((u64)hi << 32) | lo;
}
// (key, position) order: the position order inside a leaf equals the ordinal order (zb_index.cu keeps member lists
// ascending), so ties in distance are broken exactly like Entry order (D3).
__device__ __forceinline__ bool kp_less(u64 ka, u32 pa, u64 kb, u32 pb) { return ka < kb || (ka == kb && pa < pb); }

// Packed FP32 (sm_100 FFMA2 / FADD2): two IEEE-rounded f32 operations per instruction, bit-identical to the scalar
// __fmaf_rn / __fsub_rn forms of zb_device.cuh but half the issue slots, which is what lets one math warp per SM
// sub-partition keep the FMA pipe busy.
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void fma4_x2(float4& acc, const float4& a, const float4& b) {
    u64 c0 = pk2(acc.x, acc.y), c1 = pk2(acc.z, acc.w);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c0) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c1) : "l"(pk2(a.z, a.w)), "l"(pk2(b.z, b.w)));
    upk2(c0, acc.x, acc.y);
    upk2(c1, acc.z, acc.w);
}
__device__ __forceinline__ void l2acc4_x2(float4& acc, const float4& a, const float4& b) {
    u64 c0 = pk2(acc.x, acc.y), c1 = pk2(acc.z, acc.w), d0, d1;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d0) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)));
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d1) : "l"(pk2(a.z, a.w)), "l"(pk2(b.z, b.w)));
    asm("fma.rn.f32x2 %0, %1, %1, %0;" : "+l"(c0) : "l"(d0));
    asm("fma.rn.f32x2 %0, %1, %1, %0;" : "+l"(c1) : "l"(d1));
    upk2(c0, acc.x, acc.y);
    upk2(c1, acc.z, acc.w);
}
__device__ __forceinline__ float4 add4_xor(const float4& a, const float4& b, int m) {  // a + shfl_xor(b, m), componentwise
    return make_float4(__fadd_rn(a.x, __shfl_xor_sync(0xffffffffu, b.x, m)), __fadd_rn(a.y, __shfl_xor_sync(0xffffffffu, b.y, m)),
                       __fadd_rn(a.z, __shfl_xor_sync(0xffffffffu, b.z, m)), __fadd_rn(a.w, __shfl_xor_sync(0xffffffffu, b.w, m)));
}
__device__ __forceinline__ u64 sel8(const u64 (&k)[8], int i) {
    u64 r = k[0];
#pragma unroll
    for (int t = 1; t < 8; ++t) r = i == t ? k[t] : r;
    return r;
}

// Cosine epilogue from precomputed reciprocal norms: the operation order of cos_bits (zb_device.cuh) with
// ra = 1/sqrt(a2), rb = 1/sqrt(b2) hoisted (ra is +inf exactly when a2 == 0).
__device__ __forceinline__ u64 cos_bits_rinv(float ab_, double ra, double rb) {
    const double ab = (double)ab_;
    double c;
    if (isinf(ra) && isinf(rb) && ra > 0.0 && rb > 0.0) c = 0.0;
    else if (ab == 0.0) c = 1.0;
    else {
        double t = __dmul_rn(__dmul_rn(ab, ra), rb);
        double r = __dsub_rn(1.0, t);
        c = r > 0.0 ? r : 0.0;
    }
    return (u64)__double_as_longlong(__dsub_rn(1.0, c));
}

struct __align__(16) ListEntry {
    u64 key;
    u32 pos;
    u32 pad;
};

// Shared-memory view and barrier addresses of one CTA.
struct ScanCtx {
    unsigned char* s_stage;
    float* s_q;
    ListEntry* s_list;
    u32 bar_full, bar_empty;
    u32 S;
    int dimp, chunks, nsl;
};

// One math warp's share of one tile.  A quad owns NR rows x 4 queries (NR = 8: "wide" warp, 64 of the stage's 128
// rows; NR = 4: "narrow" warp, 32 rows); thread `sub` keeps lanes 4*sub..4*sub+3 of every pair's 16-lane accumulator.
// Per 16-float chunk a wide thread issues 4 + 8 LDS.128 and 128 packed FP32 instructions (L2; 64 for cosine).
// 128 accumulator registers per thread are why there are exactly 8 math warps (2 per SM sub-partition).
//   g  : query group (queries g*4 .. g*4+3 of the tile)        wr : which row slab of the group this warp scans
template <int METRIC, int NR>
__device__ __forceinline__ void scan_tile(const ScanCtx& cx, const ForestView& f, const TileParams& tp, const TileInfo& inf,
                                          const int g, const int wr, const int warp, const int lane, u32& buf, u32& ph,
                                          u32 my_np, u32 my_q, double my_qrinv, int nq_mine
#ifdef ZB_SCAN_TIMING
                                          , long long* tacc
#endif
) {
    constexpr int RSTRIDE = TS_RB / NR;              // rows between a quad's consecutive rows (16 wide, 32 narrow)
    const int qd = lane >> 2, sub = lane & 3;
    const int r0 = wr * 8 + qd;                      // rows i * RSTRIDE + r0, i = 0..NR-1
    const int dimp = cx.dimp, chunks = cx.chunks, nsl = cx.nsl;
    const u32 S = cx.S, L = inf.L;
    const u32 nblocks = (L + TS_RB - 1) / TS_RB;
    ListEntry* my_list = cx.s_list + (size_t)warp * 4 * TS_KL;
    const int qstep = dimp / 4;
    // Accumulator k of a thread belongs to query (k ^ sub) of the group: the quad's cross-thread folds then pair
    // registers with static indices (no selects), and thread `sub` ends up owning query `sub`.
    const float4* qb = reinterpret_cast<const float4*>(cx.s_q + (size_t)(g * 4) * dimp) + sub;
    const float4* qp0 = qb + (0 ^ sub) * qstep;
    const float4* qp1 = qb + (1 ^ sub) * qstep;
    const float4* qp2 = qb + (2 ^ sub) * qstep;
    const float4* qp3 = qb + (3 ^ sub) * qstep;
#pragma unroll
    for (int j = 0; j < 4; ++j) my_list[j * TS_KL + lane] = ListEntry{ZB_SENTINEL, TS_NOPOS, 0u};
    u64 mythr = ZB_SENTINEL;  // filter of MY query: the list's n'-th key or the shared bound
    __syncwarp();

    for (u32 b = 0; b < nblocks; ++b) {
        const u32 nrows = min((u32)TS_RB, L - b * TS_RB);
        const u32 base = (u32)(inf.moff + (long long)b * TS_RB);  // position of row 0 of the block
        // tombstone words covering positions base .. base+127 (at most 5 words), one per lane
        u32 tw = 0;
        if (lane < 5) tw = tp.bm_tomb[(base >> 5) + lane];
        // Bound shared by every visit of my query (other trees, other row slabs, other SMs): k distinct candidates
        // at or below it already exist, so anything above it cannot reach the query's final top-k.  Stale reads
        // only cost extra candidates.
        u64 gbound = ZB_SENTINEL;
        if (sub < nq_mine) gbound = __ldcg(tp.gthr + my_q);
        float4 acc[NR][4];
#pragma unroll
        for (int i = 0; i < NR; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[i][k] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int sl = 0; sl < nsl; ++sl) {
            const int kcs = min(TS_KC, chunks - sl * TS_KC);
            TS_T(t_w0);
            mbar_wait(cx.bar_full + 8 * buf, ph);
            TS_T(t_w1);
            TS_ACC(1, t_w0, t_w1);
            const float4* rp = reinterpret_cast<const float4*>(cx.s_stage + (size_t)buf * TS_STAGE_BYTES) + r0 * (TS_SLICE_FLOATS / 4) + sub;
            const int qo = sl * (TS_SLICE_FLOATS / 4);
            constexpr int rstep = RSTRIDE * TS_SLICE_FLOATS / 4;  // RSTRIDE rows apart, in float4 units
            auto chunk = [&](int c) {
                const float4 q0 = qp0[qo + c * 4], q1 = qp1[qo + c * 4], q2 = qp2[qo + c * 4], q3 = qp3[qo + c * 4];
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    const float4 r = rp[c * 4 + i * rstep];
                    if (METRIC == 0) {
                        fma4_x2(acc[i][0], r, q0); fma4_x2(acc[i][1], r, q1); fma4_x2(acc[i][2], r, q2); fma4_x2(acc[i][3], r, q3);
                    } else {
                        l2acc4_x2(acc[i][0], r, q0); l2acc4_x2(acc[i][1], r, q1); l2acc4_x2(acc[i][2], r, q2); l2acc4_x2(acc[i][3], r, q3);
                    }
                }
            };
            if (kcs == TS_KC) {  // the common case, straight-line: the next chunk's shared-memory loads can be hoisted over this chunk's math
#pragma unroll
                for (int c = 0; c < TS_KC; ++c) chunk(c);
            } else {
#pragma unroll 1
                for (int c = 0; c < kcs; ++c) chunk(c);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(cx.bar_empty + 8 * buf);
            if (++buf == S) { buf = 0; ph ^= 1u; }
            TS_T(t_w2);
            TS_ACC(2, t_w1, t_w2);
        }
        TS_T(t_e0);
        // ---- epilogue of the row block: fold the quad's partial sums (canonical tree: lane j + lane j+8, then
        //      + 4, then (r0+r1)+(r2+r3)); thread `sub` finishes query `sub`'s NR candidates ----
        if (gbound < mythr) mythr = gbound;
        u64 keys[NR];
        u32 hm = 0;  // candidates that pass the filter
#pragma unroll
        for (int i = 0; i < NR; ++i) {
            const float4 x0 = add4_xor(acc[i][0], acc[i][2], 2);
            const float4 x1 = add4_xor(acc[i][1], acc[i][3], 2);
            const float4 y = add4_xor(x0, x1, 1);
            const float sum = __fadd_rn(__fadd_rn(y.x, y.y), __fadd_rn(y.z, y.w));
            const u32 r = (u32)(i * RSTRIDE + r0);
            keys[i] = ZB_SENTINEL;
            if (r < nrows && sub < nq_mine) {
                if (METRIC == 0) keys[i] = cos_bits_rinv(sum, tp.bm_rinv[base + r], my_qrinv);
                else keys[i] = METRIC == 1 ? l2sq_bits(sum) : l2_bits(sum);
                if (keys[i] <= mythr) hm |= 1u << i;
            }
        }
        // ---- warp-private register top-n': lane l holds the l-th best (key, pos) of (query j, this row slab).
        //      Most blocks have no candidate under the filter: one ballot and out. ----
        unsigned anym = __ballot_sync(0xffffffffu, hm != 0);
        TS_T(t_e1);
        TS_ACC(3, t_e0, t_e1);
        if (anym) {
#pragma unroll 1
            for (int j = 0; j < nq_mine; ++j) {
                const unsigned qmask = 0x11111111u << j;  // lanes whose query is j
                if (!(anym & qmask)) continue;
                const bool mine = (qmask >> lane) & 1u;
                const int np = (int)__shfl_sync(0xffffffffu, my_np, j);
                ListEntry le = my_list[j * TS_KL + lane];
                u64 Lk = le.key;
                u32 Lp = le.pos;
                u64 thr = shfl64(mythr, j);  // lane j has sub == j
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    unsigned m = __ballot_sync(0xffffffffu, mine && ((hm >> i) & 1u) && keys[i] <= thr);
                    while (m) {
                        const int src = __ffs(m) - 1;
                        m &= m - 1;
                        const u64 nk = shfl64(keys[i], src);
                        if (nk > thr) continue;  // the filter tightened since the ballot
                        const u32 npos = base + (u32)(i * RSTRIDE + wr * 8 + (src >> 2));
                        const u32 w = __shfl_sync(0xffffffffu, tw, (int)((npos >> 5) - (base >> 5)));
                        if ((w >> (npos & 31)) & 1u) continue;  // tombstoned (D1)
                        const unsigned mm = __ballot_sync(0xffffffffu, kp_less(nk, npos, Lk, Lp));
                        const int ins = mm ? __ffs(mm) - 1 : 32;
                        if (ins >= np) continue;
                        const u64 upk = shfl_up64(Lk);
                        const u32 upp = __shfl_up_sync(0xffffffffu, Lp, 1);
                        if (lane > ins) { Lk = upk; Lp = upp; }
                        else if (lane == ins) { Lk = nk; Lp = npos; }
                        const u64 lk = shfl64(Lk, np - 1);
                        if (lk < thr) thr = lk;
                    }
                }
                my_list[j * TS_KL + lane] = ListEntry{Lk, Lp, 0u};
                if (mine) mythr = thr;
                // publish: a full list of n' == top_k distinct rows bounds the query's final k-th best
                if (lane == j && np == (int)tp.top_k && thr < gbound) atomicMin(tp.gthr + my_q, thr);
            }
            __syncwarp();
        }
        TS_T(t_e2);
        TS_ACC(4, t_e1, t_e2);
    }
}

static __host__ __device__ __forceinline__ size_t ts_team_bytes(int nst, int dimp) {
    size_t b = (size_t)nst * TS_STAGE_BYTES + (size_t)TS_QT * dimp * 4 + (size_t)TS_TWARPS * 4 * TS_KL * sizeof(ListEntry) +
               2 * sizeof(TileInfo) + (2 * TS_MAX_STAGES + 4) * 8;
    return (b + 1023) & ~(size_t)1023;
}

// Two teams per CTA, each = 4 math warps (one per SM sub-partition) + 1 producer warp, each streaming its own tiles:
// the two math warps that share a sub-partition belong to different tiles, so one warp's fold / insertion / tile
// change overlaps the other's FP32 loop, and a bandwidth-bound tile (few queries) shares the SM with a pipe-bound one.
template <int METRIC>
__global__ void __launch_bounds__(TS_THREADS, 1)
tile_scan_kernel(const __grid_constant__ CUtensorMap tmap, ForestView f, TileParams tp) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int dimp = f.dimp, chunks = f.chunks;
    const int nsl = (chunks + TS_KC - 1) / TS_KC;
    const u32 S = (u32)tp.nst;
    const size_t team_bytes = ts_team_bytes(tp.nst, dimp);
    // ---- carve shared memory (per team) ----
    const int team = warp < TS_CWARPS ? warp / TS_TWARPS : (warp - TS_CWARPS) % TS_TEAMS;
    unsigned char* tb = smem + (size_t)team * team_bytes;
    unsigned char* s_stage = tb;                                                       // [S][RB][48] f32
    float* s_q = reinterpret_cast<float*>(tb + (size_t)S * TS_STAGE_BYTES);             // [QT][dimp]
    ListEntry* s_list = reinterpret_cast<ListEntry*>(s_q + (size_t)TS_QT * dimp);       // [TWARPS][4][KL]
    TileInfo* s_info = reinterpret_cast<TileInfo*>(s_list + TS_TWARPS * 4 * TS_KL);     // [2]
    u64* s_bar = reinterpret_cast<u64*>(s_info + 2);                                    // full[8], empty[8], ifull[2], qfull, qempty
    const u32 bar_full = smem_u32(s_bar), bar_empty = smem_u32(s_bar + TS_MAX_STAGES);
    const u32 bar_ifull = smem_u32(s_bar + 2 * TS_MAX_STAGES), bar_qfull = bar_ifull + 16, bar_qempty = bar_ifull + 24;

    if (tid == 0) {
        for (int t = 0; t < TS_TEAMS; ++t) {
            const u32 o = (u32)(t * team_bytes);  // this thread is in team 0: the other teams' barriers sit team_bytes apart
            for (u32 i = 0; i < S; ++i) {
                mbar_init(bar_full + o + 8 * i, 1);
                mbar_init(bar_empty + o + 8 * i, TS_TWARPS);
            }
            mbar_init(bar_ifull + o, 1);
            mbar_init(bar_ifull + o + 8, 1);
            mbar_init(bar_qfull + o, 1);
            mbar_init(bar_qempty + o, TS_TWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (warp >= TS_CWARPS) {
        // =========================== producer warpgroup: one thread per team drives TMA ===========================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp >= TS_CWARPS + TS_TEAMS || lane != 0) return;
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
        const u32 ntiles = *tp.ntiles;
        u32 buf = 0, eph = 1;  // ring slot of the next stage to issue; parity to wait for on its empty barrier (first lap: free)
        u32 tile = atomicAdd(tp.tile_counter, 1u);
        for (u32 it = 0;; ++it) {
            TileInfo* inf = s_info + (it & 1);
            if (tile >= ntiles) {
                inf->tile = 0xFFFFFFFFu;
                mbar_arrive(bar_ifull + 8 * (it & 1));
                break;
            }
            const u32 leaf = tp.tile_leaf[tile], first = tp.tile_first[tile], nqt = tp.tile_count[tile];
            const u32 L = f.leaf_len[leaf];
            const long long moff = f.leaf_off[leaf];
            inf->tile = tile; inf->leaf = leaf; inf->first = first; inf->nqt = nqt; inf->L = L; inf->moff = moff;
            mbar_arrive(bar_ifull + 8 * (it & 1));
            const u32 nblocks = (L + TS_RB - 1) / TS_RB;
            const u32 total = nblocks * (u32)nsl;
            // Sibling tiles (same leaf, other queries) are dispatched back to back, so they start within about a
            // microsecond of each other on other SMs; pacing keeps them within TS_PACE_WINDOW stages so that the
            // second reader of a row block finds it in L2 instead of going to HBM again.
            const bool has_prev = tp.pace_window && tile > 0 && tp.tile_leaf[tile - 1] == leaf;
            const bool has_next = tp.pace_window && tile + 1 < ntiles && tp.tile_leaf[tile + 1] == leaf;
            volatile u32* prog = tp.tile_prog;
            u32 b = 0, sl = 0, done = 0;
            auto issue = [&](u32 count) {
                for (u32 j = 0; j < count; ++j, ++done) {
                    if ((has_prev || has_next) && (done % TS_PACE_EVERY) == 0) {
                        prog[tile] = done;
                        if (done > tp.pace_window) {
                            const u32 lim = done - tp.pace_window;
                            if (has_prev) while (prog[tile - 1] < lim) {}
                            if (has_next) while (prog[tile + 1] < lim) {}
                        }
                    }
                    mbar_wait(bar_empty + 8 * buf, eph);
                    mbar_arrive_expect_tx(bar_full + 8 * buf, TS_STAGE_BYTES);
                    tma_2d_g2s(smem_u32(s_stage + (size_t)buf * TS_STAGE_BYTES), &tmap, (int)(sl * TS_SLICE_FLOATS),
                               (int)(moff + (long long)b * TS_RB), bar_full + 8 * buf);
                    if (++sl == (u32)nsl) { sl = 0; ++b; }
                    if (++buf == S) { buf = 0; eph ^= 1u; }
                }
            };
            // rows of this tile may run ahead into the ring while the math warps still finish the previous tile ...
            const u32 pre = total < S ? total : S;
            issue(pre);
            // ... the resident query block is single-buffered: wait until the previous tile is done with it
            if (it > 0) mbar_wait(bar_qempty, (it - 1) & 1);
            mbar_arrive_expect_tx(bar_qfull, nqt * (u32)dimp * 4u);
            {  // address loads batched (8 independent chains), then the copies
                u32 qi[TS_QT];
#pragma unroll
                for (int j = 0; j < TS_QT; ++j) qi[j] = (u32)j < nqt ? tp.order[first + j] : 0u;
#pragma unroll
                for (int j = 0; j < TS_QT; ++j) qi[j] = (u32)j < nqt ? tp.v_q[qi[j]] : 0u;
#pragma unroll
                for (int j = 0; j < TS_QT; ++j)
                    if ((u32)j < nqt)
                        bulk_g2s(smem_u32(s_q + (size_t)j * dimp), tp.queries + (size_t)qi[j] * dimp, (u32)dimp * 4u, bar_qfull);
            }
            issue(total - pre);
            if (has_prev || has_next) prog[tile] = 0xFFFFFFFFu;
            // fetched only now (not while the tile is in flight), so consecutive tiles start back to back
            const u32 next_tile = atomicAdd(tp.tile_counter, 1u);
            atomicAdd(&tp.stats[0], (u64)nqt);
            atomicAdd(&tp.stats[1], (u64)nqt * L);
            atomicAdd(&tp.stats[2], ((u64)L + nqt) * (u64)dimp * 4ull);  // algorithmic bytes: leaf rows once + the tile's queries
            tile = next_tile;
        }
        return;
    }

    // =================================== consumer (math) warps ===================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    ScanCtx cx;
    cx.s_stage = s_stage; cx.s_q = s_q; cx.s_list = s_list;
    cx.bar_full = bar_full; cx.bar_empty = bar_empty;
    cx.S = S; cx.dimp = dimp; cx.chunks = chunks; cx.nsl = nsl;
    const int tw = warp % TS_TWARPS, sub = lane & 3;
    u32 rbuf = 0, rph = 0;  // ring position of the next stage to consume: slot and phase parity
#ifdef ZB_SCAN_TIMING
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define TS_TACC , tacc
#else
#define TS_TACC
#endif
    for (u32 it = 0;; ++it) {
        TS_T(t_tile0);
        mbar_wait(bar_ifull + 8 * (it & 1), (it >> 1) & 1);
        const TileInfo inf = s_info[it & 1];
        if (inf.tile == 0xFFFFFFFFu) break;
        const u32 nqt = inf.nqt;
        // Role of this warp for the tile: 5..8 queries = two groups of 4, each scanned by a pair of wide warps (64 rows
        // of every 128-row stage each); 1..4 queries = one group scanned by four narrow warps (32 rows each).  Either
        // way every sub-partition carries the same FMA-pipe load.
        const bool narrow = nqt <= 4;
        const int g = narrow ? 0 : tw >> 1, wr = narrow ? tw : tw & 1;
        const int nq_mine = min(4, (int)nqt - g * 4);
        // my query (slot `sub` of group g): visit, n', reciprocal norm
        u32 my_visit = 0, my_np = 0, my_q = 0;
        double my_qrinv = 0.0;
        if (sub < nq_mine) {
            my_visit = tp.order[inf.first + g * 4 + sub];
            my_np = tp.v_np[my_visit];
            my_q = tp.v_q[my_visit];
            if (METRIC == 0) my_qrinv = tp.q_rinv[my_q];
        }
        mbar_wait(bar_qfull, it & 1);
        TS_T(t_tile1);
        TS_ACC(0, t_tile0, t_tile1);
        if (narrow) scan_tile<METRIC, 4>(cx, f, tp, inf, g, wr, tw, lane, rbuf, rph, my_np, my_q, my_qrinv, nq_mine TS_TACC);
        else scan_tile<METRIC, 8>(cx, f, tp, inf, g, wr, tw, lane, rbuf, rph, my_np, my_q, my_qrinv, nq_mine TS_TACC);
        TS_T(t_m0);
        // ---- end of tile: release the query block, merge the row slabs of each group, write the visits' top lists ----
        if (lane == 0) mbar_arrive(bar_qempty);
        asm volatile("bar.sync %0, 128;" ::"r"(team + 1) : "memory");  // the team's lists are final and visible
        if (wr == 0) {  // the group's first warp merges its 2 (wide) or 4 (narrow) slabs, which sit in consecutive list blocks
            const int nslab = narrow ? 4 : 2;
            const ListEntry* mine_l = s_list + (size_t)tw * 4 * TS_KL;
#pragma unroll 1
            for (int j = 0; j < nq_mine; ++j) {
                const int np = (int)__shfl_sync(0xffffffffu, my_np, j);
                const u32 v = __shfl_sync(0xffffffffu, my_visit, j);
                ListEntry a = mine_l[j * TS_KL + lane];
                u64 k = a.key;
                u32 p = a.pos;
#pragma unroll 1
                for (int o = 1; o < nslab; ++o) {
                    const ListEntry bb = mine_l[(size_t)o * 4 * TS_KL + j * TS_KL + (31 - lane)];
                    if (kp_less(bb.key, bb.pos, k, p)) { k = bb.key; p = bb.pos; }  // 32 smallest of the union, bitonic
#pragma unroll
                    for (int x = 16; x >= 1; x >>= 1) {
                        const u64 ok = shfl_xor64(k, x);
                        const u32 op = __shfl_xor_sync(0xffffffffu, p, x);
                        const bool lower = (lane & x) == 0;
                        const bool other_less = kp_less(ok, op, k, p);
                        if (lower == other_less) { k = ok; p = op; }
                    }
                }
                const u32 e0 = tp.v_ent_off[v], e1 = tp.v_ent_off[v + 1];
                if ((u32)lane < e1 - e0) {
                    Entry e{ZB_SENTINEL, ZB_SENTINEL};
                    if (lane < np && p != TS_NOPOS) e = Entry{k, f.ord[f.members[p]]};
                    tp.entries[e0 + lane] = e;
                }
            }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(team + 1) : "memory");  // lists may be re-initialised for the next tile
        TS_T(t_m1);
        TS_ACC(5, t_m0, t_m1);
    }
#ifdef ZB_SCAN_TIMING
    if (lane == 0)
        for (int i = 0; i < 8; ++i) atomicAdd(&tp.stats[8 + i], (u64)tacc[i]);
#endif
}

// =====================================================================================================
// Third-generation fused leaf-tile scan (zb_scan3_kernel.cuh): device-side primitives, then the kernel.
// =====================================================================================================
typedef CUtensorMap T3Map;
__device__ __forceinline__ bool t3_isinf_pos(double x) { return isinf(x) && x > 0.0; }
__device__ __forceinline__ double t3_dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double t3_dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ u64 t3_dbits(double x) { return (u64)__double_as_longlong(x); }
__device__ __forceinline__ float t3_fadd(float a, float b) { return __fadd_rn(a, b); }
__host__ __device__ __forceinline__ u32 t3_fbits(float x) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(x);
#else
    u32 b; memcpy(&b, &x, 4); return b;
#endif
}
__host__ __device__ __forceinline__ float t3_bitsf(u32 b) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float x; memcpy(&x, &b, 4); return x;
#endif
}
__device__ __forceinline__ float t3_fadd_ru(float a, float b) { return __fadd_ru(a, b); }
__device__ __forceinline__ float t3_fmul_ru(float a, float b) { return __fmul_ru(a, b); }
__device__ __forceinline__ float t3_fmaf(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ float t3_fsub(float a, float b) { return __fsub_rn(a, b); }
typedef float4 T3F4;
__device__ __forceinline__ T3F4 t3_ld_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ u64 t3_pk2(float lo, float hi) { return pk2(lo, hi); }
__device__ __forceinline__ void t3_upk2(u64 v, float& lo, float& hi) { upk2(v, lo, hi); }
#ifndef T3_ASM_ORDER
#define T3_ASM_ORDER   // `volatile` pins the FP32 stream to the order the kernel body states (needed by the T3_KC == 2 pipelining; no gain for 3)
#endif
__device__ __forceinline__ u64 t3_fma2(u64 a, u64 b, u64 c) {  // two IEEE fused multiply-adds (bit-identical to __fmaf_rn per half)
    u64 d;
    asm T3_ASM_ORDER("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ u64 t3_sub2(u64 a, u64 b) {
    u64 d;
    asm T3_ASM_ORDER("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 t3_ldcg_u64(const u64* p) { return __ldcg(p); }
__device__ __forceinline__ void t3_atomic_min_u64(u64* p, u64 v) { atomicMin(p, v); }
__device__ __forceinline__ u64 t3_shfl64(u64 v, int src) { return shfl64(v, src); }
__device__ __forceinline__ double t3_shfl_f64(double v, int src) { return __longlong_as_double((long long)shfl64((u64)__double_as_longlong(v), src)); }
__device__ __forceinline__ u64 t3_shfl_up64(u64 v) { return shfl_up64(v); }
__device__ __forceinline__ void t3_team_sync(int team, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(threads) : "memory"); }
__device__ __forceinline__ void t3_fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// register split of the CTA's allocation between the math warps and the producer warpgroup (setmaxnreg): 4 math warps per team =
// 384 threads launched with 168 registers: 256 x 232 + 128 x 40 = 384 x 168;  8 per team = 640 threads launched with 96:
// 512 x 112 + 128 x 32 = 640 x 96
#ifndef T3_REGS_MATH
#define T3_REGS_MATH 232
#define T3_REGS_AUX 40
#endif
#define T3_STR2(x) #x
#define T3_STR(x) T3_STR2(x)
static_assert(256 * T3_REGS_MATH + 128 * T3_REGS_AUX <= 384 * 168, "setmaxnreg split exceeds the CTA's registers");
template <int TW>
__device__ __forceinline__ void t3_setmaxnreg_dec() {
    if (TW == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 " T3_STR(T3_REGS_AUX) ";");
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
}
template <int TW>
__device__ __forceinline__ void t3_setmaxnreg_inc() {
    if (TW == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 " T3_STR(T3_REGS_MATH) ";");
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
}
__device__ __forceinline__ void t3_prefetch_map(const T3Map& m) { asm volatile("prefetch.tensormap [%0];" ::"l"(&m) : "memory"); }
__device__ __forceinline__ void t3_tma_2d_g2s(u32 dst, const T3Map& map, int c0, long long row, u32 bar) {
    tma_2d_g2s(dst, &map, c0, (int)row, bar);
}
__device__ __forceinline__ void t3_prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ bool t3_above_from_dot(float dot, float constant) { return above_from_dot(dot, constant); }
}  // namespace zb
#include "zb_scan3_kernel.cuh"
namespace zb {

// KR = list entries per lane: 1 serves n' <= 32, 4 serves n' <= 128 (BASELINE config 5 asks for top-100); TW = math warps per team
template <int METRIC, int KR, int TW>
__global__ void __launch_bounds__(T3Shape<TW>::THREADS, 1) tile_scan3_kernel(const __grid_constant__ CUtensorMap tmap, ForestView f, T3Params tp) {
    extern __shared__ __align__(1024) unsigned char smem3[];
    t3_body<METRIC, 0, KR, TW>(tmap, f, tp, smem3);
}
// Second pass of the dot-product filter (METRIC 3 of the kernel above): exact keys of every visit's candidates, one warp per visit.
#define RF_THREADS 256
template <int METRIC>
__global__ void __launch_bounds__(RF_THREADS) refine_visits_kernel(ForestView f, T3RefineParams rp) {
    t3_refine_warp<METRIC>(f, rp, (int)(threadIdx.x & 31u));
}
// Flat-table projection on the same skeleton (MODE 1): tmap covers the INPUT rows, tp.queries the plane coefficients.
__global__ void __launch_bounds__(T3Shape<4>::THREADS, 1) project3_kernel(const __grid_constant__ CUtensorMap tmap, ForestView f, T3Params tp) {
    extern __shared__ __align__(1024) unsigned char smem3[];
    t3_body<0, 1, 1, 4>(tmap, f, tp, smem3);
}

// =====================================================================================================
// grouping of visits by leaf and tile construction (all on device; no host round trip)
// =====================================================================================================
__global__ void ts_count_kernel(ForestView f, u32 nv, const u32* __restrict__ v_leaf, const u32* __restrict__ v_np,
                                u32 min_rows, u32 kmax, u32* __restrict__ leaf_count) {
    u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    u32 leaf = v_leaf[v];
    if (f.leaf_len[leaf] >= min_rows && v_np[v] <= kmax) atomicAdd(&leaf_count[leaf], 1u);
}
__global__ void ts_tilecount_kernel(u32 nleaves, const u32* __restrict__ leaf_count, u32 tq, u32* __restrict__ tile_cnt) {
    u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l <= nleaves) tile_cnt[l] = l < nleaves ? (leaf_count[l] + tq - 1) / tq : 0u;
}
__global__ void ts_scatter_kernel(ForestView f, u32 nv, const u32* __restrict__ v_leaf, const u32* __restrict__ v_np,
                                  u32 min_rows, u32 kmax, const u32* __restrict__ leaf_start, u32* __restrict__ leaf_cursor,
                                  u32* __restrict__ order, u64* __restrict__ v_pair_len, u8* __restrict__ v_done) {
    u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    u32 leaf = v_leaf[v];
    if (f.leaf_len[leaf] >= min_rows && v_np[v] <= kmax) {
        u32 pos = leaf_start[leaf] + atomicAdd(&leaf_cursor[leaf], 1u);
        order[pos] = v;
        v_pair_len[v] = 0;
        v_done[v] = 1;
    }
}
__global__ void ts_filltiles_kernel(u32 nleaves, const u32* __restrict__ leaf_count, const u32* __restrict__ leaf_start,
                                    const u32* __restrict__ tile_start, u32 tq, u32* __restrict__ tile_leaf,
                                    u32* __restrict__ tile_first, u32* __restrict__ tile_count, const u32* __restrict__ leaf_len,
                                    u64 row_bytes, u64* __restrict__ unique_bytes) {
    u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nleaves) return;
    const u32 c = leaf_count[l], ts = tile_start[l];
    if (!c) return;
    atomicAdd(unique_bytes, (u64)leaf_len[l] * row_bytes);  // the floor of the scan's HBM traffic: every visited leaf once
    const u32 nt = (c + tq - 1) / tq;   // full tiles first, the remainder last (cost is per started query group)
    for (u32 j = 0, done = 0; j < nt; ++j) {
        const u32 n = c - done < tq ? c - done : tq;
        tile_leaf[ts + j] = l;
        tile_first[ts + j] = leaf_start[l] + done;
        tile_count[ts + j] = n;
        done += n;
    }
}

// Longest-processing-time-first dispatch: leaves ordered by (rows x visiting queries) descending, the tiles of one leaf
// kept together (sibling tiles start back to back and share the leaf's rows through L2).  The persistent teams pull tiles
// from one counter, so the big tiles go first and the short ones fill the tail.
__global__ void ts_leafkey_kernel(u32 nleaves, const u32* __restrict__ leaf_count, const u32* __restrict__ leaf_len,
                                  u32* __restrict__ key, u32* __restrict__ val) {
    const u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nleaves) return;
    const u64 cost = (u64)leaf_count[l] * leaf_len[l];
    key[l] = leaf_count[l] ? ~(u32)(cost > 0xFFFFFFFEull ? 0xFFFFFFFEull : cost) : 0xFFFFFFFFu;  // ascending sort = cost descending, unvisited leaves last
    val[l] = l;
}
__global__ void ts_tilecount_sorted_kernel(u32 nleaves, const u32* __restrict__ sorted_leaf, const u32* __restrict__ leaf_count, u32 tq,
                                           u32* __restrict__ tile_cnt) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= nleaves) tile_cnt[i] = i < nleaves ? (leaf_count[sorted_leaf[i]] + tq - 1) / tq : 0u;
}
__global__ void ts_filltiles_sorted_kernel(u32 nleaves, const u32* __restrict__ sorted_leaf, const u32* __restrict__ leaf_count,
                                           const u32* __restrict__ leaf_start, const u32* __restrict__ tile_start, u32 tq,
                                           u32* __restrict__ tile_leaf, u32* __restrict__ tile_first, u32* __restrict__ tile_count,
                                           const u32* __restrict__ leaf_len, u64 row_bytes, u64* __restrict__ unique_bytes) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nleaves) return;
    const u32 l = sorted_leaf[i];
    const u32 c = leaf_count[l], ts = tile_start[i];
    if (!c) return;
    atomicAdd(unique_bytes, (u64)leaf_len[l] * row_bytes);
    const u32 nt = (c + tq - 1) / tq;
    // the leaf's queries spread evenly over its tiles: 17 queries are 9 + 8, not 16 + 1 (the cost of a tile grows in steps of QH)
    const u32 per = c / nt, extra = c - per * nt;
    for (u32 j = 0, done = 0; j < nt; ++j) {
        const u32 n = per + (j < extra ? 1u : 0u);
        tile_leaf[ts + j] = l;
        tile_first[ts + j] = leaf_start[l] + done;
        tile_count[ts + j] = n;
        done += n;
    }
}

// reciprocal norms 1/sqrt(|x|^2) in f64 from the canonical f32 squared norm (one quad per vector)
__global__ void __launch_bounds__(128) rinv_kernel(const float* __restrict__ x_, u64 n, int dimp, double* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    const float4* x = reinterpret_cast<const float4*>(x_ + i * dimp);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < dimp / 16; ++c) {
        float4 v = x[c * 4 + sub];
        fma4(acc, v, v);
    }
    float sum = quad_reduce16(acc, quad_mask());
    if (sub == 0) out[i] = __ddiv_rn(1.0, __dsqrt_rn((double)sum));
}
void launch_rinv(const float* d_x, u64 n, int dimp, double* d_out, cudaStream_t s) {
    if (!n) return;
    rinv_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_x, n, dimp, d_out);
}

// canonical squared norms in f32 (one quad per vector): what METRIC 3 of the third-generation scan adds to -2 a.q
__global__ void __launch_bounds__(128) n2_kernel(const float* __restrict__ x_, u64 n, int dimp, float* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    const float4* x = reinterpret_cast<const float4*>(x_ + i * dimp);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < dimp / 16; ++c) {
        float4 v = x[c * 4 + sub];
        fma4(acc, v, v);
    }
    float sum = quad_reduce16(acc, quad_mask());
    if (sub == 0) out[i] = sum;
}
void launch_n2(const float* d_x, u64 n, int dimp, float* d_out, cudaStream_t s) {
    if (!n) return;
    n2_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_x, n, dimp, d_out);
}
// largest usable squared norm of every leaf (one warp per leaf): the leaf's share of the filter's error bound
__global__ void __launch_bounds__(256) leaf_n2max_kernel(u32 nleaves, const long long* __restrict__ leaf_off, const u32* __restrict__ leaf_len,
                                                         const float* __restrict__ n2, float* __restrict__ out) {
    const u32 l = blockIdx.x * 8u + (threadIdx.x >> 5);
    if (l >= nleaves) return;
    const u32 lane = threadIdx.x & 31u, len = leaf_len[l];
    const float* x = n2 + leaf_off[l];
    float m = 0.f;
    for (u32 i = lane; i < len; i += 32u) {
        const float v = x[i];
        if (v <= T3_N2_LIMIT && v > m) m = v;   // NaN and inf compare false
    }
    for (int o = 16; o >= 1; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) out[l] = m;
}
void launch_leaf_n2max(u32 nleaves, const long long* d_leaf_off, const u32* d_leaf_len, const float* d_n2, float* d_out, cudaStream_t s) {
    if (!nleaves) return;
    leaf_n2max_kernel<<<(nleaves + 7) / 8, 256, 0, s>>>(nleaves, d_leaf_off, d_leaf_len, d_n2, d_out);
}

static size_t ts_smem_bytes(int nst, int dimp) { return TS_TEAMS * ts_team_bytes(nst, dimp) + 1024; }

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        ZB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        ZB_REQUIRE(p && qres == cudaDriverEntryPointSuccess, ZB_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
        fn = (EncodeTiledFn)p;
    }
    return fn;
}
void make_row_tile_map(void* out_map128, const float* bm_rows, u64 positions, int dimp, int box_rows, int box_floats) {
    CUtensorMap* m = reinterpret_cast<CUtensorMap*>(out_map128);
    cuuint64_t gdim[2] = {(cuuint64_t)dimp, (cuuint64_t)(positions ? positions : 1)};
    cuuint64_t gstride[1] = {(cuuint64_t)dimp * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_floats, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode_tiled_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)bm_rows, gdim, gstride, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    ZB_REQUIRE(r == CUDA_SUCCESS, ZB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
}

int tile_scan_box_floats(int generation) { return generation == 2 ? TS_SLICE_FLOATS : T3_SLICE_FLOATS; }

bool tile_scan_supported(int dimp, u32 top_k) {
    int dev = 0, max_smem = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    return top_k >= 1 && top_k <= TS_KL && ts_smem_bytes(2, dimp) <= (size_t)max_smem;
}

void tile_scan(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
               u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, u64* v_pair_len,
               u8* v_done, Entry* entries, u32 top_k, u32 min_rows, u32 tile_queries, u32 nleaves, cudaStream_t s) {
    ws.launched = false;
    ws.filtered = false;
    const u32 pace_window = tile_queries >> 9;  // knob: bits 9.. of tile_queries carry the pacing window (tests / ablations)
    const bool lpt_order = false;               // second generation: tiles stay in leaf order
    tile_queries &= 0xFF;
    if (!nv || !nleaves || !tile_scan_supported(f.dimp, top_k)) return;
    const u32 tq = tile_queries >= 1 && tile_queries <= TS_QT ? tile_queries : TS_QT;
    int dev = 0, max_smem = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int nst = 0;
    for (int cand = TS_MAX_STAGES; cand >= 2; --cand)
        if (ts_smem_bytes(cand, f.dimp) <= (size_t)max_smem) { nst = cand; break; }
    if (!nst) return;
    const size_t smem = ts_smem_bytes(nst, f.dimp);

    ws.leaf_count.ensure(nleaves + 1);
    ws.leaf_start.ensure(nleaves + 1);
    ws.leaf_cursor.ensure(nleaves + 1);
    ws.order.ensure(nv);
    ws.tile_leaf.ensure(nv);
    ws.tile_first.ensure(nv);
    ws.counters.ensure(64);
    ws.tile_prog.ensure(nv);
    ZB_CUDA(cudaMemsetAsync(ws.tile_prog.p, 0, (size_t)nv * 4, s));
    ws.gthr.ensure(nq ? nq : 1);
    ZB_CUDA(cudaMemsetAsync(ws.gthr.p, 0xFF, (size_t)(nq ? nq : 1) * 8, s));
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const u32*)nullptr, (u32*)nullptr, (long long)(nleaves + 1));
    ws.tmp.ensure(tmp_bytes + 256);

    ZB_CUDA(cudaMemsetAsync(ws.leaf_count.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.leaf_cursor.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    const u32 kmax = top_k;
    ts_count_kernel<<<(nv + 255) / 256, 256, 0, s>>>(f, nv, v_leaf, v_np, min_rows, kmax, ws.leaf_count.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.leaf_count.p, ws.leaf_start.p, (long long)(nleaves + 1), s);
    ts_scatter_kernel<<<(nv + 255) / 256, 256, 0, s>>>(f, nv, v_leaf, v_np, min_rows, kmax, ws.leaf_start.p,
                                                       ws.leaf_cursor.p, ws.order.p, v_pair_len, v_done);
    // tiles: per-leaf counts -> exclusive scan (tile_start, total at [nleaves]) -> fill
    ws.tile_per_leaf.ensure(nleaves + 1);
    ws.tile_start.ensure(nleaves + 1);
    ws.tile_cnt.ensure(nv);
    if (lpt_order) {
        for (int b = 0; b < 2; ++b) {
            ws.sort_key[b].ensure(nleaves);
            ws.sort_val[b].ensure(nleaves);
        }
        size_t sort_bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const u32*)nullptr, (u32*)nullptr, (const u32*)nullptr, (u32*)nullptr,
                                        (long long)nleaves, 0, 32, s);
        ws.sort_tmp.ensure(sort_bytes + 256);
        ts_leafkey_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, f.leaf_len, ws.sort_key[0].p, ws.sort_val[0].p);
        cub::DeviceRadixSort::SortPairs(ws.sort_tmp.p, sort_bytes, ws.sort_key[0].p, ws.sort_key[1].p, ws.sort_val[0].p, ws.sort_val[1].p,
                                        (long long)nleaves, 0, 32, s);
        ts_tilecount_sorted_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.sort_val[1].p, ws.leaf_count.p, tq, ws.tile_per_leaf.p);
        cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
        ts_filltiles_sorted_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.sort_val[1].p, ws.leaf_count.p, ws.leaf_start.p,
                                                                         ws.tile_start.p, tq, ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p,
                                                                         f.leaf_len, (u64)f.dimp * 4ull,
                                                                         reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    } else {
        ts_tilecount_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, tq, ws.tile_per_leaf.p);
        cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
        ts_filltiles_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, ws.leaf_start.p, ws.tile_start.p, tq,
                                                                  ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p, f.leaf_len,
                                                                  (u64)f.dimp * 4ull, reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    }

    TileParams tp;
    tp.tile_leaf = ws.tile_leaf.p;
    tp.tile_first = ws.tile_first.p;
    tp.tile_count = ws.tile_cnt.p;
    tp.ntiles = ws.tile_start.p + nleaves;
    ws.ntiles_ptr = tp.ntiles;
    tp.tile_counter = ws.counters.p;
    tp.order = ws.order.p;
    tp.v_np = v_np;
    tp.v_q = v_q;
    tp.v_ent_off = v_ent_off;
    tp.entries = entries;
    tp.queries = d_q;
    tp.q_rinv = d_q_rinv;
    tp.bm_rinv = bm.rinv;
    tp.bm_tomb = bm.tomb;
    tp.stats = reinterpret_cast<u64*>(ws.counters.p + 4);
    tp.pace_window = pace_window;
    tp.tile_prog = ws.tile_prog.p;
    tp.gthr = ws.gthr.p;
    tp.top_k = top_k;
    tp.nst = nst;
    const CUtensorMap& tmap = *reinterpret_cast<const CUtensorMap*>(bm.tmap);
    const int grid = sms;
    if (!ws.ev0) {
        ZB_CUDA(cudaEventCreate(&ws.ev0));
        ZB_CUDA(cudaEventCreate(&ws.ev1));
    }
    ZB_CUDA(cudaEventRecord(ws.ev0, s));
    if (metric == 0) {
        ZB_CUDA(cudaFuncSetAttribute(tile_scan_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tile_scan_kernel<0><<<grid, TS_THREADS, smem, s>>>(tmap, f, tp);
    } else if (metric == 1) {
        ZB_CUDA(cudaFuncSetAttribute(tile_scan_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tile_scan_kernel<1><<<grid, TS_THREADS, smem, s>>>(tmap, f, tp);
    } else {
        ZB_CUDA(cudaFuncSetAttribute(tile_scan_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tile_scan_kernel<2><<<grid, TS_THREADS, smem, s>>>(tmap, f, tp);
    }
    ZB_CUDA(cudaGetLastError());
    ZB_CUDA(cudaEventRecord(ws.ev1, s));
    ws.launched = true;
    ws.launches = 7;
}

// Statistics of the last tile_scan launch (visits, scored pairs, bytes asked of HBM by design); call after the
// stream has been synchronised.
void tile_scan_stats(ScanWorkspace& ws, cudaStream_t s, u64* tile_visits, u64* tile_pairs, u64* moved_bytes, float* kernel_ms,
                     u32* tiles, u64* unique_bytes, u64* flagged_visits, u64* refined_rows, float* refine_ms) {
    *tile_visits = *tile_pairs = *moved_bytes = *unique_bytes = 0;
    *kernel_ms = 0.f;
    *tiles = 0;
    if (flagged_visits) *flagged_visits = 0;
    if (refined_rows) *refined_rows = 0;
    if (refine_ms) *refine_ms = 0.f;
    if (!ws.launched) return;
    u64 h[6] = {0, 0, 0, 0, 0, 0};
    ZB_CUDA(cudaMemcpyAsync(h, reinterpret_cast<u64*>(ws.counters.p + 4), 48, cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaMemcpyAsync(tiles, ws.ntiles_ptr, 4, cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaStreamSynchronize(s));
    cudaEventElapsedTime(kernel_ms, ws.ev0, ws.ev1);
    *tile_visits = h[0];
    *tile_pairs = h[1];
    *moved_bytes = h[2];
    *unique_bytes = h[3];
    if (ws.filtered) {
        if (flagged_visits) *flagged_visits = h[4];
        if (refined_rows) *refined_rows = h[5];
        if (refine_ms) cudaEventElapsedTime(refine_ms, ws.ev1, ws.ev2);
    }
#ifdef ZB_SCAN_TIMING
    u64 t[8];
    ZB_CUDA(cudaMemcpy(t, reinterpret_cast<u64*>(ws.counters.p + 4) + 8, 64, cudaMemcpyDeviceToHost));
    fprintf(stderr, "[scan timing, Mcycles summed over math warps] tile-wait %.1f stage-wait %.1f math %.1f fold %.1f insert %.1f merge %.1f idle %.1f\n",
            t[0] / 1e6, t[1] / 1e6, t[2] / 1e6, t[3] / 1e6, t[4] / 1e6, t[5] / 1e6, t[7] / 1e6);
#endif
}

// ---- third generation (zb_scan3_kernel.cuh): same visit grouping, tiles of up to 16 queries, 64-row stages ----
static size_t t3_smem_bytes(int nst, int dimp, int qcap, int kr) { return T3_TEAMS * (size_t)t3_layout(nst, dimp, qcap, kr).total + 1024; }
static int t3_kr(u32 top_k) { return top_k <= T3_KL ? 1 : T3_KR_MAX; }
// ring depth and query capacity for this row length: the largest tile (16, then 8, then 4 queries) that leaves >= 3 stages
static bool t3_config(int dimp, int kr, int* nst_out, int* qcap_out) {
    int dev = 0, max_smem = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    for (int qcap = T3_QT; qcap >= 4; qcap >>= 1)
        for (int nst = T3_MAX_STAGES; nst >= 3; --nst)
            if (t3_smem_bytes(nst, dimp, qcap, kr) <= (size_t)max_smem) {
                *nst_out = nst;
                *qcap_out = qcap;
                return true;
            }
    return false;
}
bool tile_scan3_supported(int dimp, u32 top_k) {
    int nst, qcap;
    return top_k >= 1 && top_k <= T3_KL * T3_KR_MAX && t3_config(dimp, t3_kr(top_k), &nst, &qcap);
}
static void t3_launch(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
                      u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, Entry* entries, u32 top_k,
                      int kr, int nst, int qcap, int sms, const u32* ntiles, const u32* nvisits, cudaStream_t s);

void tile_scan3(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
                u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, u64* v_pair_len,
                u8* v_done, Entry* entries, u32 top_k, u32 min_rows, u32 tile_queries, u32 nleaves, cudaStream_t s) {
    ws.launched = false;
    ws.filtered = false;
    int nst = 0, qcap = 0;
    const int kr = t3_kr(top_k);
    if (!nv || !nleaves || top_k < 1 || top_k > T3_KL * T3_KR_MAX || !t3_config(f.dimp, kr, &nst, &qcap)) return;
    const bool lpt_order = ((tile_queries >> 8) & 1u) == 0;  // knob bit 8 of tile_queries: 1 = tiles in leaf order (ablation)
    tile_queries &= 0xFF;
    const u32 tq = tile_queries >= 1 && tile_queries <= (u32)qcap ? tile_queries : (u32)qcap;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);

    ws.leaf_count.ensure(nleaves + 1);
    ws.leaf_start.ensure(nleaves + 1);
    ws.leaf_cursor.ensure(nleaves + 1);
    ws.order.ensure(nv);
    ws.tile_leaf.ensure(nv);
    ws.tile_first.ensure(nv);
    ws.counters.ensure(64);
    ws.gthr.ensure(nq ? nq : 1);
    ZB_CUDA(cudaMemsetAsync(ws.gthr.p, 0xFF, (size_t)(nq ? nq : 1) * 8, s));
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const u32*)nullptr, (u32*)nullptr, (long long)(nleaves + 1));
    ws.tmp.ensure(tmp_bytes + 256);
    ZB_CUDA(cudaMemsetAsync(ws.leaf_count.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.leaf_cursor.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    const u32 kmax = top_k;
    ts_count_kernel<<<(nv + 255) / 256, 256, 0, s>>>(f, nv, v_leaf, v_np, min_rows, kmax, ws.leaf_count.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.leaf_count.p, ws.leaf_start.p, (long long)(nleaves + 1), s);
    ts_scatter_kernel<<<(nv + 255) / 256, 256, 0, s>>>(f, nv, v_leaf, v_np, min_rows, kmax, ws.leaf_start.p,
                                                       ws.leaf_cursor.p, ws.order.p, v_pair_len, v_done);
    ws.tile_per_leaf.ensure(nleaves + 1);
    ws.tile_start.ensure(nleaves + 1);
    ws.tile_cnt.ensure(nv);
    if (lpt_order) {
        for (int b = 0; b < 2; ++b) {
            ws.sort_key[b].ensure(nleaves);
            ws.sort_val[b].ensure(nleaves);
        }
        size_t sort_bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const u32*)nullptr, (u32*)nullptr, (const u32*)nullptr, (u32*)nullptr,
                                        (long long)nleaves, 0, 32, s);
        ws.sort_tmp.ensure(sort_bytes + 256);
        ts_leafkey_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, f.leaf_len, ws.sort_key[0].p, ws.sort_val[0].p);
        cub::DeviceRadixSort::SortPairs(ws.sort_tmp.p, sort_bytes, ws.sort_key[0].p, ws.sort_key[1].p, ws.sort_val[0].p, ws.sort_val[1].p,
                                        (long long)nleaves, 0, 32, s);
        ts_tilecount_sorted_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.sort_val[1].p, ws.leaf_count.p, tq, ws.tile_per_leaf.p);
        cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
        ts_filltiles_sorted_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.sort_val[1].p, ws.leaf_count.p, ws.leaf_start.p,
                                                                         ws.tile_start.p, tq, ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p,
                                                                         f.leaf_len, (u64)f.dimp * 4ull,
                                                                         reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    } else {
        ts_tilecount_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, tq, ws.tile_per_leaf.p);
        cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
        ts_filltiles_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, ws.leaf_start.p, ws.tile_start.p, tq,
                                                                  ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p, f.leaf_len,
                                                                  (u64)f.dimp * 4ull, reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    }
    t3_launch(ws, f, bm, metric, d_q, d_q_rinv, nq, nv, v_leaf, v_np, v_q, v_ent_off, entries, top_k, kr, nst, qcap, sms,
              ws.tile_start.p + nleaves, ws.leaf_start.p + nleaves, s);
}

// The fused kernel (and the filter's second pass) over the tiles in ws.tile_leaf / tile_first / tile_cnt (*ntiles of them) and
// the visits in ws.order (*nvisits of them), both device scalars.
static void t3_launch(ScanWorkspace& ws, const ForestView& f, const BucketMajor& bm, u32 metric, const float* d_q, const double* d_q_rinv,
                      u32 nq, u32 nv, const u32* v_leaf, const u32* v_np, const u32* v_q, const u32* v_ent_off, Entry* entries, u32 top_k,
                      int kr, int nst, int qcap, int sms, const u32* ntiles, const u32* nvisits, cudaStream_t s) {
    const size_t smem = t3_smem_bytes(nst, f.dimp, qcap, kr);
    // L2 / L2 squared with short lists: score through the dot product (half the FP32 work), exact second pass below
    const bool filt = ws.l2_filter && (metric == 1 || metric == 2) && kr == 1 && top_k <= ZB_L2_FILTER_MAX_K && bm.n2 && bm.leaf_n2max;
    ws.filtered = filt;
    T3Params tp{};
    if (filt) {
        ws.q_n2.ensure(nq ? nq : 1);
        launch_n2(d_q, nq, f.dimp, ws.q_n2.p, s);
        ws.cand.ensure((size_t)nv * T3_KL);
        ws.cand_cut.ensure(nv);
        ws.cand_flag.ensure(nv);
        tp.bm_n2 = bm.n2;
        tp.q_n2 = ws.q_n2.p;
        tp.leaf_n2max = bm.leaf_n2max;
        tp.ecoef = (float)(4 * f.chunks + 32) * 5.9604645e-8f * 1.01f;   // DESIGN 3.1b
        tp.cand = ws.cand.p;
        tp.cand_cut = ws.cand_cut.p;
        tp.cand_flag = ws.cand_flag.p;
    }
    tp.tile_leaf = ws.tile_leaf.p;
    tp.tile_first = ws.tile_first.p;
    tp.tile_count = ws.tile_cnt.p;
    tp.ntiles = ntiles;
    ws.ntiles_ptr = tp.ntiles;
    tp.tile_counter = ws.counters.p;
    tp.order = ws.order.p;
    tp.v_np = v_np;
    tp.v_q = v_q;
    tp.v_ent_off = v_ent_off;
    tp.entries = entries;
    tp.queries = d_q;
    tp.q_rinv = d_q_rinv;
    tp.bm_rinv = bm.rinv;
    tp.bm_tomb = bm.tomb;
    tp.stats = reinterpret_cast<u64*>(ws.counters.p + 4);
    tp.gthr = ws.gthr.p;
    tp.top_k = top_k;
    tp.nst = nst;
    tp.qcap = qcap;
    tp.kr = kr;
    const CUtensorMap& tmap = *reinterpret_cast<const CUtensorMap*>(bm.tmap3);
    const int grid = sms;
    if (!ws.ev0) {
        ZB_CUDA(cudaEventCreate(&ws.ev0));
        ZB_CUDA(cudaEventCreate(&ws.ev1));
    }
    ZB_CUDA(cudaEventRecord(ws.ev0, s));
    auto launch = [&](auto kern, int threads) {
        ZB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, threads, smem, s>>>(tmap, f, tp);
    };
    // short lists (n' <= 32): 4 math warps per team x 16 rows;  long lists (top-100): 8 x 8 rows -- sixteen warps keep the lists (measured, T3Shape)
    if (filt) launch(tile_scan3_kernel<3, 1, 4>, T3Shape<4>::THREADS);
    else if (kr == 1) {
        if (metric == 0) launch(tile_scan3_kernel<0, 1, 4>, T3Shape<4>::THREADS);
        else if (metric == 1) launch(tile_scan3_kernel<1, 1, 4>, T3Shape<4>::THREADS);
        else launch(tile_scan3_kernel<2, 1, 4>, T3Shape<4>::THREADS);
    } else if (ws.long_list_warps == 4) {   // knob long_list_warps (ablation)
        if (metric == 0) launch(tile_scan3_kernel<0, T3_KR_MAX, 4>, T3Shape<4>::THREADS);
        else if (metric == 1) launch(tile_scan3_kernel<1, T3_KR_MAX, 4>, T3Shape<4>::THREADS);
        else launch(tile_scan3_kernel<2, T3_KR_MAX, 4>, T3Shape<4>::THREADS);
    } else {
        if (metric == 0) launch(tile_scan3_kernel<0, T3_KR_MAX, 8>, T3Shape<8>::THREADS);
        else if (metric == 1) launch(tile_scan3_kernel<1, T3_KR_MAX, 8>, T3Shape<8>::THREADS);
        else launch(tile_scan3_kernel<2, T3_KR_MAX, 8>, T3Shape<8>::THREADS);
    }
    ZB_CUDA(cudaGetLastError());
    ZB_CUDA(cudaEventRecord(ws.ev1, s));
    ws.launched = true;
    ws.launches = 7;
    if (filt) {
        T3RefineParams rp{};
        rp.bm_rows = bm.rows;
        rp.bm_tomb = bm.tomb;
        rp.queries = d_q;
        rp.order = ws.order.p;
        rp.nvisits = nvisits;
        rp.v_leaf = v_leaf;
        rp.v_np = v_np;
        rp.v_q = v_q;
        rp.v_ent_off = v_ent_off;
        rp.cand = ws.cand.p;
        rp.cand_cut = ws.cand_cut.p;
        rp.cand_flag = ws.cand_flag.p;
        rp.gthr = ws.gthr.p;
        rp.q_n2 = ws.q_n2.p;
        rp.leaf_n2max = bm.leaf_n2max;
        rp.ecoef = tp.ecoef;
        rp.entries = entries;
        rp.work_counter = ws.counters.p + 1;
        rp.stats = tp.stats;
        const int rgrid = sms * 6;   // 48 warps per SM: the pass is a latency-bound gather of ~10 rows per visit
        if (metric == 1) refine_visits_kernel<1><<<rgrid, RF_THREADS, 0, s>>>(f, rp);
        else refine_visits_kernel<2><<<rgrid, RF_THREADS, 0, s>>>(f, rp);
        ZB_CUDA(cudaGetLastError());
        if (!ws.ev2) ZB_CUDA(cudaEventCreate(&ws.ev2));
        ZB_CUDA(cudaEventRecord(ws.ev2, s));
        ws.launches = 9;   // + the queries' norms and the second pass
    }
}

// ---- flat-table projection on the third-generation skeleton (t3_body MODE 1) ----
// tiles = (range of `range_rows` input rows, <= qcap planes); tile t = range t / npt, plane tile t % npt, so the plane
// tiles of one row range are handed out back to back and meet the range's rows in L2.
__global__ void pj_tiles_kernel(u32 nranges, u32 npt, u32 range_rows, u64 n, u32 H, u32 tq, long long* __restrict__ leaf_off,
                                u32* __restrict__ leaf_len, u32* __restrict__ tile_leaf, u32* __restrict__ tile_first,
                                u32* __restrict__ tile_count, u32* __restrict__ ntiles) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *ntiles = nranges * npt;
    if (i < nranges) {
        leaf_off[i] = (long long)i * range_rows;
        const u64 left = n - (u64)i * range_rows;
        leaf_len[i] = left < range_rows ? (u32)left : range_rows;
    }
    if (i < nranges * npt) {
        const u32 r = i / npt, p = i - r * npt;
        tile_leaf[i] = r;
        tile_first[i] = p * tq;
        tile_count[i] = H - p * tq < tq ? H - p * tq : tq;
    }
}
bool project3_supported(int dimp) {
    int nst, qcap;
    return t3_config(dimp, 1, &nst, &qcap);
}
// sign[n][Hp] = Hyperplane::point_is_above (lsh.rs:39-43) of every (row, plane); rows = [n][dimp] f32, 16-byte aligned.
void project3(ScanWorkspace& ws, const float* d_rows, u64 n, const float* d_coef, const float* d_cst, int H, int dimp, u8* d_sign, int Hp,
              cudaStream_t s) {
    int nst = 0, qcap = 0;
    if (!n || !H) return;
    ZB_REQUIRE(t3_config(dimp, 1, &nst, &qcap), ZB_ERR_STATE, "project3: rows of %d floats do not fit the tile kernel", dimp);
    ZB_REQUIRE(n < (1ull << 31), ZB_ERR_INVALID, "project3: too many rows in one call");
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const u32 tq = (u32)qcap;
    const u32 npt = ((u32)H + tq - 1) / tq;
    // enough tiles for every team several times over, ranges a multiple of the 64-row stage
    u32 range_rows = 2048;
    while (range_rows > 64 && (n + range_rows - 1) / range_rows * npt < (u64)sms * T3_TEAMS * 8) range_rows >>= 1;
    const u32 nranges = (u32)((n + range_rows - 1) / range_rows);
    const u64 nt = (u64)nranges * npt;
    ZB_REQUIRE(nt < (1ull << 31), ZB_ERR_INVALID, "project3: too many tiles");
    ws.pj_off.ensure(nranges);
    ws.leaf_count.ensure(nranges);   // leaf_len of the ranges
    ws.tile_leaf.ensure(nt);
    ws.tile_first.ensure(nt);
    ws.tile_cnt.ensure(nt);
    ws.counters.ensure(64);
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    pj_tiles_kernel<<<(u32)((nt + 255) / 256), 256, 0, s>>>(nranges, npt, range_rows, n, (u32)H, tq, ws.pj_off.p, ws.leaf_count.p,
                                                           ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p, ws.counters.p + 2);
    alignas(64) CUtensorMap tmap;
    make_row_tile_map(&tmap, d_rows, n, dimp, T3_RB, T3_SLICE_FLOATS);
    ForestView f{};
    f.leaf_off = ws.pj_off.p;
    f.leaf_len = ws.leaf_count.p;
    f.dimp = dimp;
    f.dim = dimp;
    f.chunks = dimp / 16;
    T3Params tp{};
    tp.tile_leaf = ws.tile_leaf.p;
    tp.tile_first = ws.tile_first.p;
    tp.tile_count = ws.tile_cnt.p;
    tp.ntiles = ws.counters.p + 2;
    tp.tile_counter = ws.counters.p;
    tp.queries = d_coef;
    tp.stats = reinterpret_cast<u64*>(ws.counters.p + 4);
    tp.nst = nst;
    tp.qcap = qcap;
    tp.kr = 1;
    tp.pj_cst = d_cst;
    tp.pj_sign = d_sign;
    tp.pj_hp = Hp;
    const size_t smem = t3_smem_bytes(nst, dimp, qcap, 1);
    ZB_CUDA(cudaFuncSetAttribute(project3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    project3_kernel<<<sms, T3Shape<4>::THREADS, smem, s>>>(tmap, f, tp);
    ZB_CUDA(cudaGetLastError());
}

// ---- exact mode: every (row range, query) pair of a plain store is a visit with n' = top_k ----
// Visit v = q * nranges + r (query-major: query q's visits are woff[q] .. woff[q + 1], its entries v * top_k ..); tile t = range
// t / ntq, query tile t % ntq, the queries of a range spread evenly over its ntq tiles (order is range-major).
__global__ void ex_visits_kernel(u32 nranges, u32 nq, u32 ntq, u32 range_rows, u64 n, u32 top_k, long long* __restrict__ leaf_off,
                                 u32* __restrict__ leaf_len, u32* __restrict__ v_leaf, u32* __restrict__ v_np, u32* __restrict__ v_q,
                                 u32* __restrict__ order, u32* __restrict__ ent_off, u32* __restrict__ woff, u32* __restrict__ tile_leaf,
                                 u32* __restrict__ tile_first, u32* __restrict__ tile_count, u32* __restrict__ counters) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 nv = (u64)nranges * nq, nt = (u64)nranges * ntq;
    if (i == 0) {
        counters[2] = (u32)nt;   // tiles
        counters[3] = (u32)nv;   // visits (the filter's second pass)
    }
    if (i < nranges) {
        leaf_off[i] = (long long)i * range_rows;
        const u64 left = n - i * range_rows;
        leaf_len[i] = left < range_rows ? (u32)left : range_rows;
    }
    if (i < nv) {
        const u32 q = (u32)(i / nranges), r = (u32)(i - (u64)q * nranges);
        v_leaf[i] = r;
        v_np[i] = top_k;
        v_q[i] = q;
        order[(u64)r * nq + q] = (u32)i;
    }
    if (i <= nv) ent_off[i] = (u32)(i * top_k);
    if (i <= nq) woff[i] = (u32)(i * nranges);
    if (i < nt) {
        const u32 r = (u32)(i / ntq), j = (u32)(i - (u64)r * ntq);
        const u32 per = nq / ntq, extra = nq - per * ntq;
        tile_leaf[i] = r;
        tile_first[i] = r * nq + j * per + (j < extra ? j : extra);
        tile_count[i] = per + (j < extra ? 1u : 0u);
    }
}

static u64 ex_visit_bytes(u32 top_k, bool l2_filter) {
    // v_leaf, v_np, v_q, ent_off, order + a tile's three words + the list; the filter's 32 candidates, cutoff and flag
    return 5 * 4 + 3 * 4 + (u64)top_k * sizeof(Entry) + (l2_filter ? (u64)T3_KL * 8 + 4 + 1 : 0);
}

ExactPlan exact_plan(u64 n, u64 nq, int dimp, u32 top_k, bool l2_filter, u64 per_query_bytes, u64 budget_bytes) {
    ExactPlan p;
    int nst = 0, qcap = 0;
    ZB_REQUIRE(t3_config(dimp, t3_kr(top_k), &nst, &qcap), ZB_ERR_INVALID, "exact search: rows of %d floats do not fit the tile kernel", dimp);
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const u64 vb = ex_visit_bytes(top_k, l2_filter);
    n = n ? n : 1;
    auto nranges = [&](u64 rr) { return (n + rr - 1) / rr; };
    auto chunk = [&](u64 rr) { return std::max<u64>(1, budget_bytes / (nranges(rr) * vb + per_query_bytes + 16)); };
    // longest ranges that still give every team several tiles (like project3); long ranges keep the visit count small
    u64 rr = 4096;
    while (rr > 64 && nranges(rr) * ((std::min(nq, chunk(rr)) + qcap - 1) / qcap) < (u64)sms * T3_TEAMS * 8) rr >>= 1;
    // one query's visits must fit the budget
    while (nranges(rr) * vb + per_query_bytes > budget_bytes && rr < (1ull << 24)) rr <<= 1;
    p.range_rows = (u32)rr;
    p.chunk = std::min<u64>(chunk(rr), nq ? nq : 1);
    ZB_REQUIRE(nranges(rr) * p.chunk < (1ull << 31) && nranges(rr) * p.chunk * top_k < (1ull << 32), ZB_ERR_INVALID,
               "exact search: too many visits in one chunk");
    return p;
}

__global__ void ex_empty_kernel(u32 nq, u32 top_k, u64* __restrict__ out_ord, u64* __restrict__ out_bits, u32* __restrict__ out_counts) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (u64)nq * top_k) out_ord[i] = out_bits[i] = ZB_SENTINEL;
    if (i < nq) out_counts[i] = 0;
}

void exact_scan3(ScanWorkspace& ws, const ForestView& store, const BucketMajor& bm, u64 n, u32 metric, const float* d_q, u32 nq,
                 u32 range_rows, u32 top_k, bool l2_filter, u64* out_ord, u64* out_bits, u32* out_counts, cudaStream_t s) {
    ws.launched = false;
    ws.filtered = false;
    if (!nq || !top_k) return;
    if (!n) {
        const u64 tot = std::max<u64>((u64)nq * top_k, nq);
        ex_empty_kernel<<<(u32)((tot + 255) / 256), 256, 0, s>>>(nq, top_k, out_ord, out_bits, out_counts);
        ZB_CUDA(cudaGetLastError());
        return;
    }
    int nst = 0, qcap = 0;
    const int kr = t3_kr(top_k);
    ZB_REQUIRE(metric <= 2 && top_k <= T3_KL * T3_KR_MAX && t3_config(store.dimp, kr, &nst, &qcap), ZB_ERR_INVALID,
               "exact search: no fused-kernel configuration for metric %u, top_k %u, %d floats", metric, top_k, store.dimp);
    ZB_REQUIRE(n < (1ull << 31) && range_rows % T3_RB == 0, ZB_ERR_INVALID, "exact search: %llu rows in ranges of %u",
               (unsigned long long)n, range_rows);
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const u32 nranges = (u32)((n + range_rows - 1) / range_rows);
    const u32 ntq = (nq + (u32)qcap - 1) / (u32)qcap;
    const u64 nv = (u64)nranges * nq, nt = (u64)nranges * ntq;
    ZB_REQUIRE(nv < (1ull << 31) && nv * top_k < (1ull << 32), ZB_ERR_INVALID, "exact search: too many visits in one call");
    ws.pj_off.ensure(nranges);
    ws.leaf_count.ensure(nranges);   // leaf_len of the ranges
    ws.ex_leaf.ensure(nv);
    ws.ex_np.ensure(nv);
    ws.ex_q.ensure(nv);
    ws.order.ensure(nv);
    ws.ex_ent_off.ensure(nv + 1);
    ws.ex_woff.ensure((u64)nq + 1);
    ws.tile_leaf.ensure(nt);
    ws.tile_first.ensure(nt);
    ws.tile_cnt.ensure(nt);
    ws.ex_entries.ensure(nv * top_k);
    ws.counters.ensure(64);
    ws.gthr.ensure(nq);
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.gthr.p, 0xFF, (size_t)nq * 8, s));
    ex_visits_kernel<<<(u32)((nv + 1 + 255) / 256), 256, 0, s>>>(nranges, nq, ntq, range_rows, n, top_k, ws.pj_off.p, ws.leaf_count.p,
                                                                ws.ex_leaf.p, ws.ex_np.p, ws.ex_q.p, ws.order.p, ws.ex_ent_off.p,
                                                                ws.ex_woff.p, ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p,
                                                                ws.counters.p);
    ZB_CUDA(cudaGetLastError());
    ForestView f = store;
    f.leaf_off = ws.pj_off.p;
    f.leaf_len = ws.leaf_count.p;
    f.num_trees = 1;
    BucketMajor b = bm;
    const double* q_rinv = nullptr;
    if (metric == 0) {
        ws.ex_q_rinv.ensure(nq);
        launch_rinv(d_q, nq, f.dimp, ws.ex_q_rinv.p, s);
        q_rinv = ws.ex_q_rinv.p;
    }
    ws.l2_filter = l2_filter && (metric == 1 || metric == 2) && bm.n2;
    if (ws.l2_filter) {   // the filter's error bound per range
        ws.ex_n2max.ensure(nranges);
        launch_leaf_n2max(nranges, ws.pj_off.p, ws.leaf_count.p, bm.n2, ws.ex_n2max.p, s);
        b.leaf_n2max = ws.ex_n2max.p;
    }
    t3_launch(ws, f, b, metric, d_q, q_rinv, nq, (u32)nv, ws.ex_leaf.p, ws.ex_np.p, ws.ex_q.p, ws.ex_ent_off.p, ws.ex_entries.p, top_k, kr,
              nst, qcap, sms, ws.counters.p + 2, ws.counters.p + 3, s);
    launch_merge_queries(nq, 1, ws.ex_woff.p, ws.ex_ent_off.p, ws.ex_entries.p, top_k, out_ord, out_bits, out_counts, s);
}

// =====================================================================================================
// Leaf-tile scan for the SCALAR metrics (distance.rs:51-190, zb_metrics.cuh) -- SURVEY 8(f) row 3.
// A sequential f32 fold per pair cannot be split inside the pair, so one thread owns (row, the <= 8 queries of the
// tile): the row element is loaded ONCE (128-bit __ldg) and folded into one accumulator per query, the queries sit in
// shared memory and are read as broadcasts.  Visits are grouped by leaf exactly like the fused kernel's tiles, so a
// leaf's rows cross HBM once per tile instead of once per visit (config 2: 27 GB instead of 173 GB per batch).  Keys go
// to the gather path's pair_key layout ([visit][member]); the per-visit top-n' stays with select_visits_kernel.
// =====================================================================================================
#define SQ_THREADS 256
#define SQ_TQ 8
#define SQ_CTAS_PER_SM 4

__global__ void sq_count_kernel(u32 nv, const u32* __restrict__ v_leaf, const u64* __restrict__ v_pair_off, u32* __restrict__ leaf_count) {
    u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    if (v_pair_off[v + 1] > v_pair_off[v]) atomicAdd(&leaf_count[v_leaf[v]], 1u);  // visits with pairs to score
}
__global__ void sq_scatter_kernel(u32 nv, const u32* __restrict__ v_leaf, const u64* __restrict__ v_pair_off,
                                  const u32* __restrict__ leaf_start, u32* __restrict__ leaf_cursor, u32* __restrict__ order) {
    u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    if (v_pair_off[v + 1] > v_pair_off[v]) {
        const u32 leaf = v_leaf[v];
        order[leaf_start[leaf] + atomicAdd(&leaf_cursor[leaf], 1u)] = v;
    }
}

struct SeqTileParams {
    const u32* tile_leaf;
    const u32* tile_first;
    const u32* tile_count;
    const u32* ntiles;
    u32* tile_counter;
    const u32* order;
    const u32* v_q;
    const u64* v_pair_off;
    u64* pair_key;
    const float* queries;
    u64* stats;  // [0] visits, [1] pairs, [2] bytes asked of HBM by design
    int power;
    int pf_lines;  // L2 prefetch distance in 128-byte lines of the row (0 = off)
};

template <int CODE, int NQ>
__device__ __forceinline__ void seq_tile_rows(const ForestView& f, const SeqTileParams& tp, const float* __restrict__ s_q,
                                              const u64* __restrict__ s_pbase, u32 c, u32 leaf) {
    const u32 len = f.leaf_len[leaf];
    const long long off = f.leaf_off[leaf];
    const int n4 = f.dim >> 2, q4 = f.dimp >> 2;
    const int n8 = n4 >> 1;  // groups of two float4 = one 32-byte sector of the row
    const int pf = tp.pf_lines * 8;  // prefetch distance in float4
    const float4* q = reinterpret_cast<const float4*>(s_q);
    for (u32 r = threadIdx.x; r < len; r += SQ_THREADS) {
        const u32 slot = f.members[off + r];
        if (tomb_test(f.tomb, slot)) {
#pragma unroll
            for (int j = 0; j < NQ; ++j)
                if ((u32)j < c) tp.pair_key[s_pbase[j] + r] = ZB_SENTINEL;
            continue;
        }
        SeqAcc st[NQ];
#pragma unroll
        for (int j = 0; j < NQ; ++j) seq_init(st[j]);
        const float* row = f.rows + (size_t)slot * f.dimp;
        const float4* a = reinterpret_cast<const float4*>(row);
        // software pipeline: the next sector of the row is in flight while this one is folded into the NQ accumulators
        // (the profile of the first version was 56 % long-scoreboard stalls on the row loads, issue slots 24 % busy)
        float4 c0 = make_float4(0.f, 0.f, 0.f, 0.f), c1 = c0;
        if (n8 > 0) { c0 = __ldg(a); c1 = __ldg(a + 1); }
#pragma unroll 1
        for (int g = 0; g < n8; ++g) {
            float4 x0 = c0, x1 = c1;
            if (g + 1 < n8) { c0 = __ldg(a + 2 * g + 2); c1 = __ldg(a + 2 * g + 3); }
            // one prefetch per 128-byte line, pf_lines lines ahead: the line waits in L2 when its loads are issued, so
            // the row stream is bounded by L2 latency, not by DRAM latency x the registers a deeper pipeline would need
            if (pf != 0 && (g & 3) == 0 && 2 * g + pf < n4) asm volatile("prefetch.global.L2 [%0];" ::"l"(a + 2 * g + pf));
#pragma unroll
            for (int j = 0; j < NQ; ++j) {
                const float4 b0 = q[j * q4 + 2 * g], b1 = q[j * q4 + 2 * g + 1];  // same address across the warp: broadcasts
                seq_step<CODE>(st[j], x0.x, b0.x, tp.power);
                seq_step<CODE>(st[j], x0.y, b0.y, tp.power);
                seq_step<CODE>(st[j], x0.z, b0.z, tp.power);
                seq_step<CODE>(st[j], x0.w, b0.w, tp.power);
                seq_step<CODE>(st[j], x1.x, b1.x, tp.power);
                seq_step<CODE>(st[j], x1.y, b1.y, tp.power);
                seq_step<CODE>(st[j], x1.z, b1.z, tp.power);
                seq_step<CODE>(st[j], x1.w, b1.w, tp.power);
            }
        }
        for (int i = n8 * 2; i < n4; ++i) {  // an odd float4 left over
            const float4 av = __ldg(a + i);
#pragma unroll
            for (int j = 0; j < NQ; ++j) {
                const float4 bv = q[j * q4 + i];
                seq_step<CODE>(st[j], av.x, bv.x, tp.power);
                seq_step<CODE>(st[j], av.y, bv.y, tp.power);
                seq_step<CODE>(st[j], av.z, bv.z, tp.power);
                seq_step<CODE>(st[j], av.w, bv.w, tp.power);
            }
        }
        for (int i = n4 * 4; i < f.dim; ++i) {  // dim % 4 tail (never the padding)
            const float x = __ldg(row + i);
#pragma unroll
            for (int j = 0; j < NQ; ++j) seq_step<CODE>(st[j], x, s_q[j * f.dimp + i], tp.power);
        }
#pragma unroll
        for (int j = 0; j < NQ; ++j)
            if ((u32)j < c) tp.pair_key[s_pbase[j] + r] = seq_finish<CODE>(st[j], tp.power);
    }
}

template <int CODE>
__global__ void __launch_bounds__(SQ_THREADS, SQ_CTAS_PER_SM) seq_tile_kernel(ForestView f, SeqTileParams tp) {
    extern __shared__ __align__(16) float s_q[];  // [SQ_TQ][dimp]
    __shared__ u32 s_tile;
    __shared__ u32 s_v[SQ_TQ];
    __shared__ u64 s_pbase[SQ_TQ];  // where each visit's keys start in pair_key
    const u32 ntiles = *tp.ntiles;
    const int q4 = f.dimp >> 2;
    for (;;) {
        __syncthreads();  // the previous tile's queries are no longer read
        if (threadIdx.x == 0) s_tile = atomicAdd(tp.tile_counter, 1u);
        __syncthreads();
        const u32 tile = s_tile;
        if (tile >= ntiles) break;
        const u32 leaf = tp.tile_leaf[tile], first = tp.tile_first[tile], c = tp.tile_count[tile];
        if (threadIdx.x < SQ_TQ) {
            const u32 v = tp.order[first + (threadIdx.x < c ? threadIdx.x : 0u)];
            s_v[threadIdx.x] = v;
            s_pbase[threadIdx.x] = tp.v_pair_off[v];
        }
        __syncthreads();
        const u32 nqp = c <= 1 ? 1u : (c <= 2 ? 2u : (c <= 4 ? 4u : 8u));  // query slots the row loop folds
        for (u32 idx = threadIdx.x; idx < nqp * (u32)q4; idx += SQ_THREADS) {
            const u32 j = idx / (u32)q4, k = idx - j * (u32)q4;
            reinterpret_cast<float4*>(s_q)[idx] =
                j < c ? __ldg(reinterpret_cast<const float4*>(tp.queries + (size_t)tp.v_q[s_v[j]] * f.dimp) + k)
                      : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        if (nqp == 1) seq_tile_rows<CODE, 1>(f, tp, s_q, s_pbase, c, leaf);
        else if (nqp == 2) seq_tile_rows<CODE, 2>(f, tp, s_q, s_pbase, c, leaf);
        else if (nqp == 4) seq_tile_rows<CODE, 4>(f, tp, s_q, s_pbase, c, leaf);
        else seq_tile_rows<CODE, 8>(f, tp, s_q, s_pbase, c, leaf);
        if (threadIdx.x == 0) {
            const u64 len = f.leaf_len[leaf];
            atomicAdd(&tp.stats[0], (u64)c);
            atomicAdd(&tp.stats[1], len * c);
            atomicAdd(&tp.stats[2], (len + c) * 4ull * (u64)f.dim);
        }
    }
}

bool seq_tile_scan_supported(int dimp) { return (size_t)SQ_TQ * dimp * 4 <= 96 * 1024; }

void seq_tile_scan(ScanWorkspace& ws, const ForestView& f, u32 metric, int power, const float* d_q, u32 nv, const u32* v_leaf,
                   const u32* v_q, const u64* v_pair_off, u64* pair_key, u32 nleaves, int prefetch_lines, cudaStream_t s) {
    ws.seq_launched = false;
    if (!nv || !nleaves || metric <= M_L2 || !seq_tile_scan_supported(f.dimp)) return;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    ws.leaf_count.ensure(nleaves + 1);
    ws.leaf_start.ensure(nleaves + 1);
    ws.leaf_cursor.ensure(nleaves + 1);
    ws.tile_per_leaf.ensure(nleaves + 1);
    ws.tile_start.ensure(nleaves + 1);
    ws.order.ensure(nv);
    ws.tile_leaf.ensure(nv);
    ws.tile_first.ensure(nv);
    ws.tile_cnt.ensure(nv);
    ws.counters.ensure(64);
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const u32*)nullptr, (u32*)nullptr, (long long)(nleaves + 1));
    ws.tmp.ensure(tmp_bytes + 256);
    ZB_CUDA(cudaMemsetAsync(ws.leaf_count.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.leaf_cursor.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    sq_count_kernel<<<(nv + 255) / 256, 256, 0, s>>>(nv, v_leaf, v_pair_off, ws.leaf_count.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.leaf_count.p, ws.leaf_start.p, (long long)(nleaves + 1), s);
    sq_scatter_kernel<<<(nv + 255) / 256, 256, 0, s>>>(nv, v_leaf, v_pair_off, ws.leaf_start.p, ws.leaf_cursor.p, ws.order.p);
    ts_tilecount_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, SQ_TQ, ws.tile_per_leaf.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
    ts_filltiles_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, ws.leaf_start.p, ws.tile_start.p, SQ_TQ,
                                                              ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p, f.leaf_len,
                                                              (u64)f.dim * 4ull, reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    SeqTileParams tp;
    tp.tile_leaf = ws.tile_leaf.p;
    tp.tile_first = ws.tile_first.p;
    tp.tile_count = ws.tile_cnt.p;
    tp.ntiles = ws.tile_start.p + nleaves;
    ws.ntiles_ptr = tp.ntiles;
    tp.tile_counter = ws.counters.p;
    tp.order = ws.order.p;
    tp.v_q = v_q;
    tp.v_pair_off = v_pair_off;
    tp.pair_key = pair_key;
    tp.queries = d_q;
    tp.stats = reinterpret_cast<u64*>(ws.counters.p + 4);
    tp.power = power;
    tp.pf_lines = prefetch_lines < 0 ? 0 : (prefetch_lines > 64 ? 64 : prefetch_lines);
    // the opt-in is set whatever the size: the kernel's static shared memory counts against the 48 KB default too, so rows of
    // 1536 floats (exactly 48 KB of queries) failed to launch without it
    const size_t smem = (size_t)SQ_TQ * f.dimp * 4;
    const int grid = sms * SQ_CTAS_PER_SM;
    if (!ws.ev0) {
        ZB_CUDA(cudaEventCreate(&ws.ev0));
        ZB_CUDA(cudaEventCreate(&ws.ev1));
    }
    ZB_CUDA(cudaEventRecord(ws.ev0, s));
#define ZB_SQ_CALL(C)                                                                                                        \
    do {                                                                                                                     \
        ZB_CUDA(cudaFuncSetAttribute(seq_tile_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));            \
        seq_tile_kernel<C><<<grid, SQ_THREADS, smem, s>>>(f, tp);                                                            \
    } while (0)
    switch (metric) {
        case M_CHEBYSHEV: ZB_SQ_CALL(M_CHEBYSHEV); break;
        case M_CANBERRA: ZB_SQ_CALL(M_CANBERRA); break;
        case M_BRAY_CURTIS: ZB_SQ_CALL(M_BRAY_CURTIS); break;
        case M_MANHATTAN: ZB_SQ_CALL(M_MANHATTAN); break;
        case M_L3: ZB_SQ_CALL(M_L3); break;
        case M_L4: ZB_SQ_CALL(M_L4); break;
        case M_HAMMING: ZB_SQ_CALL(M_HAMMING); break;
        case M_MINKOWSKI: ZB_SQ_CALL(M_MINKOWSKI); break;
        default: ZB_SQ_CALL(M_PNORM); break;
    }
#undef ZB_SQ_CALL
    ZB_CUDA(cudaGetLastError());
    ZB_CUDA(cudaEventRecord(ws.ev1, s));
    ws.seq_launched = true;
}

// Statistics of the last seq_tile_scan launch; call after the stream has been synchronised.
void seq_tile_scan_stats(ScanWorkspace& ws, cudaStream_t s, u64* moved_bytes, float* kernel_ms, u32* tiles) {
    *moved_bytes = 0;
    *kernel_ms = 0.f;
    *tiles = 0;
    if (!ws.seq_launched) return;
    u64 h[4] = {0, 0, 0, 0};
    ZB_CUDA(cudaMemcpyAsync(h, reinterpret_cast<u64*>(ws.counters.p + 4), 32, cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaMemcpyAsync(tiles, ws.ntiles_ptr, 4, cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaStreamSynchronize(s));
    cudaEventElapsedTime(kernel_ms, ws.ev0, ws.ev1);
    *moved_bytes = h[2];
}

// =====================================================================================================
// Keys-only leaf-tile scan for cosine / L2 (zb_quadtile.cuh): the visits the fused kernel does not take (n' > 32, e.g.
// BASELINE config 5's top-100) grouped by leaf into (leaf, <= 8 queries) tiles; a quad scores 4 rows x 4 queries per pass
// in the canonical order and writes the keys into the gather path's pair_key layout; select_visits_kernel keeps each
// visit's top-n'.  Rows cross HBM once per tile instead of once per pair.  Knob quad_tile (default 0 until measured).
// =====================================================================================================
}  // namespace zb
#include "zb_quadtile_kernel.cuh"
namespace zb {

bool quad_tile_scan_supported(int dimp) { return (size_t)8 * dimp * 4 <= 96 * 1024; }

void quad_tile_scan(ScanWorkspace& ws, const ForestView& f, u32 metric, const float* d_q, u32 nv, const u32* v_leaf, const u32* v_q,
                    const u64* v_pair_off, u64* pair_key, u32 nleaves, cudaStream_t s) {
    ws.seq_launched = false;
    if (!nv || !nleaves || metric > M_L2 || !quad_tile_scan_supported(f.dimp)) return;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    ws.leaf_count.ensure(nleaves + 1);
    ws.leaf_start.ensure(nleaves + 1);
    ws.leaf_cursor.ensure(nleaves + 1);
    ws.tile_per_leaf.ensure(nleaves + 1);
    ws.tile_start.ensure(nleaves + 1);
    ws.order.ensure(nv);
    ws.tile_leaf.ensure(nv);
    ws.tile_first.ensure(nv);
    ws.tile_cnt.ensure(nv);
    ws.counters.ensure(64);
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const u32*)nullptr, (u32*)nullptr, (long long)(nleaves + 1));
    ws.tmp.ensure(tmp_bytes + 256);
    ZB_CUDA(cudaMemsetAsync(ws.leaf_count.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.leaf_cursor.p, 0, (size_t)(nleaves + 1) * 4, s));
    ZB_CUDA(cudaMemsetAsync(ws.counters.p, 0, 64 * 4, s));
    sq_count_kernel<<<(nv + 255) / 256, 256, 0, s>>>(nv, v_leaf, v_pair_off, ws.leaf_count.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.leaf_count.p, ws.leaf_start.p, (long long)(nleaves + 1), s);
    sq_scatter_kernel<<<(nv + 255) / 256, 256, 0, s>>>(nv, v_leaf, v_pair_off, ws.leaf_start.p, ws.leaf_cursor.p, ws.order.p);
    ts_tilecount_kernel<<<(nleaves + 256) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, 8, ws.tile_per_leaf.p);
    cub::DeviceScan::ExclusiveSum(ws.tmp.p, tmp_bytes, ws.tile_per_leaf.p, ws.tile_start.p, (long long)(nleaves + 1), s);
    ts_filltiles_kernel<<<(nleaves + 255) / 256, 256, 0, s>>>(nleaves, ws.leaf_count.p, ws.leaf_start.p, ws.tile_start.p, 8,
                                                              ws.tile_leaf.p, ws.tile_first.p, ws.tile_cnt.p, f.leaf_len,
                                                              (u64)f.dim * 4ull, reinterpret_cast<u64*>(ws.counters.p + 4) + 3);
    QuadTileParams tp;
    tp.tile_leaf = ws.tile_leaf.p;
    tp.tile_first = ws.tile_first.p;
    tp.tile_count = ws.tile_cnt.p;
    tp.ntiles = ws.tile_start.p + nleaves;
    ws.ntiles_ptr = tp.ntiles;
    tp.tile_counter = ws.counters.p;
    tp.order = ws.order.p;
    tp.v_q = v_q;
    tp.v_pair_off = v_pair_off;
    tp.pair_key = pair_key;
    tp.queries = d_q;
    tp.stats = reinterpret_cast<u64*>(ws.counters.p + 4);
    const size_t smem = (size_t)8 * f.dimp * 4;   // opt-in set whatever the size, as for seq_tile_kernel (static shared memory)
    const int grid = sms * 2;
    if (!ws.ev0) {
        ZB_CUDA(cudaEventCreate(&ws.ev0));
        ZB_CUDA(cudaEventCreate(&ws.ev1));
    }
    ZB_CUDA(cudaEventRecord(ws.ev0, s));
#define ZB_QT_CALL(M)                                                                                                    \
    do {                                                                                                                 \
        ZB_CUDA(cudaFuncSetAttribute(quad_tile_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));       \
        quad_tile_kernel<M><<<grid, QT_THREADS, smem, s>>>(f, tp);                                                       \
    } while (0)
    if (metric == 0) ZB_QT_CALL(0);
    else if (metric == 1) ZB_QT_CALL(1);
    else ZB_QT_CALL(2);
#undef ZB_QT_CALL
    ZB_CUDA(cudaGetLastError());
    ZB_CUDA(cudaEventRecord(ws.ev1, s));
    ws.seq_launched = true;  // the same stats reader as the scalar-metric scan (seq_tile_scan_stats)
}

}  // namespace zb
