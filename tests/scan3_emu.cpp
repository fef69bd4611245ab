// scan3_emu.cpp -- TEST INFRASTRUCTURE.  Runs the SOURCE of the third-generation fused leaf-tile scan
// (zebra_b200/csrc/zb_scan3_kernel.cuh, t3_body) on the CPU: one std::thread per CUDA thread of a 384-thread block;
// warp shuffles / ballots = exchanges through a per-warp mailbox, named barriers = std::barrier, mbarriers = counters with the
// PTX phase / transaction-count semantics, TMA tensor copies and 1-D bulk copies = memcpy performed LATER by a separate
// "copy engine" thread (so a consumer that does not wait for its full barrier reads stale data and fails the test), packed
// f32x2 arithmetic = two IEEE operations (build with -ffp-contract=off).  Blocks run one after the other, which is a legal
// schedule of the persistent kernel.  tests/test_scan3.py feeds it leaves, tombstones and visits and compares every
// entry the kernel writes with the oracle.
#include <math.h>
#include <stdio.h>
#include <execinfo.h>
#include <signal.h>
#include <unistd.h>
#include <cmath>
#include <stdlib.h>
#include <stdint.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <barrier>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <random>
#include <thread>
#include <unordered_map>
#include <algorithm>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
struct Dim3 { unsigned x, y, z; };
static thread_local Dim3 emu_threadIdx;
#define threadIdx emu_threadIdx

// A crash inside the emulation (abort of a protocol check, a C++ exception in a thread) says where it came from.
static void emu_abort_handler(int sig) {
    void* frames[48];
    const int n = backtrace(frames, 48);
    const char msg[] = "[scan3_emu] fatal signal, backtrace:\n";
    (void)!write(2, msg, sizeof msg - 1);
    backtrace_symbols_fd(frames, n, 2);
    signal(sig, SIG_DFL);
    raise(sig);
}
static const int emu_handler_installed = (signal(SIGABRT, emu_abort_handler), signal(SIGSEGV, emu_abort_handler), 0);

namespace zb {
typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned char u8;
struct Entry { u64 key, ord; };
#define ZB_SENTINEL 0xFFFFFFFFFFFFFFFFull
struct ForestView {  // the fields t3_body reads (names as in zb_kernels.cuh)
    const long long* leaf_off;
    const u32* leaf_len;
    const u32* members;
    const u64* ord;
    int dimp, chunks;
};
struct T3Map { const float* base; u64 rows; int dimp; };
}  // namespace zb
using zb::u32;
using zb::u64;

// ---------------------------------------------------------------- block-wide state of the emulation
static unsigned char* emu_smem = nullptr;
static std::barrier<>* emu_block_bar = nullptr;
static std::barrier<>* emu_team_bar[2] = {nullptr, nullptr};
struct WarpBox {
    u64 slot[32];
    std::barrier<> bar{32};
};
static std::vector<std::unique_ptr<WarpBox>> emu_warps;
// where every emulated thread currently waits (0: running; 1: mbarrier; 2: team barrier; 3: block barrier; 4: warp barrier),
// printed by the deadlock watchdog
static volatile unsigned emu_where[1024][3];
static inline void emu_at(unsigned code, unsigned a = 0, unsigned b = 0) { emu_where[threadIdx.x][0] = code; emu_where[threadIdx.x][1] = a; emu_where[threadIdx.x][2] = b; }
static void emu_dump_where(unsigned nthreads) {
    for (unsigned w = 0; w * 32 < nthreads; ++w) {
        fprintf(stderr, "[scan3_emu]   warp %2u:", w);
        for (unsigned l = 0; l < 32; ++l) {
            const unsigned t = w * 32 + l;
            if (l == 0 || emu_where[t][0] != emu_where[t - 1][0] || emu_where[t][1] != emu_where[t - 1][1])
                fprintf(stderr, " [lane %u: %u %u/%u]", l, emu_where[t][0], emu_where[t][1], emu_where[t][2]);
        }
        fprintf(stderr, "\n");
    }
}
#define __syncthreads() (emu_at(3), emu_block_bar->arrive_and_wait(), emu_at(0))
static inline void __syncwarp() { emu_at(4, 1); emu_warps[threadIdx.x >> 5]->bar.arrive_and_wait(); emu_at(0); }
static inline u64 emu_exchange(u64 v, int src) {
    WarpBox& w = *emu_warps[threadIdx.x >> 5];
    w.slot[threadIdx.x & 31] = v;
    emu_at(4, 2);
    w.bar.arrive_and_wait();
    const u64 r = w.slot[src & 31];
    w.bar.arrive_and_wait();
    emu_at(0);
    return r;
}
static inline u32 f2u(float f) { u32 u; memcpy(&u, &f, 4); return u; }
static inline float u2f(u32 u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __shfl_xor_sync(unsigned, float v, int m) { return u2f((u32)emu_exchange(f2u(v), (int)(threadIdx.x & 31) ^ m)); }
static inline u32 __shfl_sync(unsigned, u32 v, int src) { return (u32)emu_exchange(v, src); }
static inline u32 __shfl_up_sync(unsigned, u32 v, int d) {
    const int lane = threadIdx.x & 31;
    const u32 r = (u32)emu_exchange(v, lane - d < 0 ? lane : lane - d);
    return r;
}
static inline unsigned __ballot_sync(unsigned, bool p) {
    WarpBox& w = *emu_warps[threadIdx.x >> 5];
    w.slot[threadIdx.x & 31] = p ? 1 : 0;
    emu_at(4, 3);
    w.bar.arrive_and_wait();
    unsigned r = 0;
    for (int i = 0; i < 32; ++i) r |= (unsigned)w.slot[i] << i;
    w.bar.arrive_and_wait();
    emu_at(0);
    return r;
}
static inline int __ffs(unsigned m) { return m ? __builtin_ctz(m) + 1 : 0; }
static inline int __popc(unsigned m) { return __builtin_popcount(m); }
template <class T> static inline T min(T a, T b) { return a < b ? a : b; }
static inline u32 atomicAdd(u32* p, u32 v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline u64 atomicAdd(u64* p, u64 v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }

// ---------------------------------------------------------------- mbarriers (PTX semantics: arrival count + transaction bytes, phase parity)
struct MBar { u32 count = 0, pending = 0; long long tx = 0; u64 completed = 0; };
static std::mutex emu_mbar_mu;
static std::unordered_map<u32, MBar> emu_mbars;
static inline u32 smem_u32(const void* p) { return (u32)((const unsigned char*)p - emu_smem); }
static void mbar_check(MBar& b) {
    if (b.pending == 0 && b.tx == 0) { b.completed++; b.pending = b.count; }
}
static inline void mbar_init(u32 bar, u32 count) {
    std::lock_guard<std::mutex> lk(emu_mbar_mu);
    MBar b; b.count = b.pending = count;
    emu_mbars[bar] = b;
}
static inline void mbar_arrive(u32 bar) {
    std::lock_guard<std::mutex> lk(emu_mbar_mu);
    MBar& b = emu_mbars.at(bar);
    if (b.pending == 0) { fprintf(stderr, "[scan3_emu] mbarrier %u: more arrivals than expected (thread %u)\n", bar, threadIdx.x); abort(); }  // a protocol bug
    b.pending--;
    mbar_check(b);
}
static inline void mbar_arrive_expect_tx(u32 bar, u32 bytes) {
    std::lock_guard<std::mutex> lk(emu_mbar_mu);
    MBar& b = emu_mbars.at(bar);
    if (b.pending == 0) { fprintf(stderr, "[scan3_emu] mbarrier %u: expect_tx arrival beyond the count (thread %u)\n", bar, threadIdx.x); abort(); }
    b.tx += bytes;
    b.pending--;
    mbar_check(b);
}
static inline void mbar_complete_tx(u32 bar, u32 bytes) {
    std::lock_guard<std::mutex> lk(emu_mbar_mu);
    MBar& b = emu_mbars.at(bar);
    b.tx -= bytes;
    mbar_check(b);
}
static std::atomic<long long> emu_spins{0};
static inline void mbar_wait(u32 bar, u32 parity) {
    std::chrono::steady_clock::time_point t0;
    emu_at(1, bar, parity);
    for (long long n = 0;; ++n) {
        {
            std::lock_guard<std::mutex> lk(emu_mbar_mu);
            if ((emu_mbars.at(bar).completed & 1) != (parity & 1)) { emu_at(0); return; }
        }
        // deadlock watchdog by wall clock (a spin count says little with several hundred threads on a few cores)
        if (n == 1000) t0 = std::chrono::steady_clock::now();
        if (n > 1000 && (n & 0xFFFF) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::seconds(60)) {
            fprintf(stderr, "[scan3_emu] mbarrier %u parity %u: no progress for 60 s (thread %u)\n", bar, parity, threadIdx.x);
            emu_dump_where(1024);
            {
                std::lock_guard<std::mutex> lk(emu_mbar_mu);
                for (auto& kv : emu_mbars)
                    fprintf(stderr, "[scan3_emu]   mbarrier %u: count %u pending %u tx %lld completed %llu\n", kv.first, kv.second.count, kv.second.pending,
                            kv.second.tx, (unsigned long long)kv.second.completed);
            }
            abort();
        }
        std::this_thread::yield();
    }
}

// ---------------------------------------------------------------- the copy engine: copies land some time AFTER they were issued
struct CopyEngine {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::function<void()>> q;
    bool stop = false;
    std::thread th;
    std::mt19937 rng{12345};
    void start() {
        th = std::thread([this] {
            for (;;) {
                std::function<void()> job;
                {
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [this] { return stop || !q.empty(); });
                    if (q.empty()) return;
                    job = std::move(q.front());
                    q.pop_front();
                }
                if ((rng() & 3) == 0) std::this_thread::sleep_for(std::chrono::microseconds(rng() % 200));
                job();
            }
        });
    }
    void push(std::function<void()> f) {
        { std::lock_guard<std::mutex> lk(mu); q.push_back(std::move(f)); }
        cv.notify_one();
    }
    void finish() {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv.notify_one();
        th.join();
    }
};
static CopyEngine* emu_dma = nullptr;
static inline void bulk_g2s(u32 dst, const void* src, u32 bytes, u32 bar) {
    unsigned char* d = emu_smem + dst;
    emu_dma->push([=] { memcpy(d, src, bytes); mbar_complete_tx(bar, bytes); });
}

namespace zb {
#define T3_EMU_STAGE_ROWS 64
#ifndef T3_KC
#define T3_KC 3
#endif
#define T3_EMU_SLICE (T3_KC * 16)
static inline void t3_tma_2d_g2s(u32 dst, const T3Map& map, int c0, long long row, u32 bar) {
    float* d = reinterpret_cast<float*>(emu_smem + dst);
    const T3Map m = map;
    emu_dma->push([=] {
        for (int r = 0; r < T3_EMU_STAGE_ROWS; ++r)
            for (int c = 0; c < T3_EMU_SLICE; ++c) {
                const long long rr = row + r;
                const int cc = c0 + c;
                d[r * T3_EMU_SLICE + c] = (rr >= 0 && (u64)rr < m.rows && cc < m.dimp) ? m.base[(size_t)rr * m.dimp + cc] : 0.0f;  // out of bounds: zero fill
            }
        mbar_complete_tx(bar, T3_EMU_STAGE_ROWS * T3_EMU_SLICE * 4);
    });
}
static inline bool t3_isinf_pos(double x) { return isinf(x) && x > 0.0; }
static inline double t3_dmul(double a, double b) { return a * b; }
static inline double t3_dsub(double a, double b) { return a - b; }
static inline u64 t3_dbits(double x) { u64 u; memcpy(&u, &x, 8); return u; }
static inline float t3_fadd(float a, float b) { return a + b; }
static inline u32 t3_fbits(float x) { return f2u(x); }
static inline float t3_bitsf(u32 b) { return u2f(b); }
static inline float t3_fadd_ru(float a, float b) { const float r = a + b; return r == r && !std::isinf(r) ? nextafterf(r, INFINITY) : r; }   // at least as large as the device's round-up
static inline float t3_fmul_ru(float a, float b) { const float r = a * b; return r == r && !std::isinf(r) ? nextafterf(r, INFINITY) : r; }
static inline float t3_fmaf(float a, float b, float c) { return fmaf(a, b, c); }
static inline float t3_fsub(float a, float b) { return a - b; }
struct T3F4 { float x, y, z, w; };
static inline T3F4 t3_ld_f4(const float* p) { T3F4 v; memcpy(&v, p, 16); return v; }
static inline u64 t3_pk2(float lo, float hi) { return (u64)f2u(lo) | ((u64)f2u(hi) << 32); }
static inline void t3_upk2(u64 v, float& lo, float& hi) { lo = u2f((u32)v); hi = u2f((u32)(v >> 32)); }
static inline u64 t3_fma2(u64 a, u64 b, u64 c) {
    return t3_pk2(fmaf(u2f((u32)a), u2f((u32)b), u2f((u32)c)), fmaf(u2f((u32)(a >> 32)), u2f((u32)(b >> 32)), u2f((u32)(c >> 32))));
}
static inline u64 t3_sub2(u64 a, u64 b) { return t3_pk2(u2f((u32)a) - u2f((u32)b), u2f((u32)(a >> 32)) - u2f((u32)(b >> 32))); }
static inline u64 t3_ldcg_u64(const u64* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline void t3_atomic_min_u64(u64* p, u64 v) {
    u64 cur = __atomic_load_n(p, __ATOMIC_SEQ_CST);
    while (v < cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {}
}
static inline u64 t3_shfl64(u64 v, int src) { return emu_exchange(v, src); }
static inline double t3_shfl_f64(double v, int src) { u64 u; memcpy(&u, &v, 8); u = emu_exchange(u, src); double r; memcpy(&r, &u, 8); return r; }
static inline u64 t3_shfl_up64(u64 v) {
    const int lane = threadIdx.x & 31;
    return emu_exchange(v, lane == 0 ? 0 : lane - 1);
}
static inline void t3_team_sync(int team, int /*threads: the barrier objects are built for the launch's team size*/) { emu_at(2, (unsigned)team); emu_team_bar[team]->arrive_and_wait(); emu_at(0); }
static inline void t3_fence_barrier_init() {}
template <int TW> static inline void t3_setmaxnreg_dec() {}
template <int TW> static inline void t3_setmaxnreg_inc() {}
static inline void t3_prefetch_map(const T3Map&) {}
static inline void t3_prefetch_l1(const void*) {}
static inline bool t3_above_from_dot(float dot, float constant) { return (double)dot + (double)constant >= 0.0; }
static inline u64 l2sq_bits(float s) { return t3_dbits((double)s); }
static inline u64 l2_bits(float s) { return t3_dbits(sqrt((double)s)); }
}  // namespace zb

#include "../zebra_b200/csrc/zb_scan3_kernel.cuh"
static_assert(T3_EMU_SLICE == T3_SLICE_FLOATS && T3_EMU_STAGE_ROWS == T3_RB, "the emulated TMA box is the kernel's stage");
static_assert(zb::T3Shape<8>::THREADS <= 1024, "emu_where holds 1024 threads");

// Tiles are given directly (what ts_count / ts_scatter / ts_filltiles build on the device).  The bucket-major store is
// addressed by position: members = identity is supplied by the caller together with ord[position].
// math warps per team of the next emu_scan3 / emu_project3 launch (the kernel body's TW: 4 or 8)
static int emu_tw = 4;
extern "C" __attribute__((visibility("default"))) int emu_scan3_set_team_warps(int tw) {
    if (tw != 4 && tw != 8) return -1;
    emu_tw = tw;
    return 0;
}
template <int TW> static void emu_run_scan3(int metric, int kr, const zb::T3Map& map, const zb::ForestView& f, const zb::T3Params& tp) {
    if (kr == 1) {
        if (metric == 0) zb::t3_body<0, 0, 1, TW>(map, f, tp, emu_smem);
        else if (metric == 1) zb::t3_body<1, 0, 1, TW>(map, f, tp, emu_smem);
        else if (metric == 3) zb::t3_body<3, 0, 1, TW>(map, f, tp, emu_smem);
        else zb::t3_body<2, 0, 1, TW>(map, f, tp, emu_smem);
    } else {
        if (metric == 0) zb::t3_body<0, 0, T3_KR_MAX, TW>(map, f, tp, emu_smem);
        else if (metric == 1) zb::t3_body<1, 0, T3_KR_MAX, TW>(map, f, tp, emu_smem);
        else zb::t3_body<2, 0, T3_KR_MAX, TW>(map, f, tp, emu_smem);
    }
}

// METRIC 3 (dot-product filter): what the launch code adds to T3Params, set before emu_scan3(metric = 3, ...)
static struct { const float* bm_n2; const float* q_n2; const float* leaf_n2max; float ecoef; uint64_t* cand; float* cand_cut; uint8_t* cand_flag; } emu_filter;
extern "C" __attribute__((visibility("default"))) void emu_scan3_set_filter(const float* bm_n2, const float* q_n2, const float* leaf_n2max, float ecoef,
                                                                          uint64_t* cand, float* cand_cut, uint8_t* cand_flag) {
    emu_filter = {bm_n2, q_n2, leaf_n2max, ecoef, cand, cand_cut, cand_flag};
}

extern "C" __attribute__((visibility("default"))) int emu_scan3(
    int metric, int blocks, int dim, int nst, int qcap, int kr, uint32_t top_k, uint64_t positions, const float* bm_rows_padded,
    const double* bm_rinv, const uint32_t* bm_tomb, const uint64_t* ord, const uint32_t* members, const long long* leaf_off,
    const uint32_t* leaf_len, uint32_t ntiles, const uint32_t* tile_leaf, const uint32_t* tile_first, const uint32_t* tile_count,
    const uint32_t* order, const uint32_t* v_np, const uint32_t* v_q, const uint32_t* v_ent_off, const float* queries_padded,
    const double* q_rinv, uint64_t* gthr, uint64_t* entries /* [slots][2] */, uint64_t* stats3) {
    zb::ForestView f;
    f.leaf_off = leaf_off; f.leaf_len = leaf_len; f.members = members; f.ord = reinterpret_cast<const zb::u64*>(ord);
    f.dimp = (dim + 15) / 16 * 16; f.chunks = f.dimp / 16;
    uint32_t counter = 0;
    zb::T3Params tp;
    tp.tile_leaf = tile_leaf; tp.tile_first = tile_first; tp.tile_count = tile_count; tp.ntiles = &ntiles; tp.tile_counter = &counter;
    tp.order = order; tp.v_np = v_np; tp.v_q = v_q; tp.v_ent_off = v_ent_off; tp.entries = reinterpret_cast<zb::Entry*>(entries);
    tp.queries = queries_padded; tp.q_rinv = q_rinv; tp.bm_rinv = bm_rinv; tp.bm_tomb = bm_tomb;
    tp.stats = reinterpret_cast<zb::u64*>(stats3); tp.gthr = reinterpret_cast<zb::u64*>(gthr); tp.top_k = top_k; tp.nst = nst; tp.qcap = qcap; tp.kr = kr;
    tp.pj_cst = nullptr; tp.pj_sign = nullptr; tp.pj_hp = 0;
    tp.bm_n2 = emu_filter.bm_n2; tp.q_n2 = emu_filter.q_n2; tp.leaf_n2max = emu_filter.leaf_n2max; tp.ecoef = emu_filter.ecoef;
    tp.cand = reinterpret_cast<zb::u64*>(emu_filter.cand); tp.cand_cut = emu_filter.cand_cut; tp.cand_flag = emu_filter.cand_flag;
    zb::T3Map map{bm_rows_padded, positions, f.dimp};
    if (kr != 1 && kr != T3_KR_MAX) return -1;
    if (metric == 3 && (kr != 1 || !tp.cand)) return -1;
    const zb::T3Layout lay = zb::t3_layout(nst, f.dimp, qcap, kr);
    std::vector<unsigned char> smem((size_t)T3_TEAMS * lay.total + 1024);
    const int tw = emu_tw;
#if T3_KC != 3 || T3_EPW
    if (tw != 4) return -1;
#endif
    const unsigned nthreads = tw == 4 ? zb::T3Shape<4>::THREADS : zb::T3Shape<8>::THREADS;
    emu_warps.clear();
    for (unsigned i = 0; i < nthreads / 32; ++i) emu_warps.emplace_back(new WarpBox());
    for (int b = 0; b < blocks; ++b) {
        // garbage in shared memory at block start: nothing may depend on its content
        for (size_t i = 0; i < smem.size(); ++i) smem[i] = (unsigned char)(0xA5 ^ (i * 131));
        emu_smem = smem.data();
        emu_mbars.clear();
        CopyEngine dma;
        emu_dma = &dma;
        dma.start();
        std::barrier<> bar(nthreads), tb0(tw * 32), tb1(tw * 32);
        emu_block_bar = &bar;
        emu_team_bar[0] = &tb0;
        emu_team_bar[1] = &tb1;
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nthreads; ++t)
            th.emplace_back([&, t] {
                emu_threadIdx = Dim3{t, 0, 0};
#if T3_KC == 3 && !T3_EPW
                if (tw == 8) emu_run_scan3<8>(metric, kr, map, f, tp);
                else
#endif
                    emu_run_scan3<4>(metric, kr, map, f, tp);
            });
        for (auto& x : th) x.join();
        dma.finish();
    }
    return (int)counter;
}

// Second pass of METRIC 3: `warps` warps (run one after the other: a legal schedule) pull visits from the work counter.
extern "C" __attribute__((visibility("default"))) int emu_refine(
    int metric /* 1 or 2 */, int warps, int dim, const float* bm_rows_padded, const uint32_t* bm_tomb, const uint64_t* ord, const uint32_t* members,
    const long long* leaf_off, const uint32_t* leaf_len, const float* queries_padded, const uint32_t* order, uint32_t nvisits,
    const uint32_t* v_leaf, const uint32_t* v_np, const uint32_t* v_q, const uint32_t* v_ent_off, const uint64_t* gthr, uint64_t* entries,
    uint64_t* stats8) {
    zb::ForestView f;
    f.leaf_off = leaf_off; f.leaf_len = leaf_len; f.members = members; f.ord = reinterpret_cast<const zb::u64*>(ord);
    f.dimp = (dim + 15) / 16 * 16; f.chunks = f.dimp / 16;
    uint32_t counter = 0;
    zb::T3RefineParams rp;
    rp.bm_rows = bm_rows_padded; rp.bm_tomb = bm_tomb; rp.queries = queries_padded; rp.order = order; rp.nvisits = &nvisits;
    rp.v_leaf = v_leaf; rp.v_np = v_np; rp.v_q = v_q; rp.v_ent_off = v_ent_off;
    rp.cand = reinterpret_cast<const zb::u64*>(emu_filter.cand); rp.cand_cut = emu_filter.cand_cut; rp.cand_flag = emu_filter.cand_flag;
    rp.gthr = reinterpret_cast<const zb::u64*>(gthr); rp.q_n2 = emu_filter.q_n2; rp.leaf_n2max = emu_filter.leaf_n2max; rp.ecoef = emu_filter.ecoef;
    rp.entries = reinterpret_cast<zb::Entry*>(entries); rp.work_counter = &counter; rp.stats = reinterpret_cast<zb::u64*>(stats8);
    emu_warps.clear();
    emu_warps.emplace_back(new WarpBox());
    for (int w = 0; w < warps; ++w) {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < 32; ++t)
            th.emplace_back([&, t] {
                emu_threadIdx = Dim3{t, 0, 0};
                if (metric == 1) zb::t3_refine_warp<1>(f, rp, (int)t);
                else zb::t3_refine_warp<2>(f, rp, (int)t);
            });
        for (auto& x : th) x.join();
    }
    return (int)counter;
}

// Projection mode: rows [n][dimp] x planes [H][dimp] -> sign[n][Hp]; tiles = (row range, <= tq planes), built here the way
// launch_project3 builds them.
extern "C" __attribute__((visibility("default"))) int emu_project3(int blocks, int dim, int nst, int qcap, uint64_t n, const float* rows_padded,
                                                                 int H, const float* coef_padded, const float* cst, uint32_t range_rows,
                                                                 uint32_t tq, uint8_t* sign, int Hp, uint64_t* stats3) {
    zb::ForestView f;
    f.dimp = (dim + 15) / 16 * 16; f.chunks = f.dimp / 16;
    const uint32_t nranges = (uint32_t)((n + range_rows - 1) / range_rows), npt = (uint32_t)((H + tq - 1) / tq);
    std::vector<long long> leaf_off(nranges);
    std::vector<uint32_t> leaf_len(nranges), tile_leaf, tile_first, tile_count;
    for (uint32_t r = 0; r < nranges; ++r) {
        leaf_off[r] = (long long)r * range_rows;
        leaf_len[r] = (uint32_t)std::min<uint64_t>(range_rows, n - (uint64_t)r * range_rows);
        for (uint32_t p = 0; p < npt; ++p) {
            tile_leaf.push_back(r); tile_first.push_back(p * tq); tile_count.push_back(std::min<uint32_t>(tq, (uint32_t)H - p * tq));
        }
    }
    f.leaf_off = leaf_off.data(); f.leaf_len = leaf_len.data(); f.members = nullptr; f.ord = nullptr;
    uint32_t counter = 0, ntiles = (uint32_t)tile_leaf.size();
    zb::T3Params tp;
    memset(&tp, 0, sizeof tp);
    tp.tile_leaf = tile_leaf.data(); tp.tile_first = tile_first.data(); tp.tile_count = tile_count.data(); tp.ntiles = &ntiles;
    tp.tile_counter = &counter; tp.queries = coef_padded; tp.stats = reinterpret_cast<zb::u64*>(stats3); tp.nst = nst; tp.qcap = qcap; tp.kr = 1;
    tp.pj_cst = cst; tp.pj_sign = sign; tp.pj_hp = Hp;
    zb::T3Map map{rows_padded, n, f.dimp};
    const zb::T3Layout lay = zb::t3_layout(nst, f.dimp, qcap, 1);
    std::vector<unsigned char> smem((size_t)T3_TEAMS * lay.total + 1024);
    const int tw = emu_tw;
#if T3_KC != 3 || T3_EPW
    if (tw != 4) return -1;
#endif
    const unsigned nthreads = tw == 4 ? zb::T3Shape<4>::THREADS : zb::T3Shape<8>::THREADS;
    emu_warps.clear();
    for (unsigned i = 0; i < nthreads / 32; ++i) emu_warps.emplace_back(new WarpBox());
    for (int b = 0; b < blocks; ++b) {
        for (size_t i = 0; i < smem.size(); ++i) smem[i] = (unsigned char)(0x5A ^ (i * 37));
        emu_smem = smem.data();
        emu_mbars.clear();
        CopyEngine dma;
        emu_dma = &dma;
        dma.start();
        std::barrier<> bar(nthreads), tb0(tw * 32), tb1(tw * 32);
        emu_block_bar = &bar; emu_team_bar[0] = &tb0; emu_team_bar[1] = &tb1;
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nthreads; ++t)
            th.emplace_back([&, t] {
                emu_threadIdx = Dim3{t, 0, 0};
#if T3_KC == 3 && !T3_EPW
                if (tw == 8) zb::t3_body<0, 1, 1, 8>(map, f, tp, emu_smem);
                else
#endif
                    zb::t3_body<0, 1, 1, 4>(map, f, tp, emu_smem);
            });
        for (auto& x : th) x.join();
        dma.finish();
    }
    return (int)counter;
}

extern "C" __attribute__((visibility("default"))) void emu_scan3_layout(int nst, int dim, int qcap, int kr, uint32_t* out8) {
    const zb::T3Layout l = zb::t3_layout(nst, (dim + 15) / 16 * 16, qcap, kr);
    out8[0] = l.stage; out8[1] = l.queries; out8[2] = l.sums; out8[3] = l.lists; out8[4] = l.meta; out8[5] = l.info; out8[6] = l.bars; out8[7] = l.total;
}
