// zb_kernels.cu -- plan / score / select / merge / hash / build / mutation kernels (sm_100a).
// The bandwidth-critical leaf-tile scan lives in zb_scan.cu; the kernels here are the general path that is
// correct for every forest shape (deep trees with tiny leaves included) and the build/mutation machinery.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "zb_kernels.cuh"

namespace zb {

// =====================================================================================================
// plan: the control flow of LSHIndex::tree_result (/root/reference/src/database/index/lsh.rs:290-348).
// One quad per (query, tree) "walker".  The walk is distance independent (survey Q3): a leaf visited with
// budget n returns min(live, n), so which leaves are visited, and with which budget, depends only on the
// query's sign bits and on the live leaf sizes.  The walker emits (leaf, n) records; scoring happens later.
// =====================================================================================================
// The dot product of the tail kernel (walkers the count cascade sends past their first leaf).  A walk is a chain of dependent
// nodes; a walker that Q1 sends through dozens of tiny leaves visits hundreds of them, long after the bulk of the batch
// (L2-bandwidth bound) has finished: alone on the machine its time is round trips to L2 per node, and with quad_dot's 4 chunks
// in flight a 768-float node costs 12 of them -- one such walker held a whole 8-GPU step back by ~1 ms
// (profiles/r02q_trace_8gpu_all_ranks_peer_push.txt: the same (batch, rank) pairs in every run).  Here 24 chunks of the plane
// row are requested before the first is consumed.  ptxas, left alone, interleaves requests and FFMAs to save registers (the
// first FFMA then stalls with 4-6 requests in flight), so the requests are `volatile` loads (kept in program order; they
// bypass L1, which holds nothing of a deep node's plane anyway) and the head of every accumulator chain is made to depend
// on the LAST request by or-ing in `bits & zero`.  Same fused multiply-add sequence per accumulator lane as quad_dot.
// N2 (probe walk, first descent): the plane's canonical self-dot is accumulated from the same loads into *n2.
template <bool N2 = false>
__device__ __forceinline__ float quad_dot_tail(const float4* __restrict__ a, const float4* __restrict__ b, int chunks, int sub, unsigned mask,
                                               const u32 zero /* 0, derived from a kernel argument: the compiler cannot know */,
                                               float* n2 = nullptr) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
    int c = 0;
    for (; c + 24 <= chunks; c += 24) {
        float4 av[24];
#pragma unroll
        for (int i = 0; i < 24; ++i)
            asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(av[i].x), "=f"(av[i].y), "=f"(av[i].z), "=f"(av[i].w) : "l"(a + (c + i) * 4 + sub));
        const u32 dep = __float_as_uint(av[23].w) & zero;
        av[0].x = __uint_as_float(__float_as_uint(av[0].x) | dep);
        av[0].y = __uint_as_float(__float_as_uint(av[0].y) | dep);
        av[0].z = __uint_as_float(__float_as_uint(av[0].z) | dep);
        av[0].w = __uint_as_float(__float_as_uint(av[0].w) | dep);
#pragma unroll
        for (int i = 0; i < 24; ++i) {
            fma4(acc, av[i], __ldg(b + (c + i) * 4 + sub));   // the query: L1 hits
            if (N2) fma4(acc2, av[i], av[i]);
        }
    }
    for (; c + 4 <= chunks; c += 4) {
        float4 a0 = __ldg(a + (c + 0) * 4 + sub), a1 = __ldg(a + (c + 1) * 4 + sub);
        float4 a2 = __ldg(a + (c + 2) * 4 + sub), a3 = __ldg(a + (c + 3) * 4 + sub);
        float4 b0 = __ldg(b + (c + 0) * 4 + sub), b1 = __ldg(b + (c + 1) * 4 + sub);
        float4 b2 = __ldg(b + (c + 2) * 4 + sub), b3 = __ldg(b + (c + 3) * 4 + sub);
        fma4(acc, a0, b0);
        fma4(acc, a1, b1);
        fma4(acc, a2, b2);
        fma4(acc, a3, b3);
        if (N2) {
            fma4(acc2, a0, a0);
            fma4(acc2, a1, a1);
            fma4(acc2, a2, a2);
            fma4(acc2, a3, a3);
        }
    }
    for (; c < chunks; ++c) {
        const float4 ac = __ldg(a + c * 4 + sub);
        fma4(acc, ac, __ldg(b + c * 4 + sub));
        if (N2) fma4(acc2, ac, ac);
    }
    if (N2) *n2 = quad_reduce16(acc2, mask);
    return quad_reduce16(acc, mask);
}

// quad_dot (zb_device.cuh) with the plane's canonical self-dot accumulated from the same loads into n2.
__device__ __forceinline__ float quad_dot_n2(const float4* __restrict__ a, const float4* __restrict__ b, int chunks, int sub,
                                             unsigned mask, float& n2) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
    int c = 0;
    for (; c + 4 <= chunks; c += 4) {
        float4 a0 = __ldg(a + (c + 0) * 4 + sub), a1 = __ldg(a + (c + 1) * 4 + sub);
        float4 a2 = __ldg(a + (c + 2) * 4 + sub), a3 = __ldg(a + (c + 3) * 4 + sub);
        float4 b0 = __ldg(b + (c + 0) * 4 + sub), b1 = __ldg(b + (c + 1) * 4 + sub);
        float4 b2 = __ldg(b + (c + 2) * 4 + sub), b3 = __ldg(b + (c + 3) * 4 + sub);
        fma4(acc, a0, b0);
        fma4(acc, a1, b1);
        fma4(acc, a2, b2);
        fma4(acc, a3, b3);
        fma4(acc2, a0, a0);
        fma4(acc2, a1, a1);
        fma4(acc2, a2, a2);
        fma4(acc2, a3, a3);
    }
    for (; c < chunks; ++c) {
        const float4 ac = __ldg(a + c * 4 + sub);
        fma4(acc, ac, __ldg(b + c * 4 + sub));
        fma4(acc2, ac, ac);
    }
    n2 = quad_reduce16(acc2, mask);
    return quad_reduce16(acc, mask);
}

// Margin key of a main-path node (DESIGN 3.9): |v| / sqrt(n2) in f64, v = (f64)dot + (f64)cst the value point_is_above tests,
// n2 the plane's canonical self-dot; +inf when v is NaN or n2 is 0 or not finite.
__device__ __forceinline__ double probe_key(float dot, float cst, float n2f) {
    const double v = __dadd_rn((double)dot, (double)cst);
    const double n2 = (double)n2f;
    if (isnan(v) || !(n2 > 0.0) || isinf(n2)) return __longlong_as_double(0x7FF0000000000000ll);
    return __ddiv_rn(fabs(v), __dsqrt_rn(n2));
}

// One walker.  TAIL == false (plan_walk_kernel): with `defer` set, a walker whose first leaf cannot fill its budget (the count
// cascade goes on) is put on the tail list and left to plan_walk_tail_kernel, which walks it again from the root with
// quad_dot_tail; returns without writing anything for it.
// PROBE (multi-probe search, DESIGN 3.9): the first descent also keeps each main-path node's margin key and backup child; after
// the reference walk the `probes` nodes with the smallest (key, depth) are flipped, each backup side is descended greedily to
// one probe leaf, and every probe leaf with live rows is appended as a visit with n' = top_k.
template <bool TAIL, bool PROBE = false>
__device__ __forceinline__ void plan_walk_one(const ForestView& f, const float* __restrict__ queries, const u32 w, const int sub,
                                              const unsigned mask, const u32 top_k, const u32 vpw, uint2* __restrict__ wvisits,
                                              u32* __restrict__ wcounts, u32* __restrict__ overflow, u32* __restrict__ tail_list,
                                              u32* __restrict__ tail_count, const u32 probes = 0) {
    const u32 q = w / (u32)f.num_trees;
    const u32 t = w - q * (u32)f.num_trees;
    const float4* qv = reinterpret_cast<const float4*>(queries + (size_t)q * f.dimp);

    int stack_node[ZB_MAX_DEPTH + 2];
    int stack_n[ZB_MAX_DEPTH + 2];
    double pkey[PROBE ? ZB_MAX_DEPTH + 2 : 1];  // main path: margin key by depth
    int pback[PROBE ? ZB_MAX_DEPTH + 2 : 1];    // main path: backup child by depth
    int plen = -1;                              // main-path length, known once the first descent has reached its leaf
    int sp = 0;
    int cur = f.roots[t];
    int n = (int)top_k;
    u32 nvis = 0, ovf = 0;
    const u32 cap = vpw - 1;  // slot 0 of a walker's region is its header {visit count, overflow flag}
    for (;;) {
        int4 nd = f.nodes[cur];
        while (nd.x >= 0) {  // inner node: lsh.rs:333-338
            const float cst = f.cst[nd.x];
            const float4* plane = reinterpret_cast<const float4*>(f.coef + (size_t)nd.x * f.dimp);
            float d, n2 = 0.f;
            if (PROBE && plen < 0)
                d = TAIL ? quad_dot_tail<true>(plane, qv, f.chunks, sub, mask, top_k >> 31, &n2) : quad_dot_n2(plane, qv, f.chunks, sub, mask, n2);
            else
                d = TAIL ? quad_dot_tail(plane, qv, f.chunks, sub, mask, top_k >> 31) : quad_dot(plane, qv, f.chunks, sub, mask);
            bool ab = above_from_dot(d, cst);
            if (sp < ZB_MAX_DEPTH + 2) {
                stack_node[sp] = ab ? nd.y : nd.z;  // backup
                stack_n[sp] = n;
                if (PROBE && plen < 0) {
                    pkey[sp] = probe_key(d, cst, n2);
                    pback[sp] = ab ? nd.y : nd.z;
                }
            }
            ++sp;
            cur = ab ? nd.z : nd.y;  // main
            nd = f.nodes[cur];
        }
        if (PROBE && plen < 0) plen = sp;
        if (sp > ZB_MAX_DEPTH + 2) {  // cannot happen for forests accepted by the host (depth checked)
            ovf = 2;
            break;
        }
        const int live = (int)f.leaf_plan[nd.w];
        const int r = live < n ? live : n;  // lsh.rs:307 / :329
        if (!TAIL && tail_list && nvis == 0 && sp > 0 && r < n) {
            // first leaf, budget not filled, backups exist (they all carry n = top_k > r): the walk goes on -> tail kernel
            if (sub == 0) tail_list[atomicAdd(tail_count, 1u)] = w;
            return;
        }
        if (live > 0 && n > 0) {
            if (nvis < cap && sub == 0) wvisits[(size_t)w * vpw + 1 + nvis] = make_uint2((u32)nd.w, (u32)n);
            ++nvis;
        }
        bool again = false;
        while (sp > 0) {  // unwind: lsh.rs:340-345 (k < n -> backup with n - k, its result REPLACES k: Q1)
            --sp;
            const int nn = stack_n[sp];
            if (r < nn) {
                cur = stack_node[sp];
                n = nn - r;
                again = true;
                break;
            }
        }
        if (!again) break;
    }
    if (PROBE && !ovf) {
        // the i-th probe is the smallest (key, depth) after the (i-1)-th: depths are distinct, so no node is picked twice
        const int np = (int)probes < plen ? (int)probes : plen;
        double lk = -1.0;
        int ld = -1;
        for (int i = 0; i < np; ++i) {
            double bk = __longlong_as_double(0x7FF0000000000000ll);
            int bd = 0x7FFFFFFF;
            for (int dd = 0; dd < plen; ++dd) {
                const double k = pkey[dd];
                if ((k > lk || (k == lk && dd > ld)) && (k < bk || (k == bk && dd < bd))) {
                    bk = k;
                    bd = dd;
                }
            }
            lk = bk;
            ld = bd;
            int4 nd = f.nodes[pback[bd]];
            while (nd.x >= 0) {  // greedy descent of the backup side, no further flips
                const float4* plane = reinterpret_cast<const float4*>(f.coef + (size_t)nd.x * f.dimp);
                float d = TAIL ? quad_dot_tail(plane, qv, f.chunks, sub, mask, top_k >> 31) : quad_dot(plane, qv, f.chunks, sub, mask);
                nd = f.nodes[above_from_dot(d, f.cst[nd.x]) ? nd.z : nd.y];
            }
            if (f.leaf_plan[nd.w] > 0) {
                if (nvis < cap && sub == 0) wvisits[(size_t)w * vpw + 1 + nvis] = make_uint2((u32)nd.w, top_k);
                ++nvis;
            }
        }
    }
    if (sub == 0) {
        if (nvis > cap && !ovf) ovf = 1;
        const u32 c = nvis < cap ? nvis : cap;
        wcounts[w] = c;
        wvisits[(size_t)w * vpw] = make_uint2(c, ovf);  // the header travels with the visits (sharded: ONE allgather)
        if (ovf) atomicMax(overflow, ovf);
    }
}

__global__ void __launch_bounds__(128) plan_walk_kernel(ForestView f, const float* __restrict__ queries, u32 nq,
                                                        u32 top_k, u32 vpw, uint2* __restrict__ wvisits,
                                                        u32* __restrict__ wcounts, u32* __restrict__ overflow,
                                                        u32* __restrict__ tail_list, u32* __restrict__ tail_count) {
    const u32 w = blockIdx.x * 32u + (threadIdx.x >> 2);
    const u32 nwalkers = nq * (u32)f.num_trees;
    if (w >= nwalkers) return;
    plan_walk_one<false>(f, queries, w, (int)(threadIdx.x & 3), quad_mask(), top_k, vpw, wvisits, wcounts, overflow, tail_list, tail_count);
}
// The walkers the main kernel set aside, one quad each, a quad taking list entries in a grid-stride loop.
__global__ void __launch_bounds__(128, 1) plan_walk_tail_kernel(ForestView f, const float* __restrict__ queries, u32 top_k, u32 vpw,
                                                                uint2* __restrict__ wvisits, u32* __restrict__ wcounts,
                                                                u32* __restrict__ overflow, const u32* __restrict__ tail_list,
                                                                const u32* __restrict__ tail_count) {
    const u32 n = *tail_count;
    const unsigned mask = quad_mask();
    for (u32 i = blockIdx.x * 32u + (threadIdx.x >> 2); i < n; i += gridDim.x * 32u)
        plan_walk_one<true>(f, queries, tail_list[i], (int)(threadIdx.x & 3), mask, top_k, vpw, wvisits, wcounts, overflow, nullptr, nullptr);
}
// The same two kernels for a multi-probe batch (probes >= 1).
__global__ void __launch_bounds__(128) plan_walk_probe_kernel(ForestView f, const float* __restrict__ queries, u32 nq, u32 top_k,
                                                              u32 probes, u32 vpw, uint2* __restrict__ wvisits,
                                                              u32* __restrict__ wcounts, u32* __restrict__ overflow,
                                                              u32* __restrict__ tail_list, u32* __restrict__ tail_count) {
    const u32 w = blockIdx.x * 32u + (threadIdx.x >> 2);
    const u32 nwalkers = nq * (u32)f.num_trees;
    if (w >= nwalkers) return;
    plan_walk_one<false, true>(f, queries, w, (int)(threadIdx.x & 3), quad_mask(), top_k, vpw, wvisits, wcounts, overflow, tail_list,
                               tail_count, probes);
}
__global__ void __launch_bounds__(128, 1) plan_walk_probe_tail_kernel(ForestView f, const float* __restrict__ queries, u32 top_k,
                                                                      u32 probes, u32 vpw, uint2* __restrict__ wvisits,
                                                                      u32* __restrict__ wcounts, u32* __restrict__ overflow,
                                                                      const u32* __restrict__ tail_list,
                                                                      const u32* __restrict__ tail_count) {
    const u32 n = *tail_count;
    const unsigned mask = quad_mask();
    for (u32 i = blockIdx.x * 32u + (threadIdx.x >> 2); i < n; i += gridDim.x * 32u)
        plan_walk_one<true, true>(f, queries, tail_list[i], (int)(threadIdx.x & 3), mask, top_k, vpw, wvisits, wcounts, overflow, nullptr,
                                  nullptr, probes);
}

// tail_list: [walkers + 1] u32 scratch, element 0 is the counter; pass nullptr to keep every walker in the main kernel (what a
// forest whose leaves cannot hold top_k rows wants: there every walker cascades).  probes > 0: the multi-probe walk.
void launch_plan(const ForestView& f, const float* d_queries, u32 nq, u32 top_k, u32 probes, u32 vpw, uint2* d_wvisits,
                 u32* d_wcounts, u32* d_overflow, u32* d_tail_list, cudaStream_t s) {
    u32 nwalkers = nq * (u32)f.num_trees;
    if (!nwalkers) return;
    if (d_tail_list) cudaMemsetAsync(d_tail_list, 0, 4, s);
    if (probes)
        plan_walk_probe_kernel<<<(nwalkers + 31) / 32, 128, 0, s>>>(f, d_queries, nq, top_k, probes, vpw, d_wvisits, d_wcounts, d_overflow,
                                                                    d_tail_list ? d_tail_list + 1 : nullptr, d_tail_list);
    else
        plan_walk_kernel<<<(nwalkers + 31) / 32, 128, 0, s>>>(f, d_queries, nq, top_k, vpw, d_wvisits, d_wcounts, d_overflow,
                                                              d_tail_list ? d_tail_list + 1 : nullptr, d_tail_list);
    if (d_tail_list) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (probes)
            plan_walk_probe_tail_kernel<<<sms * 2, 128, 0, s>>>(f, d_queries, top_k, probes, vpw, d_wvisits, d_wcounts, d_overflow,
                                                                d_tail_list + 1, d_tail_list);
        else
            plan_walk_tail_kernel<<<sms * 2, 128, 0, s>>>(f, d_queries, top_k, vpw, d_wvisits, d_wcounts, d_overflow, d_tail_list + 1, d_tail_list);
    }
}

// Visit records -> flat visit arrays.  A visit the fused tile kernel will take (tile_on, leaf holds >= min_rows rows here,
// n' <= kmax) is marked done with no generic-path pairs right here, so that the entry-slot and pair totals are known
// before any scoring starts and the host needs ONE readback per batch.  Writes are guarded by `cap` (the host grows the
// arrays and reruns the compaction in the rare case the count exceeds it).
__global__ void compact_visits_kernel(ForestView f, u32 nwalkers, u32 vpw, const uint2* __restrict__ wvisits,
                                      const u32* __restrict__ wcounts, const u32* __restrict__ woff, u32 G, u32 rank, u32 cap,
                                      u32 tile_on, u32 min_rows, u32 kmax, u32* __restrict__ vleaf, u32* __restrict__ vnp,
                                      u32* __restrict__ vq, u64* __restrict__ pair_len, u32* __restrict__ ent_len,
                                      u8* __restrict__ vdone) {
    u32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwalkers) return;
    u32 c = wcounts[w], base = woff[w];
    u32 q = w / (u32)f.num_trees;
    for (u32 i = 0; i < c; ++i) {
        uint2 v = wvisits[(size_t)w * vpw + 1 + i];
        if (G > 1 && v.x % G != rank) continue;
        if (base < cap) {
            const u32 len = f.leaf_len[v.x];
            const bool tiled = tile_on && len >= min_rows && v.y <= kmax;
            vleaf[base] = v.x;
            vnp[base] = v.y;
            vq[base] = q;
            pair_len[base] = tiled ? 0ull : (u64)len;
            vdone[base] = tiled ? 1 : 0;
            u32 live = f.leaf_plan[v.x];
            ent_len[base] = live < v.y ? live : v.y;
        }
        ++base;
    }
}
void launch_compact_visits(const ForestView& f, u32 nwalkers, u32 vpw, const uint2* d_wvisits, const u32* d_wcounts,
                           const u32* d_woff, u32 G, u32 rank, u32 cap, u32 tile_on, u32 min_rows, u32 kmax, u32* d_vleaf,
                           u32* d_vnp, u32* d_vq, u64* d_pair_len, u32* d_ent_len, u8* d_vdone, cudaStream_t s) {
    if (!nwalkers) return;
    compact_visits_kernel<<<(nwalkers + 255) / 256, 256, 0, s>>>(f, nwalkers, vpw, d_wvisits, d_wcounts, d_woff, G, rank, cap, tile_on,
                                                                 min_rows, kmax, d_vleaf, d_vnp, d_vq, d_pair_len, d_ent_len, d_vdone);
}
// ---- sharded plan exchange: compacted visit records instead of padded per-walker regions ----
// A rank packs the visits of the walkers it planned into [header | records]: header = {visits, replan flag}; a record =
// {leaf, n', global walker}.  One ncclAllGather of (1 + cap) records per rank puts every rank's block on every rank; the
// header travels with the records, so the decisions "replan" and "grow cap" are taken from replicated data (identical on
// every rank: no rank can leave the loop alone).
__global__ void pack_visits_kernel(u32 nwalkers, u32 vpw, const uint2* __restrict__ wvisits, const u32* __restrict__ wcounts,
                                   const u32* __restrict__ woff, u32 walker_base, u32 cap, const u32* __restrict__ flag,
                                   uint4* __restrict__ out) {
    const u32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) out[0] = make_uint4(woff[nwalkers], flag[0], 0u, 0u);
    if (w >= nwalkers) return;
    const u32 c = wcounts[w];
    u32 base = woff[w];
    for (u32 i = 0; i < c; ++i, ++base) {
        if (base >= cap) break;
        const uint2 v = wvisits[(size_t)w * vpw + 1 + i];
        out[1 + base] = make_uint4(v.x, v.y, walker_base + w, 0u);
    }
}
void launch_pack_visits(u32 nwalkers, u32 vpw, const uint2* d_wvisits, const u32* d_wcounts, const u32* d_woff, u32 walker_base,
                        u32 cap, const u32* d_flag, uint4* d_out, cudaStream_t s) {
    pack_visits_kernel<<<(nwalkers + 256) / 256, 256, 0, s>>>(nwalkers, vpw, d_wvisits, d_wcounts, d_woff, walker_base, cap, d_flag, d_out);
}
// flags[r * cap + i] = record i of rank r exists and its leaf lives here; summary = {max replan flag, max visit count}
__global__ void own_flags_kernel(u32 G, u32 cap, size_t stride, const uint4* __restrict__ all, u32 rank, u32* __restrict__ flags,
                                 u32* __restrict__ summary) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        u32 f = 0, c = 0;
        for (u32 r = 0; r < G; ++r) {
            const uint4 h = all[(size_t)r * stride];
            f = max(f, h.y);
            c = max(c, h.x);
        }
        summary[0] = f;
        summary[1] = c;
    }
    if (i > G * cap) return;
    u32 fl = 0;
    if (i < G * cap) {
        const u32 r = i / cap, j = i - r * cap;
        const uint4* blk = all + (size_t)r * stride;
        if (j < blk[0].x) fl = (blk[1 + j].x % G == rank) ? 1u : 0u;
    }
    flags[i] = fl;  // [G * cap] = 0: the exclusive scan leaves the total there
}
void launch_own_flags(u32 G, u32 cap, size_t stride, const uint4* d_all, u32 rank, u32* d_flags, u32* d_summary, cudaStream_t s) {
    own_flags_kernel<<<(G * cap + 256) / 256, 256, 0, s>>>(G, cap, stride, d_all, rank, d_flags, d_summary);
}
// the records this rank owns -> flat visit arrays, in (planning rank, walker) order = global walker order
__global__ void own_scatter_kernel(ForestView f, u32 G, u32 cap, size_t stride, const uint4* __restrict__ all, const u32* __restrict__ flags,
                                   const u32* __restrict__ pos, u32 vcap, u32 tile_on, u32 min_rows, u32 kmax,
                                   u32* __restrict__ vleaf, u32* __restrict__ vnp, u32* __restrict__ vq, u32* __restrict__ vw,
                                   u64* __restrict__ pair_len, u32* __restrict__ ent_len, u8* __restrict__ vdone) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G * cap || !flags[i]) return;
    const u32 base = pos[i];
    if (base >= vcap) return;
    const u32 r = i / cap, j = i - r * cap;
    const uint4 v = all[(size_t)r * stride + 1 + j];
    const u32 len = f.leaf_len[v.x];
    const bool tiled = tile_on && len >= min_rows && v.y <= kmax;
    vleaf[base] = v.x;
    vnp[base] = v.y;
    vq[base] = v.z / (u32)f.num_trees;
    vw[base] = v.z;
    pair_len[base] = tiled ? 0ull : (u64)len;
    vdone[base] = tiled ? 1 : 0;
    const u32 live = f.leaf_plan[v.x];
    ent_len[base] = live < v.y ? live : v.y;
}
void launch_own_scatter(const ForestView& f, u32 G, u32 cap, size_t stride, const uint4* d_all, const u32* d_flags, const u32* d_pos, u32 vcap,
                        u32 tile_on, u32 min_rows, u32 kmax, u32* d_vleaf, u32* d_vnp, u32* d_vq, u32* d_vw, u64* d_pair_len,
                        u32* d_ent_len, u8* d_vdone, cudaStream_t s) {
    own_scatter_kernel<<<(G * cap + 255) / 256, 256, 0, s>>>(f, G, cap, stride, d_all, d_flags, d_pos, vcap, tile_on, min_rows, kmax, d_vleaf,
                                                             d_vnp, d_vq, d_vw, d_pair_len, d_ent_len, d_vdone);
}
// woff[w] = first visit of walker w (visits are in walker order), woff[nwalkers] = number of visits
__global__ void walker_offsets_kernel(u32 nwalkers, const u32* __restrict__ nv_ptr, u32 vcap, const u32* __restrict__ vw,
                                      u32* __restrict__ woff) {
    const u32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w > nwalkers) return;
    const u32 nv = *nv_ptr;
    if (w == nwalkers || nv > vcap) {  // nv > vcap: the host grows the arrays and compacts again
        woff[w] = w == nwalkers ? nv : 0u;
        return;
    }
    u32 lo = 0, hi = nv;  // first index with vw[index] >= w
    while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (vw[mid] < w) lo = mid + 1; else hi = mid;
    }
    woff[w] = lo;
}
void launch_walker_offsets(u32 nwalkers, const u32* d_nv, u32 vcap, const u32* d_vw, u32* d_woff, cudaStream_t s) {
    walker_offsets_kernel<<<(nwalkers + 256) / 256, 256, 0, s>>>(nwalkers, d_nv, vcap, d_vw, d_woff);
}

// {replan flag, visits, entry slots, generic-path pairs, largest per-rank visit count (sharded)} of the batch in one record
__global__ void plan_totals_kernel(const u32* __restrict__ flag, const u32* __restrict__ woff, u32 nwalkers, u32 cap,
                                   const u32* __restrict__ ent_off, const u64* __restrict__ pair_off, const u32* __restrict__ maxcount,
                                   u64* __restrict__ out) {
    const u32 nv = woff[nwalkers];
    const u32 at = nv < cap ? nv : cap;
    out[0] = flag[0];
    out[1] = nv;
    out[2] = ent_off[at];
    out[3] = pair_off[at];
    out[4] = maxcount ? maxcount[0] : 0u;
}
void launch_plan_totals(const u32* d_flag, const u32* d_woff, u32 nwalkers, u32 cap, const u32* d_ent_off, const u64* d_pair_off,
                        const u32* d_maxcount, u64* d_out, cudaStream_t s) {
    plan_totals_kernel<<<1, 1, 0, s>>>(d_flag, d_woff, nwalkers, cap, d_ent_off, d_pair_off, d_maxcount, d_out);
}

// =====================================================================================================
// score: metric.distance(row, query) for every (visit, member) pair -- the generic (gather) path.
// One quad per pair; 32 pairs per block.  distance.rs:19-49,:103-114 through the canonical order.
// =====================================================================================================
template <int METRIC>
__global__ void __launch_bounds__(128) score_pairs_kernel(ForestView f, const float* __restrict__ queries, u32 nv,
                                                          const u32* __restrict__ vleaf, const u32* __restrict__ vq,
                                                          const u64* __restrict__ pair_off, u64 total_pairs,
                                                          u64* __restrict__ pair_key) {
    __shared__ u32 s_v0;
    const u64 p0 = (u64)blockIdx.x * 32ull;
    if (threadIdx.x == 0) {  // visit containing pair p0: last v with pair_off[v] <= p0
        u32 lo = 0, hi = nv;
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (pair_off[mid] <= p0) lo = mid; else hi = mid;
        }
        s_v0 = lo;
    }
    __syncthreads();
    const u64 p = p0 + (threadIdx.x >> 2);
    if (p >= total_pairs) return;
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    u32 v = s_v0;
    {   // last v with pair_off[v] <= p (a binary search: runs of empty visits can be tens of thousands long)
        u32 hi = nv;
        while (hi - v > 1) {
            const u32 mid = (v + hi) >> 1;
            if (pair_off[mid] <= p) v = mid; else hi = mid;
        }
    }
    const u32 leaf = vleaf[v];
    const u32 slot = f.members[f.leaf_off[leaf] + (long long)(p - pair_off[v])];
    if (tomb_test(f.tomb, slot)) {
        if (sub == 0) pair_key[p] = ZB_SENTINEL;
        return;
    }
    const float4* a = reinterpret_cast<const float4*>(f.rows + (size_t)slot * f.dimp);
    const float4* b = reinterpret_cast<const float4*>(queries + (size_t)vq[v] * f.dimp);
    u64 key;
    if (METRIC == 0) {
        float4 ab = make_float4(0.f, 0.f, 0.f, 0.f), a2 = ab, b2 = ab;
        for (int c = 0; c < f.chunks; ++c) {
            float4 av = __ldg(a + c * 4 + sub), bv = __ldg(b + c * 4 + sub);
            fma4(ab, av, bv);
            fma4(a2, av, av);
            fma4(b2, bv, bv);
        }
        key = cos_bits(quad_reduce16(ab, mask), quad_reduce16(a2, mask), quad_reduce16(b2, mask));
    } else {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int c = 0;
        for (; c + 4 <= f.chunks; c += 4) {
            float4 a0 = __ldg(a + (c + 0) * 4 + sub), a1 = __ldg(a + (c + 1) * 4 + sub);
            float4 a2 = __ldg(a + (c + 2) * 4 + sub), a3 = __ldg(a + (c + 3) * 4 + sub);
            float4 b0 = __ldg(b + (c + 0) * 4 + sub), b1 = __ldg(b + (c + 1) * 4 + sub);
            float4 b2 = __ldg(b + (c + 2) * 4 + sub), b3 = __ldg(b + (c + 3) * 4 + sub);
            l2acc4(acc, a0, b0);
            l2acc4(acc, a1, b1);
            l2acc4(acc, a2, b2);
            l2acc4(acc, a3, b3);
        }
        for (; c < f.chunks; ++c) l2acc4(acc, __ldg(a + c * 4 + sub), __ldg(b + c * 4 + sub));
        float sum = quad_reduce16(acc, mask);
        key = METRIC == 1 ? l2sq_bits(sum) : l2_bits(sum);
    }
    if (sub == 0) pair_key[p] = key;
}

// The scalar metrics of distance.rs:51-190 (zb_metrics.cuh): a strictly sequential f32 fold per pair, so ONE THREAD owns a
// pair and walks its row once with 128-bit loads; the 32 pairs of a warp are (mostly) consecutive members of one visit, so
// the query elements are a broadcast and every row sector is consumed whole over two consecutive loads.  HBM-bound
// gather, 4N bytes per pair.
template <int CODE>
__device__ __forceinline__ u64 seq_distance_ldg(const float* __restrict__ a_, const float* __restrict__ b_, int dim, int power) {
    const float4* a = reinterpret_cast<const float4*>(a_);
    const float4* b = reinterpret_cast<const float4*>(b_);
    SeqAcc st;
    seq_init(st);
    const int n4 = dim >> 2;
#pragma unroll 2
    for (int i = 0; i < n4; ++i) {
        const float4 av = __ldg(a + i), bv = __ldg(b + i);
        seq_step<CODE>(st, av.x, bv.x, power);
        seq_step<CODE>(st, av.y, bv.y, power);
        seq_step<CODE>(st, av.z, bv.z, power);
        seq_step<CODE>(st, av.w, bv.w, power);
    }
    for (int i = n4 * 4; i < dim; ++i) seq_step<CODE>(st, __ldg(a_ + i), __ldg(b_ + i), power);  // dim % 4 tail (never the padding)
    return seq_finish<CODE>(st, power);
}

template <int CODE>
__global__ void __launch_bounds__(128) score_pairs_seq_kernel(ForestView f, int power, const float* __restrict__ queries, u32 nv,
                                                              const u32* __restrict__ vleaf, const u32* __restrict__ vq,
                                                              const u64* __restrict__ pair_off, u64 total_pairs,
                                                              u64* __restrict__ pair_key) {
    __shared__ u32 s_v0;
    const u64 p0 = (u64)blockIdx.x * 128ull;
    if (threadIdx.x == 0) {  // visit containing pair p0: last v with pair_off[v] <= p0
        u32 lo = 0, hi = nv;
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (pair_off[mid] <= p0) lo = mid; else hi = mid;
        }
        s_v0 = lo;
    }
    __syncthreads();
    const u64 p = p0 + threadIdx.x;
    if (p >= total_pairs) return;
    u32 v = s_v0;
    {
        u32 hi = nv;
        while (hi - v > 1) {
            const u32 mid = (v + hi) >> 1;
            if (pair_off[mid] <= p) v = mid; else hi = mid;
        }
    }
    const u32 leaf = vleaf[v];
    const u32 slot = f.members[f.leaf_off[leaf] + (long long)(p - pair_off[v])];
    if (tomb_test(f.tomb, slot)) {
        pair_key[p] = ZB_SENTINEL;
        return;
    }
    pair_key[p] = seq_distance_ldg<CODE>(f.rows + (size_t)slot * f.dimp, queries + (size_t)vq[v] * f.dimp, f.dim, power);
}

#define ZB_SEQ_DISPATCH(code, CALL)                     \
    switch (code) {                                     \
        case M_CHEBYSHEV: CALL(M_CHEBYSHEV); break;     \
        case M_CANBERRA: CALL(M_CANBERRA); break;       \
        case M_BRAY_CURTIS: CALL(M_BRAY_CURTIS); break; \
        case M_MANHATTAN: CALL(M_MANHATTAN); break;     \
        case M_L3: CALL(M_L3); break;                   \
        case M_L4: CALL(M_L4); break;                   \
        case M_HAMMING: CALL(M_HAMMING); break;         \
        case M_MINKOWSKI: CALL(M_MINKOWSKI); break;     \
        default: CALL(M_PNORM); break;                  \
    }

void launch_score_pairs(const ForestView& f, int metric, int power, const float* d_queries, u32 nv, const u32* d_vleaf,
                        const u32* d_vq, const u64* d_pair_off, u64 total_pairs, u64* d_pair_key, cudaStream_t s) {
    if (!total_pairs) return;
    if (metric > M_L2) {
        const u32 sblocks = (u32)((total_pairs + 127) / 128);
#define ZB_CALL(C) score_pairs_seq_kernel<C><<<sblocks, 128, 0, s>>>(f, power, d_queries, nv, d_vleaf, d_vq, d_pair_off, total_pairs, d_pair_key)
        ZB_SEQ_DISPATCH(metric, ZB_CALL)
#undef ZB_CALL
        return;
    }
    u32 blocks = (u32)((total_pairs + 31) / 32);
    if (metric == 0)
        score_pairs_kernel<0><<<blocks, 128, 0, s>>>(f, d_queries, nv, d_vleaf, d_vq, d_pair_off, total_pairs, d_pair_key);
    else if (metric == 1)
        score_pairs_kernel<1><<<blocks, 128, 0, s>>>(f, d_queries, nv, d_vleaf, d_vq, d_pair_off, total_pairs, d_pair_key);
    else
        score_pairs_kernel<2><<<blocks, 128, 0, s>>>(f, d_queries, nv, d_vleaf, d_vq, d_pair_off, total_pairs, d_pair_key);
}

// =====================================================================================================
// block-level streaming top-k with optional dedup: bitonic sort of (kept + chunk) entries in shared
// memory, keep the first k distinct.  Order = (distance bits as u64, ordinal): lsh.rs:318,:561 + D3.
// =====================================================================================================
#define TOPK_THREADS 128

__device__ __forceinline__ void bitonic_sort_block(Entry* s, int P) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P; i += TOPK_THREADS) {
                int ixj = i ^ j;
                if (ixj > i) {
                    Entry a = s[i], b = s[ixj];
                    bool up = (i & k) == 0;
                    if (entry_less(b, a) == up) {
                        s[i] = b;
                        s[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < TOPK_THREADS / 32; ++i) {
        int wv = s_warp[i];
        if (i < wid) base += wv;
        tot += wv;
    }
    __syncthreads();
    *total = tot;
    return base + x - v;
}

// buf: pmax entries, keep: k entries.  Returns the number of kept entries (sorted, distinct) in keep[0..).
template <class Loader>
__device__ int segment_topk(Entry* buf, Entry* keep, int* s_warp, const Loader& ld, long long len, int k, int pmax) {
    int kept = 0;
    const int ch = pmax - k;
    for (long long base = 0; base < len; base += ch) {
        const int c = (int)((len - base) < (long long)ch ? (len - base) : (long long)ch);
        const int total = kept + c;
        int P = 32;
        while (P < total) P <<= 1;
        for (int i = threadIdx.x; i < P; i += TOPK_THREADS) {
            if (i < kept) buf[i] = keep[i];
            else if (i < total) buf[i] = ld(base + (i - kept));
            else buf[i] = Entry{ZB_SENTINEL, ZB_SENTINEL};
        }
        __syncthreads();
        bitonic_sort_block(buf, P);
        int running = 0;
        for (int r0 = 0; r0 < P && running < k; r0 += TOPK_THREADS) {
            const int i = r0 + threadIdx.x;
            int flag = 0;
            Entry e = Entry{ZB_SENTINEL, ZB_SENTINEL};
            if (i < P) {
                e = buf[i];
                flag = (e.ord != ZB_SENTINEL) && (i == 0 || buf[i - 1].ord != e.ord || buf[i - 1].key != e.key);
            }
            int tot;
            int pos = running + block_exclusive_scan(flag, s_warp, &tot);
            if (flag && pos < k) keep[pos] = e;
            running += tot;
        }
        kept = running < k ? running : k;
        __syncthreads();
    }
    return kept;
}

struct VisitLoader {
    const u32* members;
    const u64* keys;
    const u64* ord;
    __device__ Entry operator()(long long i) const {
        u64 key = keys[i];
        if (key == ZB_SENTINEL) return Entry{ZB_SENTINEL, ZB_SENTINEL};
        return Entry{key, ord[members[i]]};
    }
};

// per-visit top-n' (lsh.rs:301-331): a leaf with live < n' contributes everything, otherwise its n' nearest.
__global__ void __launch_bounds__(TOPK_THREADS) select_visits_kernel(ForestView f, u32 nv, const u32* __restrict__ vleaf,
                                                                     const u32* __restrict__ vnp,
                                                                     const u64* __restrict__ pair_off,
                                                                     const u64* __restrict__ pair_key,
                                                                     const u32* __restrict__ ent_off,
                                                                     Entry* __restrict__ entries,
                                                                     const u8* __restrict__ vdone, int pmax, int kmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    Entry* buf = reinterpret_cast<Entry*>(smem);
    Entry* keep = buf + pmax;
    int* s_warp = reinterpret_cast<int*>(keep + kmax);
    const u32 v = blockIdx.x;
    if (v >= nv) return;
    if (vdone && vdone[v]) return;
    const u32 leaf = vleaf[v];
    const u32 slots = ent_off[v + 1] - ent_off[v];
    VisitLoader ld{f.members + f.leaf_off[leaf], pair_key + pair_off[v], f.ord};
    const int k = (int)vnp[v];
    int kept = segment_topk(buf, keep, s_warp, ld, (long long)f.leaf_len[leaf], k, pmax);
    Entry* out = entries + ent_off[v];
    for (u32 i = threadIdx.x; i < slots; i += TOPK_THREADS) out[i] = (int)i < kept ? keep[i] : Entry{ZB_SENTINEL, ZB_SENTINEL};
}

static inline int topk_pmax(u32 top_k) {
    int p = 1024;
    while (p < (int)(2 * top_k)) p <<= 1;
    return p;
}
static inline size_t topk_smem(int pmax, int kmax) { return (size_t)(pmax + kmax) * sizeof(Entry) + 64; }

template <class K>
static void set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

}  // namespace zb
#include "zb_select_kernel.cuh"
namespace zb {

void launch_select_visits(const ForestView& f, u32 nv, const u32* d_vleaf, const u32* d_vnp, const u64* d_pair_off,
                          const u64* d_pair_key, const u32* d_ent_off, Entry* d_entries, const u8* d_vdone, u32 top_k,
                          int variant, cudaStream_t s) {
    if (!nv) return;
    if (variant == 1 && top_k <= 128) {  // one warp per visit, the n' best in registers (zb_select_kernel.cuh)
        const u32 blocks = (nv + WS_WARPS - 1) / WS_WARPS;
        if (top_k <= 32)
            warp_select_visits_kernel<1><<<blocks, 32 * WS_WARPS, 0, s>>>(f, nv, d_vleaf, d_vnp, d_pair_off, d_pair_key, d_ent_off, d_entries, d_vdone);
        else if (top_k <= 64)
            warp_select_visits_kernel<2><<<blocks, 32 * WS_WARPS, 0, s>>>(f, nv, d_vleaf, d_vnp, d_pair_off, d_pair_key, d_ent_off, d_entries, d_vdone);
        else
            warp_select_visits_kernel<4><<<blocks, 32 * WS_WARPS, 0, s>>>(f, nv, d_vleaf, d_vnp, d_pair_off, d_pair_key, d_ent_off, d_entries, d_vdone);
        return;
    }
    int pmax = topk_pmax(top_k), kmax = (int)top_k;
    size_t smem = topk_smem(pmax, kmax);
    set_smem(select_visits_kernel, smem);
    select_visits_kernel<<<nv, TOPK_THREADS, smem, s>>>(f, nv, d_vleaf, d_vnp, d_pair_off, d_pair_key, d_ent_off,
                                                       d_entries, d_vdone, pmax, kmax);
}

// Sharded search: per-visit merge of the G ranks' local top-n' lists into the global top-n' (survey 8e ii).
struct RankLoader {
    const Entry* gathered;
    u32 total_slots, base, slots;
    __device__ Entry operator()(long long i) const {
        u32 r = (u32)(i / slots), j = (u32)(i % slots);
        return gathered[(size_t)r * total_slots + base + j];
    }
};
__global__ void __launch_bounds__(TOPK_THREADS) merge_ranks_kernel(u32 nv, const u32* __restrict__ ent_off, u32 total_slots,
                                                                   u32 nranks, const Entry* __restrict__ gathered,
                                                                   Entry* __restrict__ entries, int pmax, int kmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    Entry* buf = reinterpret_cast<Entry*>(smem);
    Entry* keep = buf + pmax;
    int* s_warp = reinterpret_cast<int*>(keep + kmax);
    const u32 v = blockIdx.x;
    if (v >= nv) return;
    const u32 base = ent_off[v], slots = ent_off[v + 1] - base;
    if (!slots) return;
    RankLoader ld{gathered, total_slots, base, slots};
    int kept = segment_topk(buf, keep, s_warp, ld, (long long)slots * nranks, (int)slots, pmax);
    for (u32 i = threadIdx.x; i < slots; i += TOPK_THREADS)
        entries[base + i] = (int)i < kept ? keep[i] : Entry{ZB_SENTINEL, ZB_SENTINEL};
}
void launch_merge_ranks(u32 nv, const u32* d_ent_off, u32 total_slots, u32 nranks, const Entry* d_gathered,
                        Entry* d_entries, u32 top_k, cudaStream_t s) {
    if (!nv) return;
    int pmax = topk_pmax(top_k), kmax = (int)top_k;
    size_t smem = topk_smem(pmax, kmax);
    set_smem(merge_ranks_kernel, smem);
    merge_ranks_kernel<<<nv, TOPK_THREADS, smem, s>>>(nv, d_ent_off, total_slots, nranks, d_gathered, d_entries, pmax, kmax);
}

// Union over trees and visits, dedup (DashSet, lsh.rs:550), sort ascending, take top_k (lsh.rs:561-564).
struct PlainLoader {
    const Entry* e;
    __device__ Entry operator()(long long i) const { return e[i]; }
};
__global__ void __launch_bounds__(TOPK_THREADS) merge_queries_kernel(u32 nq, u32 num_trees, const u32* __restrict__ woff,
                                                                     const u32* __restrict__ ent_off,
                                                                     const Entry* __restrict__ entries, u32 top_k,
                                                                     u64* __restrict__ out_ord, u64* __restrict__ out_bits,
                                                                     u32* __restrict__ out_counts, int pmax, int kmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    Entry* buf = reinterpret_cast<Entry*>(smem);
    Entry* keep = buf + pmax;
    int* s_warp = reinterpret_cast<int*>(keep + kmax);
    const u32 q = blockIdx.x;
    if (q >= nq) return;
    const u32 v0 = woff[(size_t)q * num_trees], v1 = woff[(size_t)(q + 1) * num_trees];
    const u32 e0 = ent_off[v0], e1 = ent_off[v1];
    PlainLoader ld{entries + e0};
    int kept = segment_topk(buf, keep, s_warp, ld, (long long)(e1 - e0), (int)top_k, pmax);
    for (u32 i = threadIdx.x; i < top_k; i += TOPK_THREADS) {
        bool ok = (int)i < kept;
        out_ord[(size_t)q * top_k + i] = ok ? keep[i].ord : ZB_SENTINEL;
        out_bits[(size_t)q * top_k + i] = ok ? keep[i].key : ZB_SENTINEL;
    }
    if (threadIdx.x == 0) out_counts[q] = (u32)kept;
}
void launch_merge_queries(u32 nq, u32 num_trees, const u32* d_woff, const u32* d_ent_off, const Entry* d_entries,
                          u32 top_k, u64* d_out_ord, u64* d_out_bits, u32* d_out_counts, cudaStream_t s) {
    if (!nq) return;
    int pmax = topk_pmax(top_k), kmax = (int)(top_k ? top_k : 1);
    size_t smem = topk_smem(pmax, kmax);
    set_smem(merge_queries_kernel, smem);
    merge_queries_kernel<<<nq, TOPK_THREADS, smem, s>>>(nq, num_trees, d_woff, d_ent_off, d_entries, top_k, d_out_ord,
                                                       d_out_bits, d_out_counts, pmax, kmax);
}

// =====================================================================================================
// hash: root-to-leaf descent by Hyperplane::point_is_above (lsh.rs:39-43 along :350-366).  One quad per
// (row, tree); the sign bits are the bucket key (MSB = root), the leaf is the bucket.
// =====================================================================================================
__global__ void __launch_bounds__(128) hash_kernel(ForestView f, const float* __restrict__ rows, u64 n,
                                                   u64* __restrict__ keys, u32* __restrict__ depths,
                                                   int* __restrict__ leaves) {
    const u64 w = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    if (w >= n * (u64)f.num_trees) return;
    const u64 r = w / (u64)f.num_trees;
    const int t = (int)(w - r * (u64)f.num_trees);
    const float4* x = reinterpret_cast<const float4*>(rows + (size_t)r * f.dimp);
    int cur = f.roots[t];
    int4 nd = f.nodes[cur];
    u64 key = 0;
    u32 depth = 0;
    while (nd.x >= 0) {
        float d = quad_dot(reinterpret_cast<const float4*>(f.coef + (size_t)nd.x * f.dimp), x, f.chunks, sub, mask);
        bool ab = above_from_dot(d, f.cst[nd.x]);
        key = (key << 1) | (ab ? 1ull : 0ull);
        ++depth;
        cur = ab ? nd.z : nd.y;
        nd = f.nodes[cur];
    }
    if (sub == 0) {
        if (keys) keys[w] = key;
        if (depths) depths[w] = depth;
        if (leaves) leaves[w] = nd.w;
    }
}
// Tree-major variant: the same quad-per-(row, tree) descent, but quad i works on tree i / n, row i % n, so the CTAs in
// flight at any moment (they are scheduled in index order) all walk ONE tree: the planes of its top levels (63 planes =
// 189 KB for six levels at N = 768) stay resident in L1 instead of being evicted by three other trees' planes, and
// only the deeper levels come from L2.  The row is read once per tree (L2 / HBM), which the plane traffic dwarfs.
__global__ void __launch_bounds__(128) hash_tree_major_kernel(ForestView f, const float* __restrict__ rows, u64 n,
                                                              u64* __restrict__ keys, u32* __restrict__ depths,
                                                              int* __restrict__ leaves) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    if (i >= n * (u64)f.num_trees) return;
    const int t = (int)(i / n);
    const u64 r = i - (u64)t * n;
    const float4* x = reinterpret_cast<const float4*>(rows + (size_t)r * f.dimp);
    int4 nd = f.nodes[f.roots[t]];
    u64 key = 0;
    u32 depth = 0;
    while (nd.x >= 0) {
        float d = quad_dot(reinterpret_cast<const float4*>(f.coef + (size_t)nd.x * f.dimp), x, f.chunks, sub, mask);
        bool ab = above_from_dot(d, f.cst[nd.x]);
        key = (key << 1) | (ab ? 1ull : 0ull);
        ++depth;
        nd = f.nodes[ab ? nd.z : nd.y];
    }
    if (sub == 0) {
        const u64 w = r * (u64)f.num_trees + t;
        if (keys) keys[w] = key;
        if (depths) depths[w] = depth;
        if (leaves) leaves[w] = nd.w;
    }
}
// Variant with the row staged in shared memory: a quad copies its row once (quad-private region, padded pitch so that the
// two quads of a quarter-warp hit disjoint banks) and walks ALL trees with it, so per level only the plane row is
// fetched (L1 / L2); the row itself is read from HBM exactly once.  32 rows per CTA.
#define HASH_ROWS_PER_CTA 32
__global__ void __launch_bounds__(128) hash_rows_kernel(ForestView f, const float* __restrict__ rows, u64 n, int pitch,
                                                        u64* __restrict__ keys, u32* __restrict__ depths,
                                                        int* __restrict__ leaves) {
    extern __shared__ __align__(16) float s_rows[];
    const int quad = threadIdx.x >> 2, sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const u64 r = (u64)blockIdx.x * HASH_ROWS_PER_CTA + quad;
    if (r >= n) return;
    float4* mine = reinterpret_cast<float4*>(s_rows + (size_t)quad * pitch);
    const float4* src = reinterpret_cast<const float4*>(rows + (size_t)r * f.dimp);
    const int chunks = f.chunks;
    for (int c = 0; c < chunks; ++c) mine[c * 4 + sub] = __ldg(src + c * 4 + sub);
    __syncwarp(mask);
    for (int t = 0; t < f.num_trees; ++t) {
        int4 nd = f.nodes[f.roots[t]];
        u64 key = 0;
        u32 depth = 0;
        while (nd.x >= 0) {
            const float4* p = reinterpret_cast<const float4*>(f.coef + (size_t)nd.x * f.dimp);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            int c = 0;
            for (; c + 8 <= chunks; c += 8) {   // 8 plane loads in flight per thread; chunk order = canonical order
                float4 p0 = __ldg(p + (c + 0) * 4 + sub), p1 = __ldg(p + (c + 1) * 4 + sub), p2 = __ldg(p + (c + 2) * 4 + sub),
                       p3 = __ldg(p + (c + 3) * 4 + sub), p4 = __ldg(p + (c + 4) * 4 + sub), p5 = __ldg(p + (c + 5) * 4 + sub),
                       p6 = __ldg(p + (c + 6) * 4 + sub), p7 = __ldg(p + (c + 7) * 4 + sub);
                fma4(acc, p0, mine[(c + 0) * 4 + sub]); fma4(acc, p1, mine[(c + 1) * 4 + sub]);
                fma4(acc, p2, mine[(c + 2) * 4 + sub]); fma4(acc, p3, mine[(c + 3) * 4 + sub]);
                fma4(acc, p4, mine[(c + 4) * 4 + sub]); fma4(acc, p5, mine[(c + 5) * 4 + sub]);
                fma4(acc, p6, mine[(c + 6) * 4 + sub]); fma4(acc, p7, mine[(c + 7) * 4 + sub]);
            }
            for (; c < chunks; ++c) fma4(acc, __ldg(p + c * 4 + sub), mine[c * 4 + sub]);
            const bool ab = above_from_dot(quad_reduce16(acc, mask), f.cst[nd.x]);
            key = (key << 1) | (ab ? 1ull : 0ull);
            ++depth;
            nd = f.nodes[ab ? nd.z : nd.y];
        }
        if (sub == 0) {
            const u64 w = r * (u64)f.num_trees + t;
            if (keys) keys[w] = key;
            if (depths) depths[w] = depth;
            if (leaves) leaves[w] = nd.w;
        }
    }
}

void launch_hash(const ForestView& f, const float* d_rows, u64 n, u64* d_keys, u32* d_depths, int* d_leaves, int variant,
                 cudaStream_t s) {
    u64 nw = n * (u64)f.num_trees;
    if (!nw) return;
    const int pitch = f.dimp + ((f.dimp % 32) == 0 ? 16 : 0);
    const size_t smem = (size_t)HASH_ROWS_PER_CTA * pitch * 4;
    if (variant == 1 && smem <= 200 * 1024) {
        static bool attr_set = false;
        if (!attr_set && smem > 48 * 1024) {
            cudaFuncSetAttribute(hash_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            attr_set = true;
        }
        hash_rows_kernel<<<(u32)((n + HASH_ROWS_PER_CTA - 1) / HASH_ROWS_PER_CTA), 128, smem, s>>>(f, d_rows, n, pitch, d_keys,
                                                                                                  d_depths, d_leaves);
        return;
    }
    if (variant == 2) {
        hash_tree_major_kernel<<<(u32)((nw + 31) / 32), 128, 0, s>>>(f, d_rows, n, d_keys, d_depths, d_leaves);
        return;
    }
    hash_kernel<<<(u32)((nw + 31) / 32), 128, 0, s>>>(f, d_rows, n, d_keys, d_depths, d_leaves);
}

// =====================================================================================================
// hash of FLAT tables (zb_project.cuh): dense projection rows x planes in the canonical order, then the K sign bits of
// every table packed into its bucket key with __ballot_sync.
// CTA = 32 quads = 8 row groups x 4 plane groups, quad tile 4 rows x 4 planes: CTA tile 32 rows x 16 planes.  Both
// operands come through L1 (__ldg): the 4 plane groups of a CTA re-read the same 32 rows, its 8 row groups the same 16
// planes.  Per thread and 16-float chunk: 8 128-bit loads feed 64 fused multiply-adds.
// =====================================================================================================
__global__ void __launch_bounds__(128) project_flat_kernel(const float* __restrict__ rows, u64 n, const float* __restrict__ coef,
                                                           const float* __restrict__ cst, int H, int dimp, int chunks,
                                                           u8* __restrict__ sign, int Hp) {
    const int quad = threadIdx.x >> 2, sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const u64 row0 = (u64)blockIdx.x * 32ull + (u64)(quad >> 2) * ZB_PJ_R;
    const int pl0 = (int)blockIdx.y * 16 + (quad & 3) * ZB_PJ_P;
    const float4* xr[ZB_PJ_R];
    const float4* pp[ZB_PJ_P];
#pragma unroll
    for (int i = 0; i < ZB_PJ_R; ++i) {  // tails: clamp the loads, mask the stores
        const u64 r = row0 + i < n ? row0 + i : n - 1;
        xr[i] = reinterpret_cast<const float4*>(rows + (size_t)r * dimp) + sub;
    }
#pragma unroll
    for (int j = 0; j < ZB_PJ_P; ++j) {
        const int h = pl0 + j < H ? pl0 + j : H - 1;
        pp[j] = reinterpret_cast<const float4*>(coef + (size_t)h * dimp) + sub;
    }
    PjAcc acc;
    pj_init(acc);
#pragma unroll 2
    for (int c = 0; c < chunks; ++c) {
        float4 x[ZB_PJ_R], p[ZB_PJ_P];
#pragma unroll
        for (int i = 0; i < ZB_PJ_R; ++i) x[i] = __ldg(xr[i] + c * 4);
#pragma unroll
        for (int j = 0; j < ZB_PJ_P; ++j) p[j] = __ldg(pp[j] + c * 4);
        pj_chunk(acc, x, p);
    }
#pragma unroll
    for (int i = 0; i < ZB_PJ_R; ++i) {
#pragma unroll
        for (int j = 0; j < ZB_PJ_P; ++j) {
            const float d = quad_reduce16(acc.a[i][j], mask);  // every thread of the quad takes part
            if (sub == 0 && row0 + i < n && pl0 + j < H)
                sign[(size_t)(row0 + i) * Hp + pl0 + j] = above_from_dot(d, __ldg(cst + pl0 + j)) ? 1 : 0;
        }
    }
}
// One warp per row: lane l holds the sign of plane t K + l (and of plane t K + 32 + l); the ballot IS the key, up to the
// bit order (MSB = plane 0 = the root decision).  leaf = the complete tree's leaf, t 2^K + key.
__global__ void __launch_bounds__(128) pack_flat_keys_kernel(const u8* __restrict__ sign, u64 n, int Hp, int T, int K,
                                                             u64* __restrict__ keys, u32* __restrict__ depths, int* __restrict__ leaves) {
    const u64 r = (u64)blockIdx.x * 4ull + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n) return;  // whole warps leave together
    const u8* s = sign + (size_t)r * Hp;
    for (int t = 0; t < T; ++t) {
        const unsigned b0 = __ballot_sync(0xffffffffu, lane < K && s[t * K + lane] != 0);
        const unsigned b1 = __ballot_sync(0xffffffffu, 32 + lane < K && s[t * K + 32 + lane] != 0);
        if (lane == 0) {
            const u64 key = K <= 32 ? (u64)(__brev(b0) >> (32 - K)) : (((u64)__brev(b0) << (K - 32)) | (u64)(__brev(b1) >> (64 - K)));
            const u64 w = r * (u64)T + t;
            if (keys) keys[w] = key;
            if (depths) depths[w] = (u32)K;
            if (leaves) leaves[w] = (int)(((u64)t << K) + key);
        }
    }
}
void launch_project_flat(const float* d_rows, u64 n, const float* d_coef, const float* d_cst, int H, int dimp, u8* d_sign, int Hp,
                         cudaStream_t s) {
    if (!n || !H) return;
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((H + 15) / 16));
    project_flat_kernel<<<grid, 128, 0, s>>>(d_rows, n, d_coef, d_cst, H, dimp, dimp / 16, d_sign, Hp);
}
void launch_pack_flat_keys(const u8* d_sign, u64 n, int Hp, int T, int K, u64* d_keys, u32* d_depths, int* d_leaves, cudaStream_t s) {
    if (!n) return;
    pack_flat_keys_kernel<<<(unsigned)((n + 3) / 4), 128, 0, s>>>(d_sign, n, Hp, T, K, d_keys, d_depths, d_leaves);
}

// =====================================================================================================
// build (lsh.rs:192-267), level synchronous.  The host keeps the list of nodes under construction
// ("segments" of a work array of slots); per level:
//   pick      two member rows per segment by seeded min-hash (D2)                    phases 0,1,2
//   planes    coef = b - a, mid = (a+b)/2, constant = -(f32)dot(coef, mid)           lsh.rs:222-225
//   classify  point_is_above for every member (the projection hot loop)              lsh.rs:236-241
//   scatter   stable partition: below first (left child), above after (right child)
// =====================================================================================================
// phase 0: minh[seg] = min hash (63-bit);  phase 1: minord[seg] = min ordinal among hash == minh;
// phase 2: slot[seg] = slot of the member whose ordinal == minord.   exclude[seg] (optional) is skipped.
__global__ void __launch_bounds__(64) pick_kernel(int phase, const Tile* __restrict__ tiles, const SegDesc* __restrict__ segs,
                                                  const u32* __restrict__ work, const u64* __restrict__ ord,
                                                  const u64* __restrict__ exclude, u64* __restrict__ minh,
                                                  u64* __restrict__ minord, int* __restrict__ slot_out) {
    const Tile tl = tiles[blockIdx.x];
    const bool active = threadIdx.x < tl.count;
    const SegDesc sg = segs[tl.seg];
    u32 slot = 0;
    u64 o = ZB_SENTINEL, h = ZB_SENTINEL;
    if (active) {
        slot = work[tl.start + threadIdx.x];
        o = ord[slot];
        if (exclude && exclude[tl.seg] == o) o = ZB_SENTINEL;
        else h = pick_hash(sg.key, (int)sg.attempt, o) >> 1;
    }
    if (phase == 0) {
        // a tile lies inside one segment: reduce over the warp first, one atomic per warp (the top levels have a handful
        // of segments, and millions of same-address atomics were what the level cost)
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const u32 lo = __shfl_xor_sync(0xffffffffu, (u32)h, m), hi = __shfl_xor_sync(0xffffffffu, (u32)(h >> 32), m);
            const u64 other = ((u64)hi << 32) | lo;
            h = other < h ? other : h;
        }
        if ((threadIdx.x & 31) == 0 && h != ZB_SENTINEL) atomicMin(&minh[tl.seg], h);
    } else if (o != ZB_SENTINEL) {
        if (phase == 1) { if (h == minh[tl.seg]) atomicMin(&minord[tl.seg], o); }
        else { if (o == minord[tl.seg]) slot_out[tl.seg] = (int)slot; }
    }
}
void launch_pick(int phase, const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work, const u64* d_ord,
                 const u64* d_exclude, u64* d_minh, u64* d_minord, int* d_slot, cudaStream_t s) {
    if (!ntiles) return;
    pick_kernel<<<ntiles, 64, 0, s>>>(phase, d_tiles, d_segs, d_work, d_ord, d_exclude, d_minh, d_minord, d_slot);
}

// pair_rows[seg][0] = row a, [seg][1] = row b (zeros when this shard does not own the row: the int32
// allreduce-sum over shards then reconstructs the exact bit patterns).
__global__ void fetch_pair_rows_kernel(u32 nsegs, const int* __restrict__ slot_a, const int* __restrict__ slot_b,
                                       const float* __restrict__ rows, int dimp, float* __restrict__ pair_rows) {
    const u32 sgi = blockIdx.x;
    for (int which = 0; which < 2; ++which) {
        int slot = which ? slot_b[sgi] : slot_a[sgi];
        float* dst = pair_rows + ((size_t)sgi * 2 + which) * dimp;
        for (int i = threadIdx.x; i < dimp; i += blockDim.x) dst[i] = slot >= 0 ? rows[(size_t)slot * dimp + i] : 0.0f;
    }
}
void launch_fetch_pair_rows(const SegDesc* d_segs, u32 nsegs, const int* d_slot_a, const int* d_slot_b,
                            const float* d_rows, int dimp, float* d_pair_rows, cudaStream_t s) {
    if (!nsegs) return;
    fetch_pair_rows_kernel<<<nsegs, 128, 0, s>>>(nsegs, d_slot_a, d_slot_b, d_rows, dimp, d_pair_rows);
}

// lsh.rs:222-225 (+ subtract/average :174-190): one quad per segment.
__global__ void __launch_bounds__(128) make_planes_kernel(const SegDesc* __restrict__ segs, u32 nsegs,
                                                          const float* __restrict__ pair_rows, int dimp,
                                                          float* __restrict__ coef, float* __restrict__ cst) {
    const u32 sgi = blockIdx.x * 32u + (threadIdx.x >> 2);
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    if (sgi >= nsegs) return;
    const float4* a = reinterpret_cast<const float4*>(pair_rows + ((size_t)sgi * 2 + 0) * dimp);
    const float4* b = reinterpret_cast<const float4*>(pair_rows + ((size_t)sgi * 2 + 1) * dimp);
    const u32 plane = segs[sgi].plane;
    float4* out = reinterpret_cast<float4*>(coef + (size_t)plane * dimp);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const int chunks = dimp / 16;
    for (int c = 0; c < chunks; ++c) {
        float4 av = a[c * 4 + sub], bv = b[c * 4 + sub];
        float4 cf = make_float4(__fsub_rn(bv.x, av.x), __fsub_rn(bv.y, av.y), __fsub_rn(bv.z, av.z), __fsub_rn(bv.w, av.w));
        float4 mid = make_float4(__fmul_rn(__fadd_rn(av.x, bv.x), 0.5f), __fmul_rn(__fadd_rn(av.y, bv.y), 0.5f),
                                 __fmul_rn(__fadd_rn(av.z, bv.z), 0.5f), __fmul_rn(__fadd_rn(av.w, bv.w), 0.5f));
        out[c * 4 + sub] = cf;
        fma4(acc, cf, mid);
    }
    float d = quad_reduce16(acc, mask);
    if (sub == 0) cst[plane] = -d;
}
void launch_make_planes(const SegDesc* d_segs, u32 nsegs, const float* d_pair_rows, int dimp, float* d_coef,
                        float* d_cst, cudaStream_t s) {
    if (!nsegs) return;
    make_planes_kernel<<<(nsegs + 31) / 32, 128, 0, s>>>(d_segs, nsegs, d_pair_rows, dimp, d_coef, d_cst);
}

// flags[pos] = point_is_above(plane of the segment, row at pos).  Tile = 64 positions, one quad each.
__global__ void __launch_bounds__(256) classify_kernel(const Tile* __restrict__ tiles, const SegDesc* __restrict__ segs,
                                                       const u32* __restrict__ work, const float* __restrict__ rows,
                                                       const float* __restrict__ coef, const float* __restrict__ cst,
                                                       int dimp, u32* __restrict__ flags) {
    const Tile tl = tiles[blockIdx.x];
    const u32 i = threadIdx.x >> 2;
    if (i >= tl.count) return;
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const u32 plane = segs[tl.seg].plane;
    const u32 slot = work[tl.start + i];
    float d = quad_dot(reinterpret_cast<const float4*>(coef + (size_t)plane * dimp),
                       reinterpret_cast<const float4*>(rows + (size_t)slot * dimp), dimp / 16, sub, mask);
    if (sub == 0) flags[tl.start + i] = above_from_dot(d, cst[plane]) ? 1u : 0u;
}
// The projection hot loop as a bandwidth kernel.  Persistent CTAs (128 threads = 32 quads) take tiles of 64 positions;
// one thread gathers the tile's rows into shared memory with one 1-D bulk copy (TMA, UBLKCP) per row -- whole 4N-byte
// rows, the access pattern that reaches HBM speed for gathered rows (profiles/r01_tma_gather_microbench.txt) -- in two
// halves of 32 rows on two mbarriers, so the quads score half 0 while half 1 is still landing.  A quad then reads its
// row from shared memory (padded pitch: the two quads of a quarter-warp hit disjoint banks) and the node's plane
// through L1 (shared by the whole tile), in the canonical chunk order.
#define CL_HALF 32
__global__ void __launch_bounds__(128, 1) classify_rows_kernel(const Tile* __restrict__ tiles, u32 ntiles, const SegDesc* __restrict__ segs,
                                                               const u32* __restrict__ work, const float* __restrict__ rows,
                                                               const float* __restrict__ coef, const float* __restrict__ cst,
                                                               int dimp, int pitch, u32* __restrict__ flags) {
    extern __shared__ __align__(128) unsigned char cl_smem[];
    float* s_rows = reinterpret_cast<float*>(cl_smem);                       // [2][CL_HALF][pitch]
    u64* s_bar = reinterpret_cast<u64*>(s_rows + (size_t)2 * CL_HALF * pitch);  // [2]
    const u32 bar0 = smem_u32(s_bar);
    const int quad = threadIdx.x >> 2, sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    if (threadIdx.x == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const int chunks = dimp / 16;
    const u32 row_bytes = (u32)dimp * 4u;
    u32 phase = 0;
    for (u32 ti = blockIdx.x; ti < ntiles; ti += gridDim.x) {
        const Tile tl = tiles[ti];
        if (threadIdx.x < 2) {  // thread h gathers half h: slots first (independent loads), then the copies
            const int h = threadIdx.x;
            const int cnt = (int)tl.count - h * CL_HALF;
            if (cnt > 0) {
                const int c = cnt < CL_HALF ? cnt : CL_HALF;
                mbar_arrive_expect_tx(bar0 + 8 * h, (u32)c * row_bytes);
                const u32* w = work + tl.start + h * CL_HALF;
                for (int i = 0; i < c; ++i)
                    bulk_g2s(smem_u32(s_rows + ((size_t)h * CL_HALF + i) * pitch), rows + (size_t)w[i] * dimp, row_bytes, bar0 + 8 * h);
            } else {
                mbar_arrive(bar0 + 8 * h);
            }
        }
        const u32 plane = segs[tl.seg].plane;
        const float4* p = reinterpret_cast<const float4*>(coef + (size_t)plane * dimp);
        const float c0 = cst[plane];
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            mbar_wait(bar0 + 8 * h, phase);
            const int i = h * CL_HALF + quad;
            if (i < (int)tl.count) {
                const float4* x = reinterpret_cast<const float4*>(s_rows + ((size_t)h * CL_HALF + quad) * pitch);
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                int c = 0;
                for (; c + 8 <= chunks; c += 8) {
                    float4 p0 = __ldg(p + (c + 0) * 4 + sub), p1 = __ldg(p + (c + 1) * 4 + sub), p2 = __ldg(p + (c + 2) * 4 + sub),
                           p3 = __ldg(p + (c + 3) * 4 + sub), p4 = __ldg(p + (c + 4) * 4 + sub), p5 = __ldg(p + (c + 5) * 4 + sub),
                           p6 = __ldg(p + (c + 6) * 4 + sub), p7 = __ldg(p + (c + 7) * 4 + sub);
                    fma4(acc, p0, x[(c + 0) * 4 + sub]); fma4(acc, p1, x[(c + 1) * 4 + sub]);
                    fma4(acc, p2, x[(c + 2) * 4 + sub]); fma4(acc, p3, x[(c + 3) * 4 + sub]);
                    fma4(acc, p4, x[(c + 4) * 4 + sub]); fma4(acc, p5, x[(c + 5) * 4 + sub]);
                    fma4(acc, p6, x[(c + 6) * 4 + sub]); fma4(acc, p7, x[(c + 7) * 4 + sub]);
                }
                for (; c < chunks; ++c) fma4(acc, __ldg(p + c * 4 + sub), x[c * 4 + sub]);
                const float d = quad_reduce16(acc, mask);
                if (sub == 0) flags[tl.start + i] = above_from_dot(d, c0) ? 1u : 0u;
            }
        }
        phase ^= 1u;
        __syncthreads();  // every quad is done with both halves before the next tile's copies overwrite them
    }
}

void launch_classify(const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work, const float* d_rows,
                     const float* d_coef, const float* d_cst, int dimp, u32* d_flags, int variant, cudaStream_t s) {
    if (!ntiles) return;
    const int pitch = dimp + ((dimp % 32) == 0 ? 16 : 0);
    const size_t smem = (size_t)2 * CL_HALF * pitch * 4 + 16;
    static int sms = 0, max_smem = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaFuncSetAttribute(classify_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
    }
    if (variant == 1 && smem <= (size_t)max_smem) {
        const u32 grid = ntiles < (u32)sms ? ntiles : (u32)sms;
        classify_rows_kernel<<<grid, 128, smem, s>>>(d_tiles, ntiles, d_segs, d_work, d_rows, d_coef, d_cst, dimp, pitch, d_flags);
        return;
    }
    classify_kernel<<<ntiles, 256, 0, s>>>(d_tiles, d_segs, d_work, d_rows, d_coef, d_cst, dimp, d_flags);
}

__global__ void seg_above_kernel(const SegDesc* __restrict__ segs, u32 nsegs, const u32* __restrict__ scan,
                                 u32* __restrict__ above) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsegs) return;
    above[i] = scan[segs[i].off + segs[i].len] - scan[segs[i].off];
}
void launch_seg_above(const SegDesc* d_segs, u32 nsegs, const u32* d_scan, u32* d_above, cudaStream_t s) {
    if (!nsegs) return;
    seg_above_kernel<<<(nsegs + 255) / 256, 256, 0, s>>>(d_segs, nsegs, d_scan, d_above);
}

__global__ void __launch_bounds__(64) scatter_kernel(const Tile* __restrict__ tiles, const SegDesc* __restrict__ segs,
                                                     const u32* __restrict__ work_in, const u32* __restrict__ flags,
                                                     const u32* __restrict__ scan, u32* __restrict__ work_out) {
    const Tile tl = tiles[blockIdx.x];
    if (threadIdx.x >= tl.count) return;
    const SegDesc sg = segs[tl.seg];
    const long long pos = tl.start + threadIdx.x;
    const u32 above_rank = scan[pos] - scan[sg.off];
    const u32 n_above = scan[sg.off + sg.len] - scan[sg.off];
    const u32 n_below = sg.len - n_above;
    const u32 local = (u32)(pos - sg.off);
    const long long dst = flags[pos] ? sg.off + n_below + above_rank : sg.off + (local - above_rank);
    work_out[dst] = work_in[pos];
}
void launch_scatter(const Tile* d_tiles, u32 ntiles, const SegDesc* d_segs, const u32* d_work_in, const u32* d_flags,
                    const u32* d_scan, u32* d_work_out, cudaStream_t s) {
    if (!ntiles) return;
    scatter_kernel<<<ntiles, 64, 0, s>>>(d_tiles, d_segs, d_work_in, d_flags, d_scan, d_work_out);
}

// slot_leaf[slot] = leaf, for the members of the tiled leaves of ONE tree.
__global__ void __launch_bounds__(64) assign_leaf_kernel(const Tile* __restrict__ tiles, const u32* __restrict__ members,
                                                         u32* __restrict__ slot_leaf) {
    const Tile tl = tiles[blockIdx.x];
    if (threadIdx.x >= tl.count) return;
    slot_leaf[members[tl.start + threadIdx.x]] = tl.seg;
}
void launch_assign_leaf(const Tile* d_tiles, u32 ntiles, const u32* d_members, u32* d_slot_leaf_tree, cudaStream_t s) {
    if (!ntiles) return;
    assign_leaf_kernel<<<ntiles, 64, 0, s>>>(d_tiles, d_members, d_slot_leaf_tree);
}

// =====================================================================================================
// mutation
// =====================================================================================================
// LSHIndex::remove under D1: set the tombstone bit, take the row out of every tree's live leaf count.
__global__ void tombstone_kernel(const u32* __restrict__ slots, u32 n, u32* __restrict__ tomb,
                                 const u32* __restrict__ slot_leaf, u64 slot_stride, int num_trees,
                                 u32* __restrict__ leaf_live, u8* __restrict__ removed) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 slot = slots[i];
    if (slot == 0xFFFFFFFFu) { removed[i] = 0; return; }
    u32 bit = 1u << (slot & 31);
    u32 old = atomicOr(&tomb[slot >> 5], bit);
    if (old & bit) { removed[i] = 0; return; }
    removed[i] = 1;
    for (int t = 0; t < num_trees; ++t) atomicSub(&leaf_live[slot_leaf[(u64)t * slot_stride + slot]], 1u);
}
void launch_tombstone(const u32* d_slots, u32 n, u32* d_tomb, const u32* d_slot_leaf, u64 slot_stride, int num_trees,
                      u32* d_leaf_live, u8* d_removed, cudaStream_t s) {
    if (!n) return;
    tombstone_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_slots, n, d_tomb, d_slot_leaf, slot_stride, num_trees, d_leaf_live,
                                                     d_removed);
}

// Bucket-major store: bm_rows[p] = rows[members[p]] for every position p of every leaf (one block per leaf), plus
// the position of each slot in each tree (slot_pos, for tombstoning) and the position-major tombstone bitmap.
__global__ void __launch_bounds__(256) bm_gather_kernel(const long long* __restrict__ leaf_off, const u32* __restrict__ leaf_len,
                                                        const u32* __restrict__ leaf_tree, const u32* __restrict__ members,
                                                        const float* __restrict__ rows, const u32* __restrict__ tomb, int dimp,
                                                        u64 slot_stride, float* __restrict__ bm_rows,
                                                        u32* __restrict__ slot_pos, u32* __restrict__ bm_tomb) {
    const u32 leaf = blockIdx.x;
    const long long off = leaf_off[leaf];
    const u32 len = leaf_len[leaf], tree = leaf_tree[leaf];
    const int q4 = dimp / 4;
    for (u32 i = 0; i < len; ++i) {
        const u32 slot = members[off + i];
        const float4* src = reinterpret_cast<const float4*>(rows + (size_t)slot * dimp);
        float4* dst = reinterpret_cast<float4*>(bm_rows + (size_t)(off + i) * dimp);
        for (int c = threadIdx.x; c < q4; c += blockDim.x) dst[c] = __ldg(src + c);
        if (threadIdx.x == 0) {
            const u64 pos = (u64)(off + i);
            slot_pos[(u64)tree * slot_stride + slot] = (u32)pos;
            if (tomb_test(tomb, slot)) atomicOr(&bm_tomb[pos >> 5], 1u << (pos & 31));
        }
    }
}
void launch_bm_gather(u32 nleaves, const long long* d_leaf_off, const u32* d_leaf_len, const u32* d_leaf_tree, const u32* d_members,
                      const float* d_rows, const u32* d_tomb, int dimp, u64 slot_stride, float* d_bm_rows, u32* d_slot_pos,
                      u32* d_bm_tomb, cudaStream_t s) {
    if (!nleaves) return;
    bm_gather_kernel<<<nleaves, 256, 0, s>>>(d_leaf_off, d_leaf_len, d_leaf_tree, d_members, d_rows, d_tomb, dimp, slot_stride,
                                             d_bm_rows, d_slot_pos, d_bm_tomb);
}
// position-major tombstones of freshly removed slots (flags[i] != 0): one bit per tree
__global__ void bm_tombstone_kernel(const u32* __restrict__ slots, const u8* __restrict__ flags, u32 n,
                                    const u32* __restrict__ slot_pos, u64 slot_stride, int num_trees, u32* __restrict__ bm_tomb) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flags[i] || slots[i] == 0xFFFFFFFFu) return;
    for (int t = 0; t < num_trees; ++t) {
        const u32 pos = slot_pos[(u64)t * slot_stride + slots[i]];
        atomicOr(&bm_tomb[pos >> 5], 1u << (pos & 31));
    }
}
void launch_bm_tombstone(const u32* d_slots, const u8* d_flags, u32 n, const u32* d_slot_pos, u64 slot_stride, int num_trees,
                         u32* d_bm_tomb, cudaStream_t s) {
    if (!n) return;
    bm_tombstone_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_slots, d_flags, n, d_slot_pos, slot_stride, num_trees, d_bm_tomb);
}

__global__ void pad_rows_kernel(const float* __restrict__ src, u64 n, int dim, int dimp, float* __restrict__ dst) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * (u64)dimp) return;
    u64 r = i / dimp;
    int c = (int)(i - r * dimp);
    dst[i] = c < dim ? src[r * dim + c] : 0.0f;
}
void launch_pad_rows(const float* d_src, u64 n, int dim, int dimp, float* d_dst, cudaStream_t s) {
    u64 tot = n * (u64)dimp;
    if (!tot) return;
    pad_rows_kernel<<<(u32)((tot + 255) / 256), 256, 0, s>>>(d_src, n, dim, dimp, d_dst);
}

__global__ void fill_u64_kernel(u64* d, u64 n, u64 v) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = v;
}
void launch_fill_u64(u64* d, u64 n, u64 v, cudaStream_t s) {
    if (!n) return;
    fill_u64_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d, n, v);
}
__global__ void iota_ord_kernel(u64* d, u64 n, u64 first, u64 stride) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = first + i * stride;
}
void launch_iota_ord(u64* d, u64 n, u64 first, u64 stride, cudaStream_t s) {
    if (!n) return;
    iota_ord_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d, n, first, stride);
}

// =====================================================================================================
// synthetic data (BASELINE.md): Philox-4x32-10, counter = (row_lo, row_hi, col/4, stream), key = seed;
// word -> f32 exactly: x = float((int32)w >> 8) * 2^-23 in [-1, 1).  No transcendental functions.
// =====================================================================================================
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const u32 M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        u32 hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        u32 hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float word_to_unit(u32 w) { return (float)((int)w >> 8) * 1.1920928955078125e-07f; }

__global__ void synth_kernel(float* __restrict__ out, u64 first_row, u64 row_stride, u64 n, u32 dim, u64 seed, u32 kind) {
    const u32 quads = (dim + 3) / 4;
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * (u64)quads) return;
    u64 ri = i / quads;
    u32 cq = (u32)(i - ri * quads);
    u64 row = first_row + ri * row_stride;
    uint2 key = make_uint2((u32)seed, (u32)(seed >> 32));
    uint4 w = philox4x32_10(make_uint4((u32)row, (u32)(row >> 32), cq, 0u), key);
    float v[4] = {word_to_unit(w.x), word_to_unit(w.y), word_to_unit(w.z), word_to_unit(w.w)};
    if (kind == 1) {
        u64 crow = row % 4096ull;
        uint4 c = philox4x32_10(make_uint4((u32)crow, 0u, cq, 1u), key);
        float cv[4] = {word_to_unit(c.x), word_to_unit(c.y), word_to_unit(c.z), word_to_unit(c.w)};
        for (int j = 0; j < 4; ++j) v[j] = __fmaf_rn(0.25f, v[j], cv[j]);
    }
    for (int j = 0; j < 4; ++j) {
        u32 col = cq * 4 + j;
        if (col < dim) out[ri * dim + col] = v[j];
    }
}
void launch_synth(float* d_out, u64 first_row, u64 row_stride, u64 n, u32 dim, u64 seed, u32 kind, cudaStream_t s) {
    u64 tot = n * (u64)((dim + 3) / 4);
    if (!tot) return;
    synth_kernel<<<(u32)((tot + 255) / 256), 256, 0, s>>>(d_out, first_row, row_stride, n, dim, seed, kind);
}


// =====================================================================================================
// element-wise entry points of the metric trait and of point_is_above (arithmetic parity tests; the
// Metric::distance of distance.rs:19-49,:103-114 and Hyperplane::point_is_above of lsh.rs:39-43 for
// n independent pairs).  One quad per pair.
// =====================================================================================================
// squared norms in the canonical order (the a2 / b2 accumulators of simsimd's cos kernel): one quad per vector
__global__ void __launch_bounds__(128) sq_norms_kernel(const float* __restrict__ x_, u64 n, int dimp, float* __restrict__ out) {
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
void launch_sq_norms(const float* d_x, u64 n, int dimp, float* d_out, cudaStream_t s) {
    if (!n) return;
    sq_norms_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_x, n, dimp, d_out);
}

template <int METRIC>
__global__ void __launch_bounds__(128) pair_metric_kernel(const float* __restrict__ a_, const float* __restrict__ b_, u64 n,
                                                          int dimp, u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const float4* a = reinterpret_cast<const float4*>(a_ + i * dimp);
    const float4* b = reinterpret_cast<const float4*>(b_ + i * dimp);
    const int chunks = dimp / 16;
    u64 key;
    if (METRIC == 0) {
        float4 ab = make_float4(0.f, 0.f, 0.f, 0.f), a2 = ab, b2 = ab;
        for (int c = 0; c < chunks; ++c) {
            float4 av = a[c * 4 + sub], bv = b[c * 4 + sub];
            fma4(ab, av, bv);
            fma4(a2, av, av);
            fma4(b2, bv, bv);
        }
        key = cos_bits(quad_reduce16(ab, mask), quad_reduce16(a2, mask), quad_reduce16(b2, mask));
    } else {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c = 0; c < chunks; ++c) l2acc4(acc, a[c * 4 + sub], b[c * 4 + sub]);
        float sum = quad_reduce16(acc, mask);
        key = METRIC == 1 ? l2sq_bits(sum) : l2_bits(sum);
    }
    if (sub == 0) out[i] = key;
}
template <int CODE>
__global__ void __launch_bounds__(128) pair_metric_seq_kernel(const float* __restrict__ a, const float* __restrict__ b, u64 n,
                                                              int dim, int dimp, int power, u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * 128ull + threadIdx.x;
    if (i >= n) return;
    out[i] = seq_distance_ldg<CODE>(a + i * dimp, b + i * dimp, dim, power);
}
void launch_pair_metric(int metric, int power, const float* d_a, const float* d_b, u64 n, int dim, int dimp, u64* d_out,
                        cudaStream_t s) {
    if (!n) return;
    if (metric > M_L2) {
        const u32 sblocks = (u32)((n + 127) / 128);
#define ZB_CALL(C) pair_metric_seq_kernel<C><<<sblocks, 128, 0, s>>>(d_a, d_b, n, dim, dimp, power, d_out)
        ZB_SEQ_DISPATCH(metric, ZB_CALL)
#undef ZB_CALL
        return;
    }
    u32 blocks = (u32)((n + 31) / 32);
    if (metric == 0) pair_metric_kernel<0><<<blocks, 128, 0, s>>>(d_a, d_b, n, dimp, d_out);
    else if (metric == 1) pair_metric_kernel<1><<<blocks, 128, 0, s>>>(d_a, d_b, n, dimp, d_out);
    else pair_metric_kernel<2><<<blocks, 128, 0, s>>>(d_a, d_b, n, dimp, d_out);
}
__global__ void __launch_bounds__(128) pair_above_kernel(const float* __restrict__ coef, const float* __restrict__ cst,
                                                         const float* __restrict__ x, u64 n, int dimp, u8* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    float d = quad_dot(reinterpret_cast<const float4*>(coef + i * dimp), reinterpret_cast<const float4*>(x + i * dimp),
                       dimp / 16, sub, quad_mask());
    if (sub == 0) out[i] = above_from_dot(d, cst[i]) ? 1 : 0;
}
void launch_pair_above(const float* d_coef, const float* d_cst, const float* d_x, u64 n, int dimp, u8* d_out, cudaStream_t s) {
    if (!n) return;
    pair_above_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_coef, d_cst, d_x, n, dimp, d_out);
}


// =====================================================================================================
// bucket-sharded store (G > 1): leaf l lives, whole, on rank l % G.  The raw row store stays sharded by
// ordinal (build / insert / delete bookkeeping); these kernels move each leaf's rows to its owner once per
// forest change and keep the position-major tombstones in step with deletes.
// =====================================================================================================
// sender: out_rows[i] = rows[slots[i]], out_key[i] = ordinal | tombstone << 63 (one warp per row)
__global__ void __launch_bounds__(256) pack_rows_kernel(const u32* __restrict__ slots, u64 n, const float* __restrict__ rows,
                                                        const u64* __restrict__ ord, const u32* __restrict__ tomb, int dimp,
                                                        float* __restrict__ out_rows, u64* __restrict__ out_key) {
    const u64 i = (u64)blockIdx.x * 8ull + (threadIdx.x >> 5);
    if (i >= n) return;
    const int lane = threadIdx.x & 31;
    const u32 slot = slots[i];
    const float4* src = reinterpret_cast<const float4*>(rows + (size_t)slot * dimp);
    float4* dst = reinterpret_cast<float4*>(out_rows + (size_t)i * dimp);
    for (int c = lane; c < dimp / 4; c += 32) dst[c] = __ldg(src + c);
    if (lane == 0) out_key[i] = ord[slot] | (tomb_test(tomb, slot) ? (1ull << 63) : 0ull);
}
void launch_pack_rows(const u32* d_slots, u64 n, const float* d_rows, const u64* d_ord, const u32* d_tomb, int dimp,
                      float* d_out_rows, u64* d_out_key, cudaStream_t s) {
    if (!n) return;
    pack_rows_kernel<<<(u32)((n + 7) / 8), 256, 0, s>>>(d_slots, n, d_rows, d_ord, d_tomb, dimp, d_out_rows, d_out_key);
}
// receiver: element i of segment (source rank, leaf) gets sort key (leaf sequence number << 40) | ordinal, so that the
// sorted order is leaf-major and ordinal-ascending inside a leaf (position order == ordinal order, D3)
__global__ void __launch_bounds__(128) seg_keys_kernel(const RecvSeg* __restrict__ segs, const u64* __restrict__ st_key,
                                                       u64* __restrict__ sort_key, u32* __restrict__ sort_val) {
    const RecvSeg sg = segs[blockIdx.x];
    for (u32 j = threadIdx.x; j < sg.count; j += blockDim.x) {
        const u64 i = sg.start + j;
        sort_key[i] = ((u64)sg.leaf_seq << 40) | (st_key[i] & ((1ull << 40) - 1));
        sort_val[i] = (u32)i;
    }
}
void launch_seg_keys(const RecvSeg* d_segs, u32 nsegs, const u64* d_st_key, u64* d_sort_key, u32* d_sort_val, cudaStream_t s) {
    if (!nsegs) return;
    seg_keys_kernel<<<nsegs, 128, 0, s>>>(d_segs, d_st_key, d_sort_key, d_sort_val);
}
// position base + p of the bucket-major store receives staging element perm[p] (one warp per row)
__global__ void __launch_bounds__(256) place_rows_kernel(const u32* __restrict__ perm, u64 n, const float* __restrict__ st_rows,
                                                         const u64* __restrict__ st_key, int dimp, u64 base,
                                                         float* __restrict__ bm_rows, u64* __restrict__ bm_ord,
                                                         u32* __restrict__ bm_tomb) {
    const u64 p = (u64)blockIdx.x * 8ull + (threadIdx.x >> 5);
    if (p >= n) return;
    const int lane = threadIdx.x & 31;
    const u32 src_i = perm[p];
    const float4* src = reinterpret_cast<const float4*>(st_rows + (size_t)src_i * dimp);
    float4* dst = reinterpret_cast<float4*>(bm_rows + (size_t)(base + p) * dimp);
    for (int c = lane; c < dimp / 4; c += 32) dst[c] = src[c];
    if (lane == 0) {
        const u64 k = st_key[src_i];
        bm_ord[base + p] = k & ~(1ull << 63);
        if (k >> 63) atomicOr(&bm_tomb[(base + p) >> 5], 1u << ((base + p) & 31));
    }
}
void launch_place_rows(const u32* d_perm, u64 n, const float* d_st_rows, const u64* d_st_key, int dimp, u64 base,
                       float* d_bm_rows, u64* d_bm_ord, u32* d_bm_tomb, cudaStream_t s) {
    if (!n) return;
    place_rows_kernel<<<(u32)((n + 7) / 8), 256, 0, s>>>(d_perm, n, d_st_rows, d_st_key, dimp, base, d_bm_rows, d_bm_ord, d_bm_tomb);
}
__global__ void iota_u32_kernel(u32* d, u64 n, u32 first) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = first + (u32)i;
}
void launch_iota_u32(u32* d, u64 n, u32 first, cudaStream_t s) {
    if (!n) return;
    iota_u32_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d, n, first);
}
// delete on a bucket-sharded store: every rank sees the whole batch; for each removed ordinal and each tree, find the
// row's position (if its leaf lives here) in the tree's ordinal-sorted index and set the position-major tombstone bit
__global__ void bm_tomb_lookup_kernel(const u64* __restrict__ ords, const u8* __restrict__ flags, u64 n, int num_trees,
                                      const u64* __restrict__ tree_base, const u64* __restrict__ srt_ord,
                                      const u32* __restrict__ srt_pos, u32* __restrict__ bm_tomb) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * (u64)num_trees) return;
    const u64 r = i / (u64)num_trees;
    const int t = (int)(i - r * (u64)num_trees);
    if (!flags[r]) return;
    const u64 o = ords[r];
    u64 lo = tree_base[t], hi = tree_base[t + 1];
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if (srt_ord[mid] < o) lo = mid + 1; else hi = mid;
    }
    if (lo < tree_base[t + 1] && srt_ord[lo] == o) {
        const u32 pos = srt_pos[lo];
        atomicOr(&bm_tomb[pos >> 5], 1u << (pos & 31));
    }
}
void launch_bm_tomb_lookup(const u64* d_ords, const u8* d_flags, u64 n, int num_trees, const u64* d_tree_base,
                           const u64* d_srt_ord, const u32* d_srt_pos, u32* d_bm_tomb, cudaStream_t s) {
    const u64 tot = n * (u64)num_trees;
    if (!tot) return;
    bm_tomb_lookup_kernel<<<(u32)((tot + 255) / 256), 256, 0, s>>>(d_ords, d_flags, n, num_trees, d_tree_base, d_srt_ord, d_srt_pos, d_bm_tomb);
}
// final merge of the ranks' per-query local top-k lists (each rank: [ord nq*k | bits nq*k]): union, dedup by id (the same
// row can be reached through trees whose leaves live on different ranks), sort (bits, id), take top_k (lsh.rs:550,:561-564)
struct GatheredLoader {
    const u64* g;
    u64 per_rank, bits_off, qbase;
    u32 k;
    __device__ Entry operator()(long long i) const {
        const u64 r = (u64)i / k, j = (u64)i % k;
        const u64* b = g + r * per_rank + qbase + j;
        return Entry{b[bits_off], b[0]};
    }
};
// gathered: per source rank one block [ord nslice*k | bits nslice*k] holding that rank's local top-k lists of the nslice
// queries this rank finishes; out_*: [nslice][k] / [nslice]
__global__ void __launch_bounds__(TOPK_THREADS) merge_gathered_kernel(u32 nq, u32 nslice, u32 top_k, u32 nranks,
                                                                      const u64* __restrict__ gathered, u64* __restrict__ out_ord,
                                                                      u64* __restrict__ out_bits, u32* __restrict__ out_counts,
                                                                      int pmax, int kmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    Entry* buf = reinterpret_cast<Entry*>(smem);
    Entry* keep = buf + pmax;
    int* s_warp = reinterpret_cast<int*>(keep + kmax);
    const u32 q = blockIdx.x;
    if (q >= nq) return;
    const u64 nsk = (u64)nslice * top_k;
    GatheredLoader ld{gathered, 2 * nsk, nsk, (u64)q * top_k, top_k};
    int kept = segment_topk(buf, keep, s_warp, ld, (long long)top_k * nranks, (int)top_k, pmax);
    for (u32 i = threadIdx.x; i < top_k; i += TOPK_THREADS) {
        bool ok = (int)i < kept;
        out_ord[(size_t)q * top_k + i] = ok ? keep[i].ord : ZB_SENTINEL;
        out_bits[(size_t)q * top_k + i] = ok ? keep[i].key : ZB_SENTINEL;
    }
    if (threadIdx.x == 0) out_counts[q] = (u32)kept;
}
void launch_merge_gathered(u32 nq, u32 nslice, u32 top_k, u32 nranks, const u64* d_gathered, u64* d_out_ord, u64* d_out_bits,
                           u32* d_out_counts, cudaStream_t s) {
    if (!nq || !top_k) return;
    int pmax = topk_pmax(top_k), kmax = (int)top_k;
    size_t smem = topk_smem(pmax, kmax);
    set_smem(merge_gathered_kernel, smem);
    merge_gathered_kernel<<<nq, TOPK_THREADS, smem, s>>>(nq, nslice, top_k, nranks, d_gathered, d_out_ord, d_out_bits, d_out_counts,
                                                         pmax, kmax);
}
// results of all slices ([G] blocks of [ord nslice*k | bits nslice*k | counts nslice (u32)], block = blk u64) -> caller's arrays
__global__ void unpack_results_kernel(const u64* __restrict__ res, u64 blk, u32 nq, u32 nslice, u32 top_k, u64* __restrict__ out_ord,
                                      u64* __restrict__ out_bits, u32* __restrict__ out_counts) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (u64)nq * top_k) return;
    const u32 q = (u32)(i / top_k), j = (u32)(i - (u64)q * top_k);
    const u32 r = q / nslice, ql = q - r * nslice;
    const u64* b = res + (u64)r * blk;
    const u64 nsk = (u64)nslice * top_k;
    out_ord[i] = b[(u64)ql * top_k + j];
    out_bits[i] = b[nsk + (u64)ql * top_k + j];
    if (j == 0) out_counts[q] = reinterpret_cast<const u32*>(b + 2 * nsk)[ql];
}
void launch_unpack_results(const u64* d_res, u64 blk, u32 nq, u32 nslice, u32 top_k, u64* d_out_ord, u64* d_out_bits,
                           u32* d_out_counts, cudaStream_t s) {
    const u64 tot = (u64)nq * top_k;
    if (!tot) return;
    unpack_results_kernel<<<(u32)((tot + 255) / 256), 256, 0, s>>>(d_res, blk, nq, nslice, top_k, d_out_ord, d_out_bits, d_out_counts);
}


// =====================================================================================================
// deduplicate (lsh.rs:270-288): rows whose BIT patterns are equal; the row with the smallest id of each group stays.
// hash every live row (128 bits, one quad per row, the row is read once) -> radix sort by hash (stable: candidates keep
// id order) -> run heads by a max-scan -> every non-head row is compared, bit for bit, with the earlier rows of its run.
// =====================================================================================================
__global__ void __launch_bounds__(128) row_hash_kernel(const u32* __restrict__ slots, u64 n, const float* __restrict__ rows, int dimp,
                                                       u64* __restrict__ h1, u64* __restrict__ h2) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const uint4* x = reinterpret_cast<const uint4*>(rows + (size_t)slots[i] * dimp);
    u64 a = 0x243F6A8885A308D3ull + sub, b = 0x13198A2E03707344ull + sub;
    for (int c = 0; c < dimp / 16; ++c) {
        const uint4 v = __ldg(x + c * 4 + sub);
        const u64 lo = ((u64)v.y << 32) | v.x, hi = ((u64)v.w << 32) | v.z;
        a = mix64(a ^ lo); a = mix64(a ^ hi);
        b = mix64(b + lo) ^ hi; b = mix64(b);
    }
    // fold the quad in a fixed order
#pragma unroll
    for (int m = 1; m <= 2; m <<= 1) {
        const u64 oa = ((u64)__shfl_xor_sync(mask, (u32)(a >> 32), m) << 32) | __shfl_xor_sync(mask, (u32)a, m);
        const u64 ob = ((u64)__shfl_xor_sync(mask, (u32)(b >> 32), m) << 32) | __shfl_xor_sync(mask, (u32)b, m);
        const bool low = (sub & m) == 0;
        a = mix64((low ? a : oa) ^ mix64(low ? oa : a));
        b = mix64((low ? b : ob) + mix64(low ? ob : b));
    }
    if (sub == 0) {
        h1[i] = a;
        if (h2) h2[i] = b;
    }
}
void launch_row_hash(const u32* d_slots, u64 n, const float* d_rows, int dimp, u64* d_h1, u64* d_h2, cudaStream_t s) {
    if (!n) return;
    row_hash_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_slots, n, d_rows, dimp, d_h1, d_h2);
}
__global__ void run_flag_kernel(const u64* __restrict__ key, u64 n, u32* __restrict__ flag) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (i == 0 || key[i] != key[i - 1]) ? (u32)i : 0u;
}
// one quad per sorted candidate: duplicate iff an earlier candidate of the same hash run has identical bits
__global__ void __launch_bounds__(128) dup_mark_kernel(const u32* __restrict__ head, const u32* __restrict__ cand, u64 n,
                                                       const u32* __restrict__ slots, const float* __restrict__ rows, int dimp,
                                                       u8* __restrict__ dup) {
    const u64 i = (u64)blockIdx.x * 32ull + (threadIdx.x >> 2);
    if (i >= n) return;
    const int sub = threadIdx.x & 3;
    const unsigned mask = quad_mask();
    const u32 h = head[i];
    u8 is_dup = 0;
    const uint4* me = reinterpret_cast<const uint4*>(rows + (size_t)slots[cand[i]] * dimp);
    for (u32 j = h; j < (u32)i && !is_dup; ++j) {
        const uint4* other = reinterpret_cast<const uint4*>(rows + (size_t)slots[cand[j]] * dimp);
        bool eq = true;
        for (int c = 0; c < dimp / 16 && eq; ++c) {
            const uint4 u = __ldg(me + c * 4 + sub), v = __ldg(other + c * 4 + sub);
            const bool same = u.x == v.x && u.y == v.y && u.z == v.z && u.w == v.w;
            eq = __all_sync(mask, same);
        }
        if (eq) is_dup = 1;
    }
    if (sub == 0) dup[i] = is_dup;
}
void launch_dup_mark(const u64* d_sorted_key, const u32* d_cand, u64 n, const u32* d_slots, const float* d_rows, int dimp,
                     u32* d_flag, u32* d_head, void* d_temp, size_t temp_bytes, u8* d_dup, cudaStream_t s) {
    if (!n) return;
    run_flag_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d_sorted_key, n, d_flag);
    cub::DeviceScan::InclusiveScan(d_temp, temp_bytes, d_flag, d_head, cub::Max(), (long long)n, s);
    dup_mark_kernel<<<(u32)((n + 31) / 32), 128, 0, s>>>(d_head, d_cand, n, d_slots, d_rows, dimp, d_dup);
}
size_t maxscan_temp_bytes(size_t n) {
    size_t b = 0;
    cub::DeviceScan::InclusiveScan(nullptr, b, (const u32*)nullptr, (u32*)nullptr, cub::Max(), (long long)n);
    return b + 256;
}

// =====================================================================================================
// rowsets (restricted search, DESIGN 3.10): a bitmap over global ordinals, and the masks a restricted search substitutes
// for the tombstones
// =====================================================================================================
__global__ void rowset_scatter_kernel(const u64* __restrict__ ords, u64 n, u64 nbits, u32* __restrict__ bits, u32* __restrict__ bad) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 o = ords[i];
    if (o >= nbits) {
        atomicOr(bad, 1u);
        return;
    }
    atomicOr(&bits[o >> 5], 1u << (o & 31));
}
void launch_rowset_scatter(const u64* d_ords, u64 n, u64 nbits, u32* d_bits, u32* d_bad, cudaStream_t s) {
    if (!n) return;
    rowset_scatter_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d_ords, n, nbits, d_bits, d_bad);
}
// exclude mode: complement over [0, nbits); bits at or above nbits are cleared either way; count += members of the set
__global__ void rowset_finish_kernel(u32* __restrict__ bits, u64 nbits, u64 words, u32 invert, u64* __restrict__ count) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 c = 0;
    if (w < words) {
        u32 v = invert ? ~bits[w] : bits[w];
        const u64 lo = w * 32;
        if (lo >= nbits) v = 0;
        else if (nbits - lo < 32) v &= (1u << (nbits - lo)) - 1u;
        bits[w] = v;
        c = __popc(v);
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, (u64)c);
}
void launch_rowset_finish(u32* d_bits, u64 nbits, u64 words, u32 invert, u64* d_count, cudaStream_t s) {
    if (!words) return;
    rowset_finish_kernel<<<(u32)((words + 255) / 256), 256, 0, s>>>(d_bits, nbits, words, invert, d_count);
}
// out bit p (p < 32 * words) = removed for a restricted search: p >= n, or own bit p set (the tombstones, when given), or the
// bit of key[p] in `bits` says so (bits_dead = 0: `bits` is the rowset, a clear or out-of-range bit excludes; bits_dead = 1:
// `bits` is a mask of removed positions).  live += positions left in.
template <class K>
__global__ void rowset_mask_kernel(const K* __restrict__ key, u64 n, const u32* __restrict__ own, const u32* __restrict__ bits,
                                   u64 nbits, u32 bits_dead, u64 words, u32* __restrict__ out, u64* __restrict__ live) {
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool dead = true;
    if (p < n) {
        const u64 k = key[p];
        const bool b = k < nbits && ((bits[k >> 5] >> (k & 31)) & 1u);
        dead = (own && tomb_test(own, (u32)p)) || (b == (bits_dead != 0));
    }
    const u32 w = __ballot_sync(0xFFFFFFFFu, dead);
    if ((threadIdx.x & 31) == 0 && (p >> 5) < words) {
        out[p >> 5] = w;
        if (live && ~w) atomicAdd(live, (u64)__popc(~w));
    }
}
void launch_rowset_mask(const u64* d_key, u64 n, const u32* d_own, const u32* d_bits, u64 nbits, u32 bits_dead, u64 words, u32* d_out,
                        u64* d_live, cudaStream_t s) {
    if (!words) return;
    rowset_mask_kernel<u64><<<(u32)((words * 32 + 255) / 256), 256, 0, s>>>(d_key, n, d_own, d_bits, nbits, bits_dead, words, d_out, d_live);
}
void launch_rowset_mask(const u32* d_key, u64 n, const u32* d_own, const u32* d_bits, u64 nbits, u32 bits_dead, u64 words, u32* d_out,
                        u64* d_live, cudaStream_t s) {
    if (!words) return;
    rowset_mask_kernel<u32><<<(u32)((words * 32 + 255) / 256), 256, 0, s>>>(d_key, n, d_own, d_bits, nbits, bits_dead, words, d_out, d_live);
}
// compaction of the positions a mask leaves in, ascending: per-word counts, (exclusive scan), then every position's rank
__global__ void rowset_word_live_kernel(const u32* __restrict__ mask, u64 words, u32* __restrict__ out) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < words) out[w] = __popc(~mask[w]);
}
void launch_rowset_word_live(const u32* d_mask, u64 words, u32* d_out, cudaStream_t s) {
    if (!words) return;
    rowset_word_live_kernel<<<(u32)((words + 255) / 256), 256, 0, s>>>(d_mask, words, d_out);
}
__global__ void rowset_compact_kernel(const u32* __restrict__ mask, u64 n, const u32* __restrict__ woff, u32* __restrict__ out) {
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const u32 m = ~mask[p >> 5], b = (u32)(p & 31);
    if ((m >> b) & 1u) out[woff[p >> 5] + __popc(m & ((1u << b) - 1u))] = (u32)p;
}
void launch_rowset_compact(const u32* d_mask, u64 n, const u32* d_woff, u32* d_out, cudaStream_t s) {
    if (!n) return;
    rowset_compact_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(d_mask, n, d_woff, d_out);
}

// =====================================================================================================
// cub scans / sorts
// =====================================================================================================
size_t scan_temp_bytes(size_t n) {
    size_t b32 = 0, b64 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, b32, (const u32*)nullptr, (u32*)nullptr, (long long)n);
    cub::DeviceScan::ExclusiveSum(nullptr, b64, (const u64*)nullptr, (u64*)nullptr, (long long)n);
    return (b32 > b64 ? b32 : b64) + 256;
}
void exclusive_scan_u32(void* d_temp, size_t temp_bytes, const u32* d_in, u32* d_out, size_t n, cudaStream_t s) {
    if (!n) return;
    cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_in, d_out, (long long)n, s);
}
void exclusive_scan_u64(void* d_temp, size_t temp_bytes, const u64* d_in, u64* d_out, size_t n, cudaStream_t s) {
    if (!n) return;
    cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_in, d_out, (long long)n, s);
}

size_t sort_temp_bytes(size_t n) {
    size_t b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b, (const u64*)nullptr, (u64*)nullptr, (const u32*)nullptr, (u32*)nullptr, (long long)n);
    return b + 256;
}
void sort_pairs_u64_u32(void* d_temp, size_t temp_bytes, const u64* d_kin, u64* d_kout, const u32* d_vin, u32* d_vout, size_t n,
                        int end_bit, cudaStream_t s) {
    if (!n) return;
    cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, d_kin, d_kout, d_vin, d_vout, (long long)n, 0, end_bit, s);
}

}  // namespace zb
