// rowset_mirror_test.cpp -- TEST INFRASTRUCTURE.  Drives the restricted search of the C++ host mirror (include/zebra_b200.hpp:
// LSHIndex::rowset / rowset_ordinals, search_batch and search_exact `within` a RowSet) on a B200 and checks it bit for bit:
//   - the LSH search within a rowset against the CPU oracle (oracle/zb_oracle.c) loaded with the same rows, the complement of
//     the set removed;
//   - the exact search within a rowset against a brute force over the set's live rows (zbo_distance_bits, (bits, ordinal)).
//   rowset_mirror_test gpu
#include <algorithm>
#include <cstdio>
#include <map>
#include <string>

#include "../../include/zebra_b200.hpp"

extern "C" {  // the oracle's C entry points (oracle/zb_oracle.c)
struct zbo_index;
zbo_index* zbo_create(int dim, int metric, uint64_t max_node_size, int num_trees, uint64_t seed);
void zbo_destroy(zbo_index* ix);
int zbo_add(zbo_index* ix, uint64_t n, const float* rows, uint64_t* out_ids);
int zbo_remove(zbo_index* ix, uint64_t n, const uint64_t* ids, uint8_t* out_removed);
int zbo_search_batch(const zbo_index* ix, uint64_t nq, const float* queries, uint64_t top_k, int nthreads, uint64_t* out_ids,
                     uint64_t* out_bits, uint32_t* out_counts);
uint64_t zbo_distance_bits(int metric, const float* row, const float* query, int n);
}

using namespace zebra;
constexpr size_t N = 64;
static int failures = 0;
static uint64_t lcg_state = 4242;
static float frand() {  // uniform in [-1, 1), exact in f32
    lcg_state = lcg_state * 6364136223846793005ull + 1442695040888963407ull;
    return (float)((int32_t)(lcg_state >> 32) >> 8) * (1.0f / 8388608.0f);
}
static void report(const char* tag, bool ok) {
    std::printf("[cpp rowset] %s: %s\n", tag, ok ? "ok" : "MISMATCH");
    if (!ok) ++failures;
}
using Results = std::vector<std::vector<std::pair<Uuid, DistanceUnit>>>;
static bool same(const Results& got, const std::map<Uuid, uint64_t>& ordinal_of, const std::vector<uint64_t>& eo,
                 const std::vector<uint64_t>& eb, const std::vector<uint32_t>& ec, size_t k) {
    for (size_t q = 0; q < got.size(); ++q) {
        if (got[q].size() != ec[q]) return false;
        for (size_t i = 0; i < ec[q]; ++i)
            if (ordinal_of.at(got[q][i].first) != eo[q * k + i] || got[q][i].second != eb[q * k + i]) return false;
    }
    return true;
}

static int run_gpu() {
    const size_t n = 3000, nq = 64, k = 10;
    std::vector<Embedding<N>> rows(n), queries(nq);
    for (size_t i = 0; i < n; ++i)
        for (auto& x : rows[i]) x = frand();
    for (size_t i = 0; i < nq; ++i) queries[i] = i % 2 ? rows[i * 13] : rows[(i * 7) % n];
    L2SquaredDistance<N> metric;
    LSHIndex<N> ix = LSHIndex<N>::create(Uuid::now_v7(), LSHIndexOptions<N>{64, 6}, metric, 0, 11);
    zbo_index* orc = zbo_create((int)N, 1, 64, 6, 11);
    std::vector<Uuid> ids = ix.add(rows);
    std::vector<uint64_t> oids(n);
    zbo_add(orc, n, rows[0].data(), oids.data());
    std::map<Uuid, uint64_t> ordinal_of;
    for (size_t i = 0; i < n; ++i) ordinal_of[ids[i]] = i;
    // the set: every third row plus one id the index does not know; the oracle loses the complement
    std::vector<Uuid> pick;
    std::vector<uint64_t> out_o;
    std::vector<uint8_t> in(n, 0);
    for (size_t i = 0; i < n; ++i) {
        if (i % 3 == 0) {
            pick.push_back(ids[i]);
            in[i] = 1;
        } else {
            out_o.push_back(i);
        }
    }
    pick.push_back(Uuid::now_v7());
    std::vector<uint8_t> found;
    auto rs = ix.rowset(pick, false, &found);
    report("rowset from ids: count and found", rs.count() == (n + 2) / 3 && found.size() == pick.size() && found.back() == 0 &&
                                                   std::count(found.begin(), found.end(), 1) == (long)((n + 2) / 3));
    zbo_remove(orc, out_o.size(), out_o.data(), nullptr);
    std::vector<uint64_t> eo(nq * k), eb(nq * k);
    std::vector<uint32_t> ec(nq);
    zbo_search_batch(orc, nq, queries[0].data(), k, 4, eo.data(), eb.data(), ec.data());
    report("search_batch within an id rowset", same(ix.search_batch(queries, k, rs), ordinal_of, eo, eb, ec, k));
    // the same set by ordinals, in exclude mode (every row except the complement)
    auto rx = ix.rowset_ordinals(out_o, true);
    report("search_batch within an exclude-mode ordinal rowset", rx.count() == rs.count() &&
                                                                    same(ix.search_batch(queries, k, rx), ordinal_of, eo, eb, ec, k));
    // exact search within the set: brute force over its live rows
    for (size_t q = 0; q < nq; ++q) {
        std::vector<std::pair<uint64_t, uint64_t>> all;
        for (size_t i = 0; i < n; ++i)
            if (in[i]) all.emplace_back(zbo_distance_bits(1, rows[i].data(), queries[q].data(), (int)N), i);
        std::sort(all.begin(), all.end());
        ec[q] = (uint32_t)std::min(k, all.size());
        for (size_t i = 0; i < ec[q]; ++i) {
            eo[q * k + i] = all[i].second;
            eb[q * k + i] = all[i].first;
        }
    }
    report("search_exact within a rowset", same(ix.search_exact(queries, k, rs), ordinal_of, eo, eb, ec, k));
    int code = 0;
    try {
        ix.rowset_ordinals({n});
    } catch (const Error& e) {
        code = e.code;
    }
    report("unknown ordinal -> ZB_ERR_INVALID", code == ZB_ERR_INVALID);
    rs.reset();
    // an empty RowSet (reset, moved-from or default) must not turn into the unrestricted search
    int refused = 0;
    LSHIndex<N>::RowSet none;
    for (const LSHIndex<N>::RowSet* w : {&rs, &none}) {
        try { ix.search_batch(queries, k, *w); } catch (const Error& e) { refused += e.code == ZB_ERR_INVALID; }
        try { ix.search_exact(queries, k, *w); } catch (const Error& e) { refused += e.code == ZB_ERR_INVALID; }
    }
    report("empty RowSet refused", refused == 4);
    rx.reset();
    zbo_destroy(orc);
    return failures;
}

int main(int argc, char** argv) {
    if (argc < 2 || std::string(argv[1]) != "gpu") {
        std::printf("usage: rowset_mirror_test gpu\n");
        return 2;
    }
    int rc = 1;
    try {
        rc = run_gpu();
    } catch (const std::exception& e) {
        std::printf("FAILED: %s\n", e.what());
    }
    if (rc == 0) std::printf("all ok\n");
    return rc;
}
