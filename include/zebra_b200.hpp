// zebra_b200.hpp -- C++ host mirror of the reference's operator interface for the query hot path, above the C ABI of
// zebra_b200.h (header only, C++17).  The reference is a Rust crate and no Rust toolchain exists in the build image, so
// the host side a Rust maintainer would write (INTEGRATION.md) is stated here in the other compiled language at hand,
// type for type and method for method:
//
//   zebra::Embedding<N>                  /root/reference/src/lib.rs:16-48            [f32; N], contiguous
//   zebra::DistanceUnit, the 13 metrics  /root/reference/src/distance.rs:13-190      `distance(&a, &b) -> u64`
//   zebra::LSHIndexOptions<N>            src/database/index/lsh.rs:122-138           defaults 5 / 15
//   zebra::LSHIndex<N>                   src/database/index/lsh.rs:145-566           new, save, deduplicate, is_empty,
//                                                                                    no_vectors, no_trees, add, remove, clear, search
//   zebra::DatabaseEmbeddingModel<N>     src/model/core.rs:12-37                     embed_documents
//   zebra::Database<N, Met, Mod>         src/database/core.rs:55-381                 open, new, new_with_path, open_or_create,
//                                                                                    save_database, clear_database, remove, deduplicate,
//                                                                                    insert_documents, insert_records, query_documents,
//                                                                                    query_vectors; `index` is public (core.rs:62)
//
// Conventions carried over: `anyhow::Result<T>` becomes T or a thrown zebra::Error (code = zb_status, message =
// zb_last_error()); `DashSet` / `DashMap` become std::set / std::map; LSHIndex and Database are cheap to copy and share
// one device index (the reference types are Clone over a shared store).  There is NO CPU compute path: every distance,
// sign test and search runs in libzebra_b200.so's CUDA kernels, and without a B200 every constructor throws
// (ZB_ERR_NO_DEVICE).  Where the device index differs from the reference it is by the documented divergences of
// DESIGN.md section 7 (tombstone delete D1, seeded sampling D2, ties by id D3, batch insert D4).
#ifndef ZEBRA_B200_HPP
#define ZEBRA_B200_HPP

#include <array>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <optional>
#include <random>
#include <set>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "zebra_b200.h"

namespace zebra {

using EmbeddingPrecision = float;  // lib.rs:48
using DistanceUnit = uint64_t;     // distance.rs:13
using Bytes = std::vector<uint8_t>;

/// anyhow::Error of a failed call: `code` is the zb_status, what() the library's message.
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int rc) {
    if (rc != ZB_OK) {
        const char* m = zb_last_error();
        throw Error(rc, std::string("zebra_b200 error ") + std::to_string(rc) + ": " + (m ? m : "?"));
    }
}

/// lib.rs:16-48: an embedding vector, N contiguous f32 (`Default` is all zeros).
template <size_t N>
struct Embedding : std::array<EmbeddingPrecision, N> {
    Embedding() { this->fill(0.0f); }
    explicit Embedding(const std::array<EmbeddingPrecision, N>& v) : std::array<EmbeddingPrecision, N>(v) {}
    /// TryFrom<Vec<f32>> (lib.rs:41-46): fails unless the length is exactly N.
    static Embedding try_from(const std::vector<EmbeddingPrecision>& v) {
        if (v.size() != N) throw Error(ZB_ERR_INVALID, "Embedding::try_from: length is not N");
        Embedding e;
        std::memcpy(e.data(), v.data(), N * sizeof(float));
        return e;
    }
};
static_assert(sizeof(Embedding<3>) == 3 * sizeof(float), "Embedding<N> must be N packed f32 (the ABI takes &Vec<Embedding<N>> as n x N floats)");

/// uuid::Uuid: 16 bytes, ordered as big-endian integers (= byte order), which is the order ties are broken by.
struct Uuid {
    std::array<uint8_t, 16> bytes{};
    const uint8_t* as_bytes() const { return bytes.data(); }
    static Uuid from_slice(const uint8_t* p) {
        Uuid u;
        std::memcpy(u.bytes.data(), p, 16);
        return u;
    }
    /// Uuid::now_v7(): 48-bit millisecond timestamp, version 7, variant 10, 74 random bits.
    static Uuid now_v7() {
        static thread_local std::mt19937_64 rng{std::random_device{}()};
        const uint64_t ms = (uint64_t)std::chrono::duration_cast<std::chrono::milliseconds>(
                                std::chrono::system_clock::now().time_since_epoch()).count();
        const uint64_t a = rng(), b = rng();
        Uuid u;
        for (int i = 0; i < 6; ++i) u.bytes[i] = (uint8_t)(ms >> (8 * (5 - i)));
        u.bytes[6] = (uint8_t)(0x70 | ((a >> 8) & 0x0F));
        u.bytes[7] = (uint8_t)a;
        u.bytes[8] = (uint8_t)(0x80 | ((b >> 56) & 0x3F));
        for (int i = 9; i < 16; ++i) u.bytes[i] = (uint8_t)(b >> (8 * (15 - i)));
        return u;
    }
    int version() const { return bytes[6] >> 4; }
    /// Uuid::as_simple(): 32 lower-case hex digits (core.rs:77, :81).
    std::string simple() const {
        static const char* hex = "0123456789abcdef";
        std::string s(32, '0');
        for (int i = 0; i < 16; ++i) {
            s[2 * i] = hex[bytes[i] >> 4];
            s[2 * i + 1] = hex[bytes[i] & 15];
        }
        return s;
    }
    bool operator==(const Uuid& o) const { return bytes == o.bytes; }
    bool operator!=(const Uuid& o) const { return bytes != o.bytes; }
    bool operator<(const Uuid& o) const { return bytes < o.bytes; }
};

// ---------------------------------------------------------------------------------------------------------------
// distance.rs: the metric structs.  `distance` keeps the trait's shape (space::Metric<Embedding<N>>, Unit = u64) and
// the reference's argument order (a = stored row, b = query; lsh.rs:314, :559); it is evaluated by the CUDA library.
// ---------------------------------------------------------------------------------------------------------------
namespace detail {
template <size_t N>
inline DistanceUnit device_distance(uint32_t metric, int32_t power, const Embedding<N>& a, const Embedding<N>& b, int device) {
    uint64_t out = 0;
    check(zb_metric_distance_batch(device, metric, power, 1, (uint32_t)N, a.data(), b.data(), &out));
    return out;
}
}  // namespace detail

#define ZEBRA_UNIT_METRIC(NAME, CODE)                                                                           \
    template <size_t N>                                                                                         \
    struct NAME {                                                                                               \
        static constexpr uint32_t ZB_METRIC = CODE;                                                             \
        static constexpr bool HAS_POWER = false;                                                                \
        int32_t zb_power() const { return 0; }                                                                  \
        DistanceUnit distance(const Embedding<N>& a, const Embedding<N>& b) const {                             \
            return detail::device_distance<N>(ZB_METRIC, 0, a, b, 0);                                           \
        }                                                                                                       \
    };
ZEBRA_UNIT_METRIC(CosineDistance, ZB_METRIC_COSINE)          // distance.rs:15-32  (1.0 - simsimd cosine).to_bits(), quirk Q4
ZEBRA_UNIT_METRIC(L2SquaredDistance, ZB_METRIC_L2SQ)         // distance.rs:34-49
ZEBRA_UNIT_METRIC(ChebyshevDistance, ZB_METRIC_CHEBYSHEV)    // distance.rs:51-61
ZEBRA_UNIT_METRIC(CanberraDistance, ZB_METRIC_CANBERRA)      // distance.rs:63-73
ZEBRA_UNIT_METRIC(BrayCurtisDistance, ZB_METRIC_BRAY_CURTIS) // distance.rs:75-85
ZEBRA_UNIT_METRIC(ManhattanDistance, ZB_METRIC_MANHATTAN)    // distance.rs:87-97
ZEBRA_UNIT_METRIC(L2Distance, ZB_METRIC_L2)                  // distance.rs:99-114
ZEBRA_UNIT_METRIC(L3Distance, ZB_METRIC_L3)                  // distance.rs:116-126
ZEBRA_UNIT_METRIC(L4Distance, ZB_METRIC_L4)                  // distance.rs:128-138
ZEBRA_UNIT_METRIC(HammingDistance, ZB_METRIC_HAMMING)        // distance.rs:140-157
#undef ZEBRA_UNIT_METRIC

#define ZEBRA_POWER_METRIC(NAME, CODE)                                                                          \
    template <size_t N>                                                                                         \
    struct NAME {                                                                                               \
        static constexpr uint32_t ZB_METRIC = CODE;                                                             \
        static constexpr bool HAS_POWER = true;                                                                 \
        int32_t power = 0; /* `pub power: i32`; Default = 0 */                                                  \
        int32_t zb_power() const { return power; }                                                              \
        DistanceUnit distance(const Embedding<N>& a, const Embedding<N>& b) const {                             \
            return detail::device_distance<N>(ZB_METRIC, power, a, b, 0);                                       \
        }                                                                                                       \
    };
ZEBRA_POWER_METRIC(MinkowskiDistance, ZB_METRIC_MINKOWSKI)   // distance.rs:159-173
ZEBRA_POWER_METRIC(PNormDistance, ZB_METRIC_PNORM)           // distance.rs:175-190
#undef ZEBRA_POWER_METRIC

/// Hyperplane<N> (lsh.rs:16-44); point_is_above runs on the device.
template <size_t N>
struct Hyperplane {
    Embedding<N> coefficients;
    EmbeddingPrecision constant = 0.0f;
    bool point_is_above(const Embedding<N>& point) const {
        uint8_t out = 0;
        check(zb_point_is_above_batch(0, 1, (uint32_t)N, coefficients.data(), &constant, point.data(), &out));
        return out != 0;
    }
};

/// lsh.rs:122-138.
template <size_t N>
struct LSHIndexOptions {
    size_t max_node_size = 5;
    size_t num_trees = 15;
    bool operator==(const LSHIndexOptions& o) const { return max_node_size == o.max_node_size && num_trees == o.num_trees; }
};

// ---------------------------------------------------------------------------------------------------------------
// LSHIndex<N> (lsh.rs:145-566) over a device index.  The reference passes the metric to search(); a device index is
// created for one metric (its scan kernels are specialised), and search() with another one throws.
// ---------------------------------------------------------------------------------------------------------------
template <size_t N>
class LSHIndex {
    struct Handle {
        zb_index* p = nullptr;
        ~Handle() {
            if (p) zb_index_destroy(p);
        }
    };
    std::shared_ptr<Handle> h_;
    LSHIndexOptions<N> options_;
    uint32_t metric_ = 0;
    int32_t power_ = 0;

  public:
    LSHIndex() = default;
    /// LSHIndex::new (lsh.rs:162-167) plus the metric (and the device placement) a device index is built for.
    template <class Met>
    static LSHIndex create(const Uuid& /*database uuid: names the fjall keyspace in the reference*/, const LSHIndexOptions<N>& options,
                           const Met& metric, int device = 0, uint64_t seed = 0, uint32_t shard_rank = 0, uint32_t shard_count = 1) {
        zb_options o;
        std::memset(&o, 0, sizeof o);
        o.dim = (uint32_t)N;
        o.metric = Met::ZB_METRIC;
        o.metric_power = metric.zb_power();
        o.max_node_size = options.max_node_size;
        o.num_trees = (uint32_t)options.num_trees;
        o.device = device;
        o.seed = seed;
        o.shard_rank = shard_rank;
        o.shard_count = shard_count;
        LSHIndex ix;
        ix.h_ = std::make_shared<Handle>();
        check(zb_index_create(&o, &ix.h_->p));
        ix.options_ = options;
        ix.metric_ = Met::ZB_METRIC;
        ix.power_ = metric.zb_power();
        return ix;
    }
    zb_index* raw() const { return h_ ? h_->p : nullptr; }
    const LSHIndexOptions<N>& options() const { return options_; }

    /// lsh.rs:170-172 (fjall persist): the key-value engine is the host's; see export_tree_blobs / export_rows.
    void save() const {}

    /// lsh.rs:270-288.
    std::set<Uuid> deduplicate() const {
        zb_stats st;
        check(zb_index_stats(raw(), &st));
        const uint64_t cap = st.total_rows ? st.total_rows : 1;
        std::vector<uint8_t> ids(cap * 16);
        uint64_t count = 0;
        check(zb_index_deduplicate(raw(), &count, nullptr, ids.data(), cap));
        std::set<Uuid> out;
        for (uint64_t i = 0; i < count && i < cap; ++i) out.insert(Uuid::from_slice(ids.data() + 16 * i));
        return out;
    }
    /// lsh.rs:389-409.
    bool no_vectors() const {
        int v = 0;
        check(zb_index_no_vectors(raw(), &v));
        return v != 0;
    }
    bool no_trees() const {
        int v = 0;
        check(zb_index_no_trees(raw(), &v));
        return v != 0;
    }
    bool is_empty() const { return no_vectors() || no_trees(); }

    /// lsh.rs:440-466 (build_index :411-429 the first time).  Ids are minted by the library (UUIDv7, id order = input order).
    std::vector<Uuid> add(const std::vector<Embedding<N>>& embeddings) const { return add_with_ids(embeddings, nullptr); }
    /// The same with caller-chosen ids (what a host that already keys its documents needs).
    std::vector<Uuid> add(const std::vector<Embedding<N>>& embeddings, const std::vector<Uuid>& ids) const {
        if (ids.size() != embeddings.size()) throw Error(ZB_ERR_INVALID, "one id per embedding");
        return add_with_ids(embeddings, &ids);
    }
    /// lsh.rs:473-503 (tombstones, DESIGN.md D1): the ids that were present and are now removed.
    std::set<Uuid> remove(const std::vector<Uuid>& embedding_ids) const {
        std::vector<uint8_t> raw_ids = pack(embedding_ids), flags(embedding_ids.size() + 1, 0);
        check(zb_index_remove(raw(), embedding_ids.size(), raw_ids.data(), flags.data()));
        std::set<Uuid> out;
        for (size_t i = 0; i < embedding_ids.size(); ++i)
            if (flags[i]) out.insert(embedding_ids[i]);
        return out;
    }
    /// lsh.rs:506-529 (without quirk Q12: trees go too).
    void clear() const { check(zb_index_clear(raw())); }

    /// lsh.rs:544-565 for ONE query -- prefer search_batch.  probes > 0: multi-probe search (zb_index_search_probe,
    /// DESIGN 3.9); 0 is the reference's search.
    template <class Met>
    std::vector<std::pair<Uuid, DistanceUnit>> search(const Embedding<N>& query, size_t top_k, const Met& metric,
                                                      uint32_t probes = 0) const {
        if (Met::ZB_METRIC != metric_ || metric.zb_power() != power_)
            throw Error(ZB_ERR_INVALID, "this device index was created for another metric");
        return std::move(search_batch(std::vector<Embedding<N>>{query}, top_k, probes)[0]);
    }
    /// The whole batch in one device call (replaces the par_iter of core.rs:299-303): per query, ascending (distance
    /// bits, id), at most top_k entries.
    std::vector<std::vector<std::pair<Uuid, DistanceUnit>>> search_batch(const std::vector<Embedding<N>>& queries, size_t top_k,
                                                                         uint32_t probes = 0) const {
        const size_t nq = queries.size();
        std::vector<uint8_t> ids(nq * top_k * 16 + 1);
        std::vector<uint64_t> bits(nq * top_k + 1);
        std::vector<uint32_t> counts(nq + 1, 0);
        if (probes)
            check(zb_index_search_probe(raw(), nq, nq ? queries[0].data() : nullptr, top_k, probes, ids.data(), nullptr, bits.data(),
                                        counts.data()));
        else
            check(zb_index_search_batch(raw(), nq, nq ? queries[0].data() : nullptr, top_k, ids.data(), nullptr, bits.data(), counts.data()));
        std::vector<std::vector<std::pair<Uuid, DistanceUnit>>> out(nq);
        for (size_t q = 0; q < nq; ++q)
            for (uint32_t i = 0; i < counts[q]; ++i) {
                const size_t o = q * top_k + i;
                out[q].emplace_back(Uuid::from_slice(ids.data() + 16 * o), bits[o]);
            }
        return out;
    }

    /// Bucket keys (root-to-leaf sign path of lsh.rs:350-366, MSB = root): keys[i * num_trees + t], depths likewise.
    void hash(const std::vector<Embedding<N>>& rows, std::vector<uint64_t>& keys, std::vector<uint32_t>& depths) const {
        keys.assign(rows.size() * options_.num_trees, 0);
        depths.assign(rows.size() * options_.num_trees, 0);
        if (rows.empty()) return;
        check(zb_index_hash(raw(), rows.size(), rows[0].data(), keys.data(), depths.data(), nullptr));
    }

    /// FLAT tables (the K-bit LSH table): plane t * bits + d serves every node at depth d of tree t.  The rows are
    /// bucketed by one dense projection on the device; afterwards the index holds the equivalent forest.
    void load_flat(const std::vector<Embedding<N>>& rows, uint32_t bits, const std::vector<Embedding<N>>& planes,
                   const std::vector<EmbeddingPrecision>& constants, const std::vector<Uuid>* ids = nullptr) const {
        if (planes.size() != options_.num_trees * bits || constants.size() != planes.size())
            throw Error(ZB_ERR_INVALID, "load_flat takes num_trees * bits planes and constants");
        if (ids && ids->size() != rows.size()) throw Error(ZB_ERR_INVALID, "one id per row");
        std::vector<uint8_t> raw_ids;
        if (ids) raw_ids = pack(*ids);
        check(zb_index_load_flat(raw(), rows.size(), rows.empty() ? nullptr : rows[0].data(), ids ? raw_ids.data() : nullptr, bits,
                                 planes[0].data(), constants.data()));
    }

    // ---- the reference's stored values (KeyValue, lsh.rs:63-119): see INTEGRATION.md section 6 ----
    /// Replace the content with a store: (id, embedding) pairs of the `embeddings` partition and the values of `trees`.
    zb_import_report import_store(const std::vector<Uuid>& ids, const std::vector<Embedding<N>>& embeddings,
                                  const std::vector<Bytes>& tree_blobs, std::vector<Uuid>* orphans = nullptr) const {
        if (ids.size() != embeddings.size()) throw Error(ZB_ERR_INVALID, "one id per embedding");
        std::vector<uint8_t> raw_ids = pack(ids), orph(ids.size() * 16 + 1);
        std::vector<const uint8_t*> ptrs;
        std::vector<uint64_t> sizes;
        for (const Bytes& b : tree_blobs) {
            ptrs.push_back(b.data());
            sizes.push_back(b.size());
        }
        zb_import_report rep;
        check(zb_index_import_store(raw(), ids.size(), raw_ids.data(), embeddings.empty() ? nullptr : embeddings[0].data(),
                                    (uint32_t)tree_blobs.size(), ptrs.data(), sizes.data(), &rep, orph.data(), ids.size()));
        if (orphans) {
            orphans->clear();
            for (uint64_t i = 0; i < rep.orphan_rows; ++i) orphans->push_back(Uuid::from_slice(orph.data() + 16 * i));
        }
        return rep;
    }
    /// Every row with its id and live flag (removed rows: the reference would have deleted the key).
    void export_rows(std::vector<Uuid>& ids, std::vector<Embedding<N>>& embeddings, std::vector<uint8_t>& live) const {
        zb_stats st;
        check(zb_index_stats(raw(), &st));
        const uint64_t n = st.total_rows;
        embeddings.assign(n, Embedding<N>());
        live.assign(n + 1, 0);
        std::vector<uint8_t> raw_ids(n * 16 + 1);
        check(zb_index_export_rows(raw(), 0, n, n ? embeddings[0].data() : nullptr, raw_ids.data(), live.data()));
        live.resize(n);
        ids.clear();
        for (uint64_t i = 0; i < n; ++i) ids.push_back(Uuid::from_slice(raw_ids.data() + 16 * i));
    }
    /// Every tree as the bincode(legacy) Node<N> value the reference stores (lsh.rs:99-105).
    std::vector<Bytes> export_tree_blobs() const {
        std::vector<uint64_t> sizes(options_.num_trees + 1, 0);
        uint64_t total = 0;
        check(zb_index_export_tree_blobs(raw(), nullptr, 0, sizes.data(), &total));  // one forest export for all trees
        Bytes all(total + 1);
        check(zb_index_export_tree_blobs(raw(), all.data(), total, sizes.data(), &total));
        std::vector<Bytes> out;
        uint64_t at = 0;
        for (size_t t = 0; t < options_.num_trees; ++t) {
            out.emplace_back(all.begin() + (std::ptrdiff_t)at, all.begin() + (std::ptrdiff_t)(at + sizes[t]));
            at += sizes[t];
        }
        return out;
    }
    zb_stats stats() const {
        zb_stats st;
        check(zb_index_stats(raw(), &st));
        return st;
    }

  private:
    static std::vector<uint8_t> pack(const std::vector<Uuid>& ids) {
        std::vector<uint8_t> raw_ids(ids.size() * 16 + 1);
        for (size_t i = 0; i < ids.size(); ++i) std::memcpy(raw_ids.data() + 16 * i, ids[i].bytes.data(), 16);
        return raw_ids;
    }
    std::vector<Uuid> add_with_ids(const std::vector<Embedding<N>>& embeddings, const std::vector<Uuid>* ids) const {
        const size_t n = embeddings.size();
        std::vector<uint8_t> out(n * 16 + 1), in;
        if (ids) in = pack(*ids);
        check(zb_index_add(raw(), n, n ? embeddings[0].data() : nullptr, ids ? in.data() : nullptr, out.data(), nullptr));
        std::vector<Uuid> res;
        for (size_t i = 0; i < n; ++i) res.push_back(Uuid::from_slice(out.data() + 16 * i));
        return res;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// Flat dump of the two key-value partitions (the format of zebra_b200/interchange.py: "ZBXSTOR1"), for hosts without
// the fjall crate.  Values are exactly what the reference stores under those keys.
// ---------------------------------------------------------------------------------------------------------------
namespace store {
struct Dump {
    uint32_t dim = 0;
    Bytes zebra;                                  // the `.zebra` file (may be empty)
    std::vector<std::pair<Uuid, Bytes>> trees;    // partition `trees`
    std::vector<Uuid> ids;                        // partition `embeddings`: keys ...
    std::vector<float> rows;                      // ... and values, n x dim
};
inline void put_u64(std::ostream& f, uint64_t v) { f.write(reinterpret_cast<const char*>(&v), 8); }
inline uint64_t get_u64(std::istream& f) {
    uint64_t v = 0;
    f.read(reinterpret_cast<char*>(&v), 8);
    if (!f) throw Error(ZB_ERR_INVALID, "store dump truncated");
    return v;
}
inline void write(const std::string& path, const Dump& d) {
    std::ofstream f(path, std::ios::binary | std::ios::trunc);
    if (!f) throw Error(ZB_ERR_INVALID, "cannot write " + path);
    f.write("ZBXSTOR1", 8);
    f.write(reinterpret_cast<const char*>(&d.dim), 4);
    put_u64(f, d.zebra.size());
    f.write(reinterpret_cast<const char*>(d.zebra.data()), (std::streamsize)d.zebra.size());
    put_u64(f, d.trees.size());
    for (const auto& kv : d.trees) {
        f.write(reinterpret_cast<const char*>(kv.first.bytes.data()), 16);
        put_u64(f, kv.second.size());
        f.write(reinterpret_cast<const char*>(kv.second.data()), (std::streamsize)kv.second.size());
    }
    put_u64(f, d.ids.size());
    for (size_t i = 0; i < d.ids.size(); ++i) {
        f.write(reinterpret_cast<const char*>(d.ids[i].bytes.data()), 16);
        put_u64(f, 4ull * d.dim);
        f.write(reinterpret_cast<const char*>(d.rows.data() + i * d.dim), 4 * (std::streamsize)d.dim);
    }
    if (!f) throw Error(ZB_ERR_INVALID, "write to " + path + " failed");
}
inline Dump read(const std::string& path) {
    std::ifstream f(path, std::ios::binary);
    char magic[8];
    f.read(magic, 8);
    if (!f || std::memcmp(magic, "ZBXSTOR1", 8) != 0) throw Error(ZB_ERR_INVALID, path + " is not a zebra_b200 store dump");
    Dump d;
    f.read(reinterpret_cast<char*>(&d.dim), 4);
    d.zebra.resize(get_u64(f));
    f.read(reinterpret_cast<char*>(d.zebra.data()), (std::streamsize)d.zebra.size());
    const uint64_t nt = get_u64(f);
    for (uint64_t t = 0; t < nt; ++t) {
        Uuid k;
        f.read(reinterpret_cast<char*>(k.bytes.data()), 16);
        Bytes v(get_u64(f));
        f.read(reinterpret_cast<char*>(v.data()), (std::streamsize)v.size());
        if (!f) throw Error(ZB_ERR_INVALID, "store dump truncated");
        d.trees.emplace_back(k, std::move(v));
    }
    const uint64_t n = get_u64(f);
    d.rows.resize(n * d.dim);
    for (uint64_t i = 0; i < n; ++i) {
        Uuid k;
        f.read(reinterpret_cast<char*>(k.bytes.data()), 16);
        if (get_u64(f) != 4ull * d.dim) throw Error(ZB_ERR_INVALID, "embedding value of the wrong size");
        f.read(reinterpret_cast<char*>(d.rows.data() + i * d.dim), 4 * (std::streamsize)d.dim);
        d.ids.push_back(k);
    }
    if (!f) throw Error(ZB_ERR_INVALID, "store dump truncated");
    return d;
}
/// A UUIDv7-shaped key for tree t of an exported store (the reference mints Uuid::now_v7(), lsh.rs:423).
inline Uuid tree_key(uint32_t t) {
    Uuid u;
    u.bytes[6] = 0x70;
    u.bytes[8] = 0x80;
    for (int i = 0; i < 4; ++i) u.bytes[15 - i] = (uint8_t)(t >> (8 * i));
    return u;
}
}  // namespace store

/// model/core.rs:12-37.  Embedding models are outside the device path; the trait stays so Database is generic over one.
template <size_t N>
struct DatabaseEmbeddingModel {
    virtual ~DatabaseEmbeddingModel() = default;
    virtual std::vector<Embedding<N>> embed_documents(const std::vector<Bytes>& /*documents*/) const {
        throw Error(ZB_ERR_STATE, "no embedding model on the device path (BASELINE configs use raw vectors)");
    }
};

// ---------------------------------------------------------------------------------------------------------------
// Database<N, Met, Mod> (core.rs:55-381).  The three call sites into the index keep their shape (remove :207,
// insert_records :250, query_vectors :299-303 -- the latter as ONE batched device call).  Documents live in memory (the
// lz4 document files of core.rs:322-380 are host I/O outside the hot path).
// ---------------------------------------------------------------------------------------------------------------
template <size_t N, class Met, class Mod = DatabaseEmbeddingModel<N>>
class Database {
    struct Shared {
        Uuid uuid;
        Mod model{};
        Met metric{};
        LSHIndexOptions<N> index_options;
        std::string path;
        std::map<Uuid, Bytes> documents;
    };
    std::shared_ptr<Shared> s_;

    static Database make(const Uuid& uuid, const Met& metric, const LSHIndexOptions<N>& options, const std::string& path) {
        Database db;
        db.s_ = std::make_shared<Shared>();
        db.s_->uuid = uuid;
        db.s_->metric = metric;
        db.s_->index_options = options;
        db.s_->path = path;
        db.index = LSHIndex<N>::create(uuid, options, metric);
        return db;
    }

  public:
    /// `pub index: LSHIndex<N>` (core.rs:62).
    LSHIndex<N> index;

    const Uuid& uuid() const { return s_->uuid; }
    const Met& metric() const { return s_->metric; }
    const LSHIndexOptions<N>& index_options() const { return s_->index_options; }
    const std::string& path() const { return s_->path; }
    std::string default_database_path() const { return s_->uuid.simple() + ".zebra"; }  // core.rs:80-82

    /// core.rs:92-104: `path` holds bincode(legacy) DatabaseInner; `path + ".store"` the dump of the index's partitions.
    static Database open(const std::string& path) {
        std::ifstream f(path, std::ios::binary);
        if (!f) throw Error(ZB_ERR_INVALID, "cannot read " + path);
        Bytes raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        Uuid uuid;
        int32_t power = 0;
        uint64_t mns = 0, nt = 0;
        check(zb_zebra_file_decode(raw.data(), raw.size(), Met::ZB_METRIC, uuid.bytes.data(), &power, &mns, &nt));
        Met metric{};
        if constexpr (Met::HAS_POWER) metric.power = power;
        (void)power;
        LSHIndexOptions<N> options;
        options.max_node_size = (size_t)mns;
        options.num_trees = (size_t)nt;
        Database db = make(uuid, metric, options, path);
        store::Dump d = store::read(path + ".store");
        if (d.dim != N) throw Error(ZB_ERR_INVALID, "the store holds vectors of another dimension");
        std::vector<Embedding<N>> rows(d.ids.size());
        if (!rows.empty()) std::memcpy(rows[0].data(), d.rows.data(), d.rows.size() * sizeof(float));
        if (d.trees.empty()) {
            if (!rows.empty()) db.index.add(rows, d.ids);
        } else {
            std::vector<Bytes> blobs;
            for (auto& kv : d.trees) blobs.push_back(std::move(kv.second));
            std::vector<Uuid> orphans;
            db.index.import_store(d.ids, rows, blobs, &orphans);
            if (!orphans.empty()) {  // embeddings some tree had lost (quirk Q11): insert them properly
                std::map<Uuid, size_t> at;
                for (size_t i = 0; i < d.ids.size(); ++i) at[d.ids[i]] = i;
                std::vector<Embedding<N>> again;
                for (const Uuid& u : orphans) again.push_back(rows[at[u]]);
                db.index.add(again, orphans);
            }
        }
        return db;
    }
    /// core.rs:110-130 (`new` is a keyword here).
    static Database create(const LSHIndexOptions<N>& index_options) {
        const Uuid uuid = Uuid::now_v7();
        Database db = make(uuid, Met{}, index_options, "");
        db.s_->path = db.default_database_path();
        db.save_database();
        return db;
    }
    /// core.rs:140-160.
    static Database new_with_path(const std::string& path, const LSHIndexOptions<N>& index_options) {
        Database db = make(Uuid::now_v7(), Met{}, index_options, path);
        db.save_database();
        return db;
    }
    /// A database with a chosen metric value (MinkowskiDistance { power }), not persisted until save_database.
    static Database with_metric(const Met& metric, const LSHIndexOptions<N>& index_options, const std::string& path = "") {
        return make(Uuid::now_v7(), metric, index_options, path);
    }
    /// core.rs:170-178.
    static Database open_or_create(const std::string& path, const LSHIndexOptions<N>& index_options) {
        try {
            return open(path);
        } catch (const Error&) {
            return new_with_path(path, index_options);
        }
    }
    /// core.rs:183-190.
    void save_database(const std::optional<std::string>& path = std::nullopt) const {
        const std::string p = path ? *path : (s_->path.empty() ? default_database_path() : s_->path);
        uint8_t buf[64];
        uint64_t need = 0;
        check(zb_zebra_file_encode(s_->uuid.bytes.data(), Met::ZB_METRIC, s_->metric.zb_power(), s_->index_options.max_node_size,
                                   s_->index_options.num_trees, buf, sizeof buf, &need));
        {
            std::ofstream f(p, std::ios::binary | std::ios::trunc);
            f.write(reinterpret_cast<const char*>(buf), (std::streamsize)need);
            if (!f) throw Error(ZB_ERR_INVALID, "cannot write " + p);
        }
        store::Dump d;
        d.dim = (uint32_t)N;
        d.zebra.assign(buf, buf + need);
        std::vector<Uuid> ids;
        std::vector<Embedding<N>> rows;
        std::vector<uint8_t> live;
        index.export_rows(ids, rows, live);
        for (size_t i = 0; i < ids.size(); ++i)
            if (live[i]) {
                d.ids.push_back(ids[i]);
                d.rows.insert(d.rows.end(), rows[i].begin(), rows[i].end());
            }
        if (!index.no_trees()) {
            std::vector<Bytes> blobs = index.export_tree_blobs();
            for (uint32_t t = 0; t < blobs.size(); ++t) d.trees.emplace_back(store::tree_key(t), std::move(blobs[t]));
        }
        store::write(p + ".store", d);
        index.save();
        s_->path = p;
    }
    /// core.rs:194-198.
    void clear_database() const {
        index.clear();
        s_->documents.clear();
        std::remove(s_->path.c_str());
        std::remove((s_->path + ".store").c_str());
    }
    /// core.rs:205-213.
    void remove(const std::vector<Uuid>& embedding_ids) const {
        for (const Uuid& u : index.remove(embedding_ids)) s_->documents.erase(u);
    }
    /// core.rs:216-224.
    void deduplicate() const {
        for (const Uuid& u : index.deduplicate()) s_->documents.erase(u);
    }
    /// core.rs:232-235.
    void insert_documents(const std::vector<Bytes>& documents) const { insert_records(s_->model.embed_documents(documents), documents); }
    /// core.rs:245-254.  Returns the ids (the reference discards them, survey quirk Q9).
    std::vector<Uuid> insert_records(const std::vector<Embedding<N>>& embeddings, const std::vector<Bytes>& documents) const {
        if (embeddings.size() != documents.size()) throw Error(ZB_ERR_INVALID, "one document per embedding");
        std::vector<Uuid> ids = index.add(embeddings);
        for (size_t i = 0; i < ids.size(); ++i) s_->documents[ids[i]] = documents[i];
        return ids;
    }
    /// core.rs:267-277.
    std::map<size_t, std::map<Uuid, Bytes>> query_documents(const std::vector<Bytes>& documents, size_t number_of_results) const {
        if (index.no_vectors()) return {};
        return query_vectors(s_->model.embed_documents(documents), number_of_results);
    }
    /// core.rs:290-313: query index -> (document id -> document bytes).
    std::map<size_t, std::map<Uuid, Bytes>> query_vectors(const std::vector<Embedding<N>>& vectors, size_t number_of_results,
                                                          uint32_t probes = 0) const {
        std::map<size_t, std::map<Uuid, Bytes>> results;
        if (index.no_vectors()) return results;
        auto all = index.search_batch(vectors, number_of_results, probes);  // was: vectors.into_par_iter() ... index.search(x, ..)
        for (size_t q = 0; q < all.size(); ++q) {
            std::map<Uuid, Bytes>& m = results[q];
            for (const auto& hit : all[q]) {
                auto it = s_->documents.find(hit.first);
                m[hit.first] = it == s_->documents.end() ? Bytes{} : it->second;
            }
        }
        return results;
    }
};

}  // namespace zebra
#endif  // ZEBRA_B200_HPP
