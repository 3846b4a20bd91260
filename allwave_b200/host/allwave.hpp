// allwave.hpp -- C++17 host-side mirror of allwave's library surface for the alignment path,
// sitting above the C ABI of liballwave_cuda.so (include/allwave_cuda.h).
//
// The reference's host code is Rust; no Rust toolchain exists in this image, so the host side is
// written in C++ with the same names, argument meaning and error behaviour:
//   Sequence, AlignmentParams, AlignmentMode, AlignmentResult, SparsificationStrategy   src/types.rs
//   parse_scores, alignment_to_paf, process_alignments_with_callback                    src/lib.rs:57-153
//   AllPairIterator {with_options, pair_count, get_pairs, for_each_with_callback, next} src/iterator.rs:25-252
//   apply_random_sparsification, compute_connectivity_probability                       src/iterator.rs:256-334
//   extract_tree_pairs, build_knn_graph, generate_random_pairs                          src/knn_graph.rs:12-174
//   mash distance from Jaccard                                                          src/mash.rs:59-74
//   the -p grammar of the CLI                                                           src/main.rs:136-203
//   wfa::{align_sequences, validate_cigar_alignment, Penalties, Mode, Result}           src/wfa.rs:7-258
// Everything numeric on the alignment path (sketches, Jaccard counts, orientation, wavefronts,
// CIGAR, PAF text) is computed on the GPU through the C ABI; this header only builds pair lists,
// partitions them and forwards results.
#pragma once
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <functional>
#include <mutex>
#include <optional>
#include <thread>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#ifdef ALLWAVE_HAVE_ZLIB
#include <zlib.h>
#endif

#include "../../include/allwave_cuda.h"

namespace allwave {

struct Sequence {
    std::string id;
    std::vector<uint8_t> seq;
};

struct AlignmentParams {
    int32_t match_score = 0;
    int32_t mismatch_penalty = 5;
    int32_t gap_open = 8;
    int32_t gap_extend = 2;
    std::optional<int32_t> gap2_open = 24;
    std::optional<int32_t> gap2_extend = 1;
    std::optional<double> max_divergence;
    // (noinline: g++ 13.3 crashes in its GIMPLE ccp pass when this is folded into a constructor's member initialiser)
    __attribute__((noinline)) static AlignmentParams edit_distance() {
        AlignmentParams p;
        p.mismatch_penalty = p.gap_open = p.gap_extend = 1;
        p.gap2_open.reset();
        p.gap2_extend.reset();
        return p;
    }
    bool operator==(const AlignmentParams& o) const {
        return match_score == o.match_score && mismatch_penalty == o.mismatch_penalty && gap_open == o.gap_open && gap_extend == o.gap_extend &&
               gap2_open == o.gap2_open && gap2_extend == o.gap2_extend && max_divergence == o.max_divergence;
    }
    aw_params to_c() const {
        aw_params p;
        std::memset(&p, 0, sizeof(p));
        p.match_score = match_score;
        p.mismatch_penalty = mismatch_penalty;
        p.gap_open = gap_open;
        p.gap_extend = gap_extend;
        if (gap2_open) { p.gap2_open = *gap2_open; p.has_gap2_open = 1; }
        if (gap2_extend) { p.gap2_extend = *gap2_extend; p.has_gap2_extend = 1; }
        return p;
    }
};

enum class AlignmentMode { EditDistance, SinglePieceAffine, TwoPieceAffine };
inline AlignmentMode alignment_mode_from_params(const AlignmentParams& p) {
    if (p.gap2_open && p.gap2_extend) return AlignmentMode::TwoPieceAffine;
    if (p.gap_open == p.gap_extend && p.gap_open == p.mismatch_penalty) return AlignmentMode::EditDistance;
    return AlignmentMode::SinglePieceAffine;
}

struct AlignmentResult {
    size_t query_idx = 0, target_idx = 0;
    size_t query_start = 0, query_end = 0, target_start = 0, target_end = 0;
    bool is_reverse = false;
    std::vector<uint8_t> cigar_bytes;  // WFA2 letters; filled only when requested
    int32_t score = 0;
    size_t num_matches = 0, alignment_length = 0;
    std::string cigar;  // cigar_bytes_to_string(cigar_bytes), produced on the GPU
    std::string paf;    // alignment_to_paf(result, sequences), produced on the GPU
};

struct SparsificationStrategy {
    enum Kind { None, Random, Auto, Connectivity, TreeSampling } kind = None;
    double value = 0.0;  // Random: keep fraction; Connectivity: giant-component probability
    size_t k_nearest = 0, k_farthest = 0;
    double random_fraction = 0.0;
    std::optional<size_t> kmer_size;
    static SparsificationStrategy none() { return {}; }
    static SparsificationStrategy random(double f) { SparsificationStrategy s; s.kind = Random; s.value = f; return s; }
    static SparsificationStrategy automatic() { SparsificationStrategy s; s.kind = Auto; return s; }
    static SparsificationStrategy connectivity(double p) { SparsificationStrategy s; s.kind = Connectivity; s.value = p; return s; }
    static SparsificationStrategy tree(size_t kn, size_t kf, double rf, std::optional<size_t> k = std::nullopt) {
        SparsificationStrategy s; s.kind = TreeSampling; s.k_nearest = kn; s.k_farthest = kf; s.random_fraction = rf; s.kmer_size = k; return s;
    }
};

// ---- parse_scores (src/lib.rs:116-153) ----
inline AlignmentParams parse_scores(const std::string& scores_str) {
    std::vector<int32_t> v;
    size_t b = 0;
    for (;;) {
        size_t e = scores_str.find(',', b);
        std::string tok = scores_str.substr(b, e == std::string::npos ? std::string::npos : e - b);
        size_t l = tok.find_first_not_of(" \t\n\r\f\v"), r = tok.find_last_not_of(" \t\n\r\f\v");
        tok = l == std::string::npos ? "" : tok.substr(l, r - l + 1);
        size_t i = 0;
        bool neg = false;
        if (i < tok.size() && (tok[i] == '+' || tok[i] == '-')) neg = tok[i++] == '-';
        if (i >= tok.size()) throw std::invalid_argument("Failed to parse scores: invalid digit found in string");
        int64_t x = 0;
        for (; i < tok.size(); ++i) {
            if (tok[i] < '0' || tok[i] > '9') throw std::invalid_argument("Failed to parse scores: invalid digit found in string");
            x = x * 10 + (tok[i] - '0');
            if (x > (int64_t)INT32_MAX + 1) throw std::invalid_argument("Failed to parse scores: number too large to fit in target type");
        }
        if (neg) x = -x;
        if (x > INT32_MAX || x < INT32_MIN) throw std::invalid_argument("Failed to parse scores: number too large to fit in target type");
        v.push_back((int32_t)x);
        if (e == std::string::npos) break;
        b = e + 1;
    }
    if (v.size() != 4 && v.size() != 6)
        throw std::invalid_argument("Invalid number of scores: " + std::to_string(v.size()) + ". Expected 4 or 6 values.");
    AlignmentParams p;
    p.match_score = v[0];
    p.mismatch_penalty = v[1];
    p.gap_open = v[2];
    p.gap_extend = v[3];
    if (v.size() == 6) {
        p.gap2_open = v[4];
        p.gap2_extend = v[5];
    } else {
        p.gap2_open.reset();
        p.gap2_extend.reset();
    }
    return p;
}

// ---- the -p grammar (src/main.rs:136-203) ----
inline SparsificationStrategy parse_sparsification(const std::string& s) {
    auto parse_f = [](const std::string& t, const char* msg) -> double {
        try {
            size_t pos = 0;
            double v = std::stod(t, &pos);
            if (pos != t.size()) throw std::invalid_argument(msg);
            return v;
        } catch (const std::exception&) { throw std::invalid_argument(msg); }
    };
    auto parse_u = [](const std::string& t, const char* msg) -> size_t {
        if (t.empty()) throw std::invalid_argument(msg);
        size_t v = 0;
        size_t i = (t[0] == '+') ? 1 : 0;
        if (i >= t.size()) throw std::invalid_argument(msg);
        for (; i < t.size(); ++i) {
            if (t[i] < '0' || t[i] > '9') throw std::invalid_argument(msg);
            v = v * 10 + (size_t)(t[i] - '0');
        }
        return v;
    };
    if (s == "none") return SparsificationStrategy::none();
    if (s == "auto") return SparsificationStrategy::automatic();
    if (s.rfind("random:", 0) == 0) {
        double f = parse_f(s.substr(7), "Invalid random fraction");
        if (f <= 0.0 || f > 1.0) throw std::invalid_argument("Random fraction must be between 0 and 1");
        return SparsificationStrategy::random(f);
    }
    if (s.rfind("giant:", 0) == 0 || s.rfind("connectivity:", 0) == 0) {
        const bool giant = s[0] == 'g';
        double p = parse_f(s.substr(giant ? 6 : 13), giant ? "Invalid giant component probability" : "Invalid connectivity probability");
        if (p <= 0.0 || p >= 1.0)
            throw std::invalid_argument(giant ? "Giant component probability must be between 0 and 1" : "Connectivity probability must be between 0 and 1");
        return SparsificationStrategy::connectivity(p);
    }
    if (s.rfind("tree:", 0) == 0) {
        std::vector<std::string> parts;
        std::string rest = s.substr(5);
        size_t b = 0;
        for (;;) {
            size_t e = rest.find(':', b);
            parts.push_back(rest.substr(b, e == std::string::npos ? std::string::npos : e - b));
            if (e == std::string::npos) break;
            b = e + 1;
        }
        if (parts.size() < 3 || parts.size() > 4)
            throw std::invalid_argument("Invalid tree format. Use: tree:<k_nearest>:<k_farthest>:<random_fraction>[:<kmer_size>]");
        size_t kn = parse_u(parts[0], "Invalid k nearest count"), kf = parse_u(parts[1], "Invalid k farthest count");
        double rf = parse_f(parts[2], "Invalid random fraction");
        if (kn == 0 && kf == 0) throw std::invalid_argument("At least one of k_nearest or k_farthest must be greater than 0");
        if (!(rf >= 0.0 && rf <= 1.0)) throw std::invalid_argument("Random fraction must be between 0 and 1");
        std::optional<size_t> k;
        if (parts.size() == 4) {
            size_t kk = parse_u(parts[3], "Invalid k-mer size");
            if (kk < 3 || kk > 31) throw std::invalid_argument("K-mer size must be between 3 and 31");
            k = kk;
        }
        return SparsificationStrategy::tree(kn, kf, rf, k);
    }
    throw std::invalid_argument("Invalid sparsification strategy. Use: none, auto, giant:<probability>, random:<fraction>, or tree:<near>:<far>:<random>[:<kmer>]");
}

// ---- Rust DefaultHasher over a str: SipHash-1-3, zero keys, bytes || 0xFF (SURVEY Appendix B) ----
inline uint64_t default_hash_str(const std::string& s) {
    auto rotl = [](uint64_t x, int b) { return (x << b) | (x >> (64 - b)); };
    uint64_t v0 = 0x736f6d6570736575ULL, v1 = 0x646f72616e646f6dULL, v2 = 0x6c7967656e657261ULL, v3 = 0x7465646279746573ULL;
    auto round = [&]() {
        v0 += v1; v1 = rotl(v1, 13); v1 ^= v0; v0 = rotl(v0, 32);
        v2 += v3; v3 = rotl(v3, 16); v3 ^= v2;
        v0 += v3; v3 = rotl(v3, 21); v3 ^= v0;
        v2 += v1; v1 = rotl(v1, 17); v1 ^= v2; v2 = rotl(v2, 32);
    };
    std::string m = s;
    m.push_back((char)0xFF);
    size_t i = 0, len = m.size();
    for (; i + 8 <= len; i += 8) {
        uint64_t w = 0;
        for (int j = 0; j < 8; ++j) w |= (uint64_t)(uint8_t)m[i + j] << (8 * j);
        v3 ^= w; round(); v0 ^= w;
    }
    uint64_t b = (uint64_t)(len & 0xff) << 56;
    for (int j = 0; i + j < len; ++j) b |= (uint64_t)(uint8_t)m[i + j] << (8 * j);
    v3 ^= b; round(); v0 ^= b;
    v2 ^= 0xff;
    round(); round(); round();
    return v0 ^ v1 ^ v2 ^ v3;
}

// hash("idA:idB") as f64 / u64::MAX as f64 < fraction (src/iterator.rs:262-280, src/knn_graph.rs:161-174)
inline bool keep_pair(const std::string& a, const std::string& b, double fraction) {
    const uint64_t h = default_hash_str(a + ":" + b);
    return (double)h / 18446744073709551616.0 < fraction;
}

// src/iterator.rs:300-334
inline double compute_connectivity_probability(size_t n, double connectivity_prob) {
    if (n <= 1) return 1.0;
    const double x = std::min(0.999, std::max(0.001, connectivity_prob));
    if (n <= 10) {
        switch (n) {
            case 2: return 1.0;
            case 3: return 0.8;
            case 4: return 0.7;
            case 5: return 0.6;
            default: return 0.5;
        }
    }
    const double n_f = (double)n, log_n = std::log(n_f), c = -std::log(-std::log(x));
    return std::min(1.0, std::max(0.001, (log_n + c) / n_f));
}

// src/mash.rs:59-74 from the GPU's Jaccard counts
inline double mash_distance_from_counts(uint32_t inter, uint32_t uni, int k) {
    const double j = uni == 0 ? 0.0 : (double)inter / (double)uni;
    if (j <= 0.0) return 1.0;
    const double ratio = (2.0 * j) / (1.0 + j);
    if (ratio <= 0.0) return 1.0;
    return (-1.0 / (double)k) * std::log(ratio);
}

// src/knn_graph.rs:112-143 (stable sort: ties keep ascending neighbour index)
inline std::vector<std::pair<size_t, size_t>> build_knn_graph(const std::vector<std::vector<double>>& dm, size_t k_neighbors, bool farthest) {
    const size_t n = dm.size();
    std::vector<std::pair<size_t, size_t>> pairs;
    for (size_t i = 0; i < n; ++i) {
        std::vector<std::pair<double, size_t>> nb;
        for (size_t j = 0; j < n; ++j)
            if (i != j) nb.emplace_back(dm[i][j], j);
        if (farthest) std::stable_sort(nb.begin(), nb.end(), [](auto& a, auto& b) { return a.first > b.first; });
        else std::stable_sort(nb.begin(), nb.end(), [](auto& a, auto& b) { return a.first < b.first; });
        for (size_t q = 0; q < std::min(k_neighbors, nb.size()); ++q) pairs.emplace_back(i, nb[q].second);
    }
    return pairs;
}

// RAII handle of one aw_ctx (one GPU)
class Context {
   public:
    explicit Context(int device = 0) {
        int rc = aw_create(device, &ctx_);
        if (rc != AW_OK) throw std::runtime_error(std::string("aw_create: ") + aw_strerror(rc) + ": " + aw_last_error());
    }
    // non-owning view of a context created elsewhere (e.g. by a foreign-language binding)
    Context(aw_ctx* borrowed, bool own) : ctx_(borrowed), own_(own) {}
    ~Context() {
        if (own_) aw_destroy(ctx_);
    }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    aw_ctx* get() const { return ctx_; }
    void load(const std::vector<Sequence>& seqs) {
        std::vector<const uint8_t*> p(seqs.size());
        std::vector<uint64_t> l(seqs.size());
        std::vector<const char*> ids(seqs.size());
        for (size_t i = 0; i < seqs.size(); ++i) {
            p[i] = seqs[i].seq.data();
            l[i] = seqs[i].seq.size();
            ids[i] = seqs[i].id.c_str();
        }
        int rc = aw_load_sequences(ctx_, (uint32_t)seqs.size(), p.data(), l.data(), ids.data());
        if (rc != AW_OK) throw std::runtime_error(std::string("aw_load_sequences: ") + aw_strerror(rc) + ": " + aw_last_error());
    }

   private:
    aw_ctx* ctx_ = nullptr;
    bool own_ = true;
};

// src/knn_graph.rs:12-52; the sketches and the n^2 Jaccard counts come from the GPU (sequences must be loaded)
inline std::vector<std::pair<size_t, size_t>> extract_tree_pairs(Context& ctx, const std::vector<Sequence>& seqs, size_t k_nearest, size_t k_farthest,
                                                                 double random_fraction, size_t kmer_size) {
    const size_t n = seqs.size();
    std::vector<std::pair<size_t, size_t>> all;
    if (n < 2) return all;
    std::vector<uint32_t> inter(n * n), uni(n * n);
    int rc = aw_mash_jaccard_counts(ctx.get(), (int)kmer_size, 1000, inter.data(), uni.data());
    if (rc != AW_OK) throw std::runtime_error(std::string("aw_mash_jaccard_counts: ") + aw_strerror(rc) + ": " + aw_last_error());
    std::vector<std::vector<double>> dm(n, std::vector<double>(n, 0.0));
    for (size_t i = 0; i < n; ++i)
        for (size_t j = i + 1; j < n; ++j) dm[i][j] = dm[j][i] = mash_distance_from_counts(inter[i * n + j], uni[i * n + j], (int)kmer_size);
    if (k_nearest > 0) {
        auto p = build_knn_graph(dm, k_nearest, false);
        all.insert(all.end(), p.begin(), p.end());
    }
    if (k_farthest > 0) {
        auto p = build_knn_graph(dm, k_farthest, true);
        all.insert(all.end(), p.begin(), p.end());
    }
    if (random_fraction > 0.0)
        for (size_t i = 0; i < n; ++i)
            for (size_t j = 0; j < n; ++j)
                if (i != j && keep_pair(seqs[i].id, seqs[j].id, random_fraction)) all.emplace_back(i, j);
    std::sort(all.begin(), all.end());
    all.erase(std::unique(all.begin(), all.end()), all.end());
    return all;
}

// the ordered pair list of AllPairIterator::with_options (src/iterator.rs:37-77)
inline std::vector<std::pair<size_t, size_t>> build_pair_list(Context& ctx, const std::vector<Sequence>& sequences, bool exclude_self,
                                                              const SparsificationStrategy& sp) {
    const size_t n = sequences.size();
    if (sp.kind == SparsificationStrategy::TreeSampling)
        return extract_tree_pairs(ctx, sequences, sp.k_nearest, sp.k_farthest, sp.random_fraction, sp.kmer_size.value_or(15));
    double keep = 1.0;
    bool filter = true;
    if (sp.kind == SparsificationStrategy::None) filter = false;
    else if (sp.kind == SparsificationStrategy::Random) keep = sp.value;
    else if (sp.kind == SparsificationStrategy::Auto) keep = compute_connectivity_probability(n, 0.95);
    else keep = compute_connectivity_probability(n, sp.value);
    std::vector<std::pair<size_t, size_t>> pairs;
    for (size_t i = 0; i < n; ++i)
        for (size_t j = 0; j < n; ++j) {
            if (exclude_self && i == j) continue;
            if (filter && !keep_pair(sequences[i].id, sequences[j].id, keep)) continue;
            pairs.emplace_back(i, j);
        }
    return pairs;
}

using Callback = std::function<void(const AlignmentResult&)>;  // throw to abort the run (mirrors a callback Err)

// ---- multi-GPU sharding (SURVEY 8e): the path shards by independent pairs, every GPU holds the whole sequence store,
// only results are gathered, so there is no collective.  Predicted cost of a pair ~ wavefront cells ~ (expected score)^2 with
// expected score = length x divergence (+ the length difference, which is a forced gap); the divergence comes from the GPU's
// stranded sketches (aw_estimate_divergence) when available.
inline double predicted_pair_cost(uint64_t len_q, uint64_t len_t, double divergence = 0.05) {
    const double s = (double)std::max(len_q, len_t) * std::min(0.5, std::max(divergence, 1e-3)) + (double)(len_q > len_t ? len_q - len_t : len_t - len_q);
    return s * s + (double)(len_q + len_t);
}
// static longest-processing-time-first partition: n_parts lists of indices into `pairs`, each ascending; deterministic.
// (The drivers below use a shared queue of cost-ordered chunks instead, which also absorbs mispredicted costs; the static
// partition remains for callers that must know the shards up front, e.g. one process per GPU.)
inline std::vector<std::vector<size_t>> partition_pairs(const std::vector<std::pair<size_t, size_t>>& pairs, const std::vector<Sequence>& seqs,
                                                        size_t n_parts, const std::vector<float>* divergence = nullptr) {
    std::vector<std::vector<size_t>> shards(std::max<size_t>(1, n_parts));
    if (n_parts <= 1) {
        shards[0].resize(pairs.size());
        for (size_t i = 0; i < pairs.size(); ++i) shards[0][i] = i;
        return shards;
    }
    std::vector<std::pair<double, size_t>> costed(pairs.size());
    for (size_t i = 0; i < pairs.size(); ++i)
        costed[i] = {predicted_pair_cost(seqs[pairs[i].first].seq.size(), seqs[pairs[i].second].seq.size(), divergence ? (double)(*divergence)[i] : 0.05), i};
    std::sort(costed.begin(), costed.end(), [](const auto& a, const auto& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; });
    std::vector<double> load(n_parts, 0.0);
    for (const auto& c : costed) {
        const size_t r = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
        shards[r].push_back(c.second);
        load[r] += c.first;
    }
    for (auto& s : shards) std::sort(s.begin(), s.end());
    return shards;
}

class AllPairIterator {
   public:
    // AllPairIterator::new (src/iterator.rs:25-28) == with_options(seqs, params, true, false, None)
    AllPairIterator(Context& ctx, const std::vector<Sequence>& sequences, const AlignmentParams& params)
        : AllPairIterator(ctx, sequences, params, true, false, SparsificationStrategy()) {}
    // with_options (src/iterator.rs:30-92); the sequences must already be loaded into ctx
    AllPairIterator(Context& ctx, const std::vector<Sequence>& sequences, const AlignmentParams& params, bool exclude_self, bool use_mash_orientation,
                    const SparsificationStrategy& sp)
        : ctx_(ctx), seqs_(sequences), params_(params), orientation_params_(AlignmentParams::edit_distance()), exclude_self_(exclude_self),
          use_mash_(use_mash_orientation) {
        pairs_ = build_pair_list(ctx, sequences, exclude_self, sp);
    }
    AllPairIterator& with_orientation_params(AlignmentParams p) {
        orientation_params_ = std::move(p);
        return *this;
    }
    size_t pair_count() const { return pairs_.size(); }
    // keeps the first n pairs of the list (benchmarks on a bounded, deterministic prefix of a huge job)
    void truncate(size_t n) {
        if (n < pairs_.size()) pairs_.resize(n);
    }
    const std::vector<std::pair<size_t, size_t>>& get_pairs() const { return pairs_; }

    // for_each_with_callback (src/iterator.rs:127-137,208-252): the whole remaining pair list goes to the GPU(s).
    // `others` are further contexts (GPUs) that hold the same sequences.  The callback may throw: the first exception
    // cancels the run on every GPU (no further chunk is started, chunks in flight are dropped) and is rethrown here,
    // like the reference's first-error capture.
    void for_each_with_callback(const Callback& cb, uint32_t flags = 0, const std::vector<Context*>& others = {}) {
        Delivery d;
        d.cb = &cb;
        drive(d, flags, others);
    }
    void for_each_with_callback_multi(const std::vector<Context*>& others, const Callback& cb, uint32_t flags = 0) { for_each_with_callback(cb, flags, others); }
    // PAF writer paths of the CLI (src/main.rs:347-374).  Blocks: newline-terminated PAF lines exactly as they leave the
    // GPU (within a block the lines are in pair order; with one GPU the blocks are too), no per-pair host work at all.
    // `flags` adds aw_align_stream flags, e.g. AW_FLAG_CS for the cs:Z: column.
    using BlockCallback = std::function<void(const char* text, size_t len, size_t n_lines)>;
    void for_each_paf_block(const BlockCallback& cb, const std::vector<Context*>& others = {}, uint32_t flags = 0) {
        Delivery d;
        d.block = &cb;
        drive(d, AW_FLAG_PAF_BLOCKS | flags, others);
    }
    // one call per line (without the newline)
    using PafCallback = std::function<void(const char*, size_t)>;
    void for_each_paf(const PafCallback& cb, const std::vector<Context*>& others = {}) {
        const BlockCallback split = [&](const char* text, size_t len, size_t) {
            const char* p = text;
            const char* end = text + len;
            while (p < end) {
                const char* nl = (const char*)std::memchr(p, '\n', (size_t)(end - p));
                if (!nl) nl = end;
                cb(p, (size_t)(nl - p));
                p = nl + 1;
            }
        };
        for_each_paf_block(split, others);
    }
    // impl Iterator::next (src/iterator.rs:151-171): strictly in pair order; batches are prefetched
    std::optional<AlignmentResult> next() {
        if (buf_pos_ == buffered_.size()) {
            buffered_.clear();
            buf_pos_ = 0;
            if (next_ >= pairs_.size()) return std::nullopt;
            const size_t cnt = std::min<size_t>(prefetch_, pairs_.size() - next_);
            const Callback keep = [&](const AlignmentResult& r) { buffered_.push_back(r); };
            Delivery d;
            d.cb = &keep;
            const size_t saved_end = limit_;
            limit_ = next_ + cnt;
            try {
                drive(d, 0, {});
            } catch (...) {
                limit_ = saved_end;
                throw;
            }
            limit_ = saved_end;
        }
        return buffered_[buf_pos_++];
    }
    void set_prefetch(size_t n) { prefetch_ = n ? n : 1; }
    // pairs per chunk handed to a GPU at a time (0 = automatic)
    void set_chunk_pairs(size_t n) { chunk_pairs_ = n; }
    // max / mean of the per-GPU busy time of the last multi-GPU run (1.0 = perfectly balanced)
    double last_imbalance() const { return last_imbalance_; }

   private:
    struct Delivery {
        const Callback* cb = nullptr;
        const BlockCallback* block = nullptr;
    };
    // one per run, shared by all GPU threads: the cost-ordered pair list, the chunk cursor, the first error
    struct Shared {
        std::vector<aw_pair> pairs;
        std::vector<size_t> chunk_begin;  // chunk c = pairs[chunk_begin[c] .. chunk_begin[c + 1])
        std::atomic<size_t> next{0};
        std::atomic<bool> cancel{false};
        std::mutex mu;  // serialises the user's callback (completion order, like the reference's rayon workers) and `err`
        std::exception_ptr err;
        Delivery d;
        uint32_t flags = 0;
    };
    static uint64_t next_chunk(void* user, const aw_pair** out) {
        Shared* sh = static_cast<Shared*>(user);
        if (sh->cancel.load(std::memory_order_relaxed)) return 0;
        const size_t c = sh->next.fetch_add(1);
        if (c + 1 >= sh->chunk_begin.size()) return 0;
        *out = sh->pairs.data() + sh->chunk_begin[c];
        return sh->chunk_begin[c + 1] - sh->chunk_begin[c];
    }
    static int fail(Shared* sh) {
        std::lock_guard<std::mutex> g(sh->mu);  // callers hold no lock
        if (!sh->err) sh->err = std::current_exception();
        sh->cancel.store(true);
        return 1;
    }
    static int c_callback(const aw_result* r, void* user) {
        Shared* sh = static_cast<Shared*>(user);
        if (sh->cancel.load(std::memory_order_relaxed)) return 1;
        AlignmentResult a;
        a.query_idx = r->query_idx;
        a.target_idx = r->target_idx;
        a.query_start = r->query_start;
        a.query_end = r->query_end;
        a.target_start = r->target_start;
        a.target_end = r->target_end;
        a.is_reverse = r->is_reverse != 0;
        a.score = r->score;
        a.num_matches = r->num_matches;
        a.alignment_length = r->alignment_length;
        if (r->cigar_bytes) a.cigar_bytes.assign(r->cigar_bytes, r->cigar_bytes + r->cigar_len);
        if (r->cg) a.cigar.assign(r->cg, r->cg_len);
        if (r->paf) a.paf.assign(r->paf, r->paf_len);
        try {
            std::lock_guard<std::mutex> g(sh->mu);
            if (sh->cancel.load()) return 1;
            (*sh->d.cb)(a);
        } catch (...) {
            return fail(sh);
        }
        return 0;
    }
    static int c_block(const char* text, uint64_t len, uint64_t n_lines, void* user) {
        Shared* sh = static_cast<Shared*>(user);
        if (sh->cancel.load(std::memory_order_relaxed)) return 1;
        try {
            std::lock_guard<std::mutex> g(sh->mu);
            if (sh->cancel.load()) return 1;
            (*sh->d.block)(text, (size_t)len, (size_t)n_lines);
        } catch (...) {
            return fail(sh);
        }
        return 0;
    }
    // the parallel driver (src/iterator.rs:208-252): one host thread per GPU pulls chunks from the shared queue and streams
    // them through aw_align_stream (two batches in flight per GPU).  With several GPUs the list is first ordered by
    // predicted cost, heaviest first, so that the chunks handed out last are the cheap ones.
    void drive(const Delivery& d, uint32_t flags, const std::vector<Context*>& others) {
        std::vector<Context*> ctxs{&ctx_};
        ctxs.insert(ctxs.end(), others.begin(), others.end());
        const size_t first = next_, last = std::min(limit_, pairs_.size());
        next_ = last;
        if (first >= last) return;
        Shared sh;
        sh.d = d;
        sh.flags = flags;
        sh.pairs.resize(last - first);
        for (size_t i = first; i < last; ++i) sh.pairs[i - first] = aw_pair{(uint32_t)pairs_[i].first, (uint32_t)pairs_[i].second};
        const size_t n = sh.pairs.size(), g_n = ctxs.size();
        const aw_params p = params_.to_c();
        if (!use_mash_) {
            const aw_params op = orientation_params_.to_c();
            for (Context* c : ctxs) {
                int rco = aw_set_orientation_params(c->get(), &op);
                if (rco != AW_OK) throw std::runtime_error(std::string("aw_set_orientation_params: ") + aw_strerror(rco) + ": " + aw_last_error());
            }
        }
        // chunks: a launch should carry enough pairs to keep its tail short -- reads by the hundred thousand, >= ~8 pairs per
        // resident CTA for kb-scale pairs, one pair per resident CTA for Mb-scale pairs (which run for minutes each) -- and
        // every GPU should get several chunks when there are enough pairs
        size_t max_len = 0;
        for (const auto& sq : seqs_) max_len = std::max(max_len, sq.seq.size());
        const size_t lo = max_len <= 1024 ? 65536 : (max_len <= 50000 ? 4736 : 296), hi = max_len <= 1024 ? 262144 : 65536;
        size_t n_chunks = chunk_pairs_ ? (n + chunk_pairs_ - 1) / chunk_pairs_ : std::max<size_t>(std::max<size_t>(g_n, (n + hi - 1) / hi), std::min<size_t>(12 * g_n, n / lo));
        n_chunks = std::max<size_t>(1, std::min(n_chunks, n));
        if (g_n > 1 && max_len > 1024) {
            // several GPUs (reads up to 1 kb cost about the same each: no ordering, the queue alone balances them):
            // order by predicted cost, heaviest first, and deal the list out to the chunks like cards (chunk c =
            // pairs c, c + C, c + 2C, ... of the ordered list): every chunk carries the same cost mix, the shared queue absorbs
            // what the prediction misses, and inside a launch the heavy pairs start first
            std::vector<float> div;
            if (use_mash_) {
                div.resize(n);
                int rc = aw_estimate_divergence(ctx_.get(), sh.pairs.data(), n, div.data());
                if (rc != AW_OK) throw std::runtime_error(std::string("aw_estimate_divergence: ") + aw_strerror(rc) + ": " + aw_last_error());
            }
            std::vector<std::pair<double, uint32_t>> costed(n);
            for (size_t i = 0; i < n; ++i)
                costed[i] = {predicted_pair_cost(seqs_[sh.pairs[i].query_idx].seq.size(), seqs_[sh.pairs[i].target_idx].seq.size(), div.empty() ? 0.05 : (double)div[i]),
                             (uint32_t)i};
            std::stable_sort(costed.begin(), costed.end(), [](const auto& a, const auto& b) { return a.first > b.first; });
            std::vector<aw_pair> ordered;
            ordered.reserve(n);
            sh.chunk_begin.push_back(0);
            for (size_t c = 0; c < n_chunks; ++c) {
                for (size_t i = c; i < n; i += n_chunks) ordered.push_back(sh.pairs[costed[i].second]);
                sh.chunk_begin.push_back(ordered.size());
            }
            sh.pairs.swap(ordered);
        } else {  // one GPU: the list stays in pair order (so does the output), cut into equal chunks
            for (size_t c = 0; c <= n_chunks; ++c) sh.chunk_begin.push_back(c * n / n_chunks);
        }
        std::vector<double> busy(g_n, 0.0);
        std::vector<int> rcs(g_n, AW_OK);
        std::vector<std::string> msgs(g_n);
        auto work = [&](size_t g) {
            const auto t0 = std::chrono::steady_clock::now();
            rcs[g] = aw_align_stream(ctxs[g]->get(), &p, use_mash_ ? AW_ORIENT_MASH : AW_ORIENT_WFA, flags, &next_chunk, &sh, d.cb ? &c_callback : nullptr,
                                     d.block ? &c_block : nullptr, &sh);
            if (rcs[g] != AW_OK && rcs[g] != AW_ECALLBACK) {
                msgs[g] = std::string("aw_align_stream: ") + aw_strerror(rcs[g]) + ": " + aw_last_error();
                sh.cancel.store(true);  // a device error on one GPU stops the others too
            }
            busy[g] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        };
        if (g_n == 1) {
            work(0);
        } else {
            std::vector<std::thread> th;
            for (size_t g = 0; g < g_n; ++g) th.emplace_back(work, g);
            for (auto& t : th) t.join();
        }
        double mx = 0.0, sum = 0.0;
        for (double b : busy) {
            mx = std::max(mx, b);
            sum += b;
        }
        last_imbalance_ = sum > 0.0 ? mx / (sum / (double)g_n) : 1.0;
        if (sh.err) std::rethrow_exception(sh.err);
        for (size_t g = 0; g < g_n; ++g)
            if (rcs[g] != AW_OK && rcs[g] != AW_ECALLBACK) throw std::runtime_error(msgs[g]);
    }
    Context& ctx_;
    const std::vector<Sequence>& seqs_;
    AlignmentParams params_, orientation_params_;
    bool exclude_self_, use_mash_;
    std::vector<std::pair<size_t, size_t>> pairs_;
    size_t next_ = 0, limit_ = (size_t)-1, prefetch_ = 4096, buf_pos_ = 0, chunk_pairs_ = 0;
    double last_imbalance_ = 1.0;
    std::vector<AlignmentResult> buffered_;
};

// src/lib.rs:57-68
inline void process_alignments_with_callback(Context& ctx, const std::vector<Sequence>& sequences, AlignmentParams params, const SparsificationStrategy& sp,
                                             const Callback& cb) {
    AllPairIterator it(ctx, sequences, std::move(params), true, true, sp);
    it.for_each_with_callback(cb);
}

// src/lib.rs:71-112: the PAF line is produced on the GPU together with the CIGAR
inline const std::string& alignment_to_paf(const AlignmentResult& r, const std::vector<Sequence>&) { return r.paf; }

// ---- src/wfa.rs: the legacy one-pair entry point (test-only caller in the reference), over the aw_aligner_* calls ----
namespace wfa {
enum class Mode { EditDistance, SinglePieceAffine, TwoPieceAffine };  // src/wfa.rs:7-12
struct Penalties {                                                      // src/wfa.rs:27-33
    int32_t mismatch, gap_opening1, gap_extension1, gap_opening2, gap_extension2;
};
struct Result {  // src/wfa.rs:35-47; insertions / deletions in the standard (PAF) convention, i.e. WFA2's D / I
    int32_t score = 0;
    std::string cigar;
    size_t matches = 0, mismatches = 0, insertions = 0, deletions = 0, alignment_length = 0;
};
struct AlignmentError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// src/wfa.rs:105-176: the op string must be made of M = X I D only, stay inside both sequences and consume both completely
// (WFA2 letters: I consumes the reference/text, D the query/pattern).  Returns the reference's message, empty when valid.
inline std::string validate_cigar_alignment(const uint8_t* cigar, size_t n, size_t query_len, size_t reference_len) {
    size_t q = 0, r = 0;
    char buf[160];
    for (size_t i = 0; i < n; ++i) {
        const uint8_t op = cigar[i];
        if (op == 'M' || op == '=' || op == 'X') {
            if (q >= query_len || r >= reference_len) {
                std::snprintf(buf, sizeof(buf), "CIGAR extends beyond sequences at M/=/X op: q_pos=%zu, r_pos=%zu, query_len=%zu, ref_len=%zu", q, r, query_len, reference_len);
                return buf;
            }
            ++q;
            ++r;
        } else if (op == 'I') {
            if (r >= reference_len) {
                std::snprintf(buf, sizeof(buf), "CIGAR extends beyond reference at I op: r_pos=%zu, ref_len=%zu", r, reference_len);
                return buf;
            }
            ++r;
        } else if (op == 'D') {
            if (q >= query_len) {
                std::snprintf(buf, sizeof(buf), "CIGAR extends beyond query at D op: q_pos=%zu, query_len=%zu", q, query_len);
                return buf;
            }
            ++q;
        } else {
            std::snprintf(buf, sizeof(buf), "Invalid CIGAR operation: %c (0x%02x)", (char)op, (unsigned)op);
            return buf;
        }
    }
    if (q != query_len) {
        std::snprintf(buf, sizeof(buf), "CIGAR doesn't cover full query: %zu vs %zu", q, query_len);
        return buf;
    }
    if (r != reference_len) {
        std::snprintf(buf, sizeof(buf), "CIGAR doesn't cover full reference: %zu vs %zu", r, reference_len);
        return buf;
    }
    return std::string();
}

// src/wfa.rs:49-83: run-length encode, M -> '=', X -> 'X', I -> 'D', D -> 'I', anything else '?'
inline std::string cigar_bytes_to_string(const uint8_t* cigar, size_t n) {
    std::string out;
    for (size_t i = 0; i < n;) {
        size_t j = i + 1;
        while (j < n && cigar[j] == cigar[i]) ++j;
        const uint8_t op = cigar[i];
        out += std::to_string(j - i);
        out += (op == 'M') ? '=' : (op == 'X') ? 'X' : (op == 'I') ? 'D' : (op == 'D') ? 'I' : '?';
        i = j;
    }
    return out;
}

// src/wfa.rs:178-258: a fresh aligner per call, configured for an exact global alignment; the CIGAR is validated before use
inline Result align_sequences(Context& ctx, const std::vector<uint8_t>& pattern, const std::vector<uint8_t>& text, const Penalties& pen, Mode mode) {
    aw_aligner* wf = nullptr;
    int rc;
    if (mode == Mode::EditDistance) rc = aw_aligner_new_affine(ctx.get(), 0, pen.mismatch, pen.mismatch, pen.mismatch, AW_MEMORY_ULTRALOW, &wf);
    else if (mode == Mode::SinglePieceAffine) rc = aw_aligner_new_affine(ctx.get(), 0, pen.mismatch, pen.gap_opening1, pen.gap_extension1, AW_MEMORY_ULTRALOW, &wf);
    else rc = aw_aligner_new_affine2p(ctx.get(), 0, pen.mismatch, pen.gap_opening1, pen.gap_extension1, pen.gap_opening2, pen.gap_extension2, AW_MEMORY_ULTRALOW, &wf);
    if (rc != AW_OK) throw AlignmentError(std::string("Alignment failed with status: ") + aw_strerror(rc) + ": " + aw_last_error());
    struct Guard {
        aw_aligner* a;
        ~Guard() { aw_aligner_delete(a); }
    } guard{wf};
    aw_aligner_set_alignment_scope(wf, AW_SCOPE_ALIGNMENT);
    aw_aligner_set_alignment_span(wf, AW_SPAN_END2END);
    aw_aligner_set_heuristic(wf, AW_HEURISTIC_NONE);
    rc = aw_aligner_align(wf, pattern.data(), (int32_t)pattern.size(), text.data(), (int32_t)text.size());
    if (rc != AW_OK) throw AlignmentError(std::string("Alignment failed with status: ") + aw_strerror(rc));
    uint64_t n = 0;
    const uint8_t* ops = aw_aligner_cigar(wf, &n);
    const std::string bad = validate_cigar_alignment(ops, (size_t)n, pattern.size(), text.size());
    if (!bad.empty()) throw AlignmentError("CIGAR validation failed: " + bad);
    Result r;
    r.score = aw_aligner_score(wf);
    r.cigar = cigar_bytes_to_string(ops, (size_t)n);
    for (uint64_t i = 0; i < n; ++i) {  // src/wfa.rs:85-103
        r.matches += ops[i] == 'M';
        r.mismatches += ops[i] == 'X';
        r.deletions += ops[i] == 'I';
        r.insertions += ops[i] == 'D';
    }
    r.alignment_length = r.matches + r.mismatches;
    return r;
}
}  // namespace wfa

// src/alignment.rs:178-190 (API surface only; the aligner uses the device copy)
inline std::vector<uint8_t> reverse_complement(const std::vector<uint8_t>& seq) {
    std::vector<uint8_t> out(seq.size());
    for (size_t i = 0; i < seq.size(); ++i) {
        const uint8_t b = seq[seq.size() - 1 - i];
        out[i] = (b == 'A' || b == 'a') ? 'T' : (b == 'T' || b == 't') ? 'A' : (b == 'C' || b == 'c') ? 'G' : (b == 'G' || b == 'g') ? 'C' : 'N';
    }
    return out;
}

// plain FASTA (src/main.rs:206-234; ids up to the first whitespace).  bgzf input is out of scope (SURVEY 8f rank 2)
// FASTA ingest (src/main.rs:206-234): plain files, and .gz / bgzf files through zlib (bgzf is a series of gzip members,
// which gzread decodes transparently) when the translation unit is built with -DALLWAVE_HAVE_ZLIB -lz
namespace detail {
inline void fasta_line(std::vector<Sequence>& seqs, std::string& line) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.empty()) return;
    if (line[0] == '>') {
        size_t e = line.find_first_of(" \t", 1);
        seqs.push_back(Sequence{line.substr(1, e == std::string::npos ? std::string::npos : e - 1), {}});
    } else if (!seqs.empty()) {
        seqs.back().seq.insert(seqs.back().seq.end(), line.begin(), line.end());
    }
}
}  // namespace detail
inline std::vector<Sequence> read_fasta(const std::string& path) {
    std::vector<Sequence> seqs;
    std::string line;
    if (path.size() > 3 && path.compare(path.size() - 3, 3, ".gz") == 0) {
#ifdef ALLWAVE_HAVE_ZLIB
        gzFile gz = gzopen(path.c_str(), "rb");
        if (!gz) throw std::runtime_error("cannot open " + path);
        gzbuffer(gz, 1 << 20);
        std::vector<char> buf(1 << 20);
        int n;
        while ((n = gzread(gz, buf.data(), (unsigned)buf.size())) > 0) {
            const char* p = buf.data();
            const char* end = p + n;
            while (p < end) {
                const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
                if (!nl) {
                    line.append(p, end);
                    break;
                }
                line.append(p, nl);
                detail::fasta_line(seqs, line);
                line.clear();
                p = nl + 1;
            }
        }
        const bool bad = n < 0;
        gzclose(gz);
        if (bad) throw std::runtime_error("error while decompressing " + path);
        if (!line.empty()) detail::fasta_line(seqs, line);
        return seqs;
#else
        throw std::runtime_error("gzipped FASTA needs a build with zlib (-DALLWAVE_HAVE_ZLIB -lz); decompress first");
#endif
    }
    std::ifstream in(path);
    if (!in) throw std::runtime_error("cannot open " + path);
    while (std::getline(in, line)) detail::fasta_line(seqs, line);
    return seqs;
}

// parse_ani_preset (src/main.rs:83-124): -x 95% | 95 | 0.95 -> score string
inline std::string parse_ani_preset(const std::string& preset) {
    double ani;
    auto parse_num = [](const std::string& s, double& out) -> bool {
        if (s.empty()) return false;
        char* end = nullptr;
        out = std::strtod(s.c_str(), &end);
        return end && *end == 0;
    };
    if (preset.find('.') != std::string::npos) {
        double v;
        if (!parse_num(preset, v) || !(v > 0.0 && v <= 1.0)) throw std::invalid_argument("Invalid ANI value: " + preset + ". Use 0.5-1.0 or 50%-100%");
        ani = v * 100.0;
    } else if (!preset.empty() && preset.back() == '%') {
        double v;
        if (!parse_num(preset.substr(0, preset.size() - 1), v) || !(v >= 50.0 && v <= 100.0))
            throw std::invalid_argument("Invalid ANI percentage: " + preset + ". Use 50%-100%");
        ani = v;
    } else {
        double v;
        if (!parse_num(preset, v) || !(v >= 50.0 && v <= 100.0)) throw std::invalid_argument("Invalid ANI percentage: " + preset + ". Use 50%-100% or 50-100");
        ani = v;
    }
    if (ani >= 95.0) return "0,7,12,2,36,1";
    if (ani >= 85.0) return "0,5,8,2,24,1";
    if (ani >= 75.0) return "0,4,6,2,18,1";
    if (ani >= 65.0) return "0,3,4,1";
    return "0,1,1,1";
}

// -k / -e prefix filters (src/main.rs:237-277); returns the number of sequences removed
inline size_t filter_by_prefixes(std::vector<Sequence>& seqs, const std::string& comma_list, bool keep) {
    std::vector<std::string> prefixes;
    size_t pos = 0;
    while (pos <= comma_list.size()) {
        size_t c = comma_list.find(',', pos);
        if (c == std::string::npos) c = comma_list.size();
        std::string s = comma_list.substr(pos, c - pos);
        const size_t a = s.find_first_not_of(" \t"), b = s.find_last_not_of(" \t");
        prefixes.push_back(a == std::string::npos ? std::string() : s.substr(a, b - a + 1));
        pos = c + 1;
    }
    const size_t before = seqs.size();
    seqs.erase(std::remove_if(seqs.begin(), seqs.end(),
                              [&](const Sequence& s) {
                                  bool any = false;
                                  for (const auto& p : prefixes) any = any || s.id.compare(0, p.size(), p) == 0;
                                  return keep ? !any : any;
                              }),
               seqs.end());
    return before - seqs.size();
}

// --mash-matrix (src/main.rs:280-293, src/mash.rs:141-184): mash distances from the GPU sketches, printed like the reference
inline void print_mash_matrix(Context& ctx, const std::vector<Sequence>& seqs, size_t kmer_size, FILE* out) {
    const size_t n = seqs.size();
    std::vector<uint32_t> inter(std::max<size_t>(1, n * n)), uni(std::max<size_t>(1, n * n));
    if (n >= 1) {
        int rc = aw_mash_jaccard_counts(ctx.get(), (int)kmer_size, 1000, inter.data(), uni.data());
        if (rc != AW_OK) throw std::runtime_error(std::string("aw_mash_jaccard_counts: ") + aw_strerror(rc) + ": " + aw_last_error());
    }
    std::fputs("sequence", out);
    for (const auto& s : seqs) std::fprintf(out, "\t%s", s.id.c_str());
    std::fputc('\n', out);
    for (size_t i = 0; i < n; ++i) {
        std::fputs(seqs[i].id.c_str(), out);
        for (size_t j = 0; j < n; ++j) std::fprintf(out, "\t%.6f", i == j ? 0.0 : mash_distance_from_counts(inter[i * n + j], uni[i * n + j], (int)kmer_size));
        std::fputc('\n', out);
    }
}

}  // namespace allwave
