// host_capi.cpp -- C exports of the C++ host mirror (allwave.hpp) so that tests written in
// Python can check pair scheduling and flag parsing against the oracle.
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "allwave.hpp"

using namespace allwave;

static thread_local std::string g_msg;

extern "C" {

const char* awh_last_message(void) { return g_msg.c_str(); }

int awh_parse_scores(const char* s, aw_params* out) {
    try {
        *out = parse_scores(s).to_c();
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

int awh_parse_sparsification(const char* s, int* kind, double* value, uint64_t* kn, uint64_t* kf, double* rf, int* kmer) {
    try {
        SparsificationStrategy sp = parse_sparsification(s);
        *kind = (int)sp.kind;
        *value = sp.value;
        *kn = sp.k_nearest;
        *kf = sp.k_farthest;
        *rf = sp.random_fraction;
        *kmer = sp.kmer_size ? (int)*sp.kmer_size : 0;
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

double awh_connectivity_probability(uint64_t n, double p) { return compute_connectivity_probability((size_t)n, p); }
uint64_t awh_hash_str(const char* s) { return default_hash_str(s); }
int awh_mode_from_params(const aw_params* p) {
    AlignmentParams a;
    a.match_score = p->match_score;
    a.mismatch_penalty = p->mismatch_penalty;
    a.gap_open = p->gap_open;
    a.gap_extend = p->gap_extend;
    a.gap2_open.reset();
    a.gap2_extend.reset();
    if (p->has_gap2_open) a.gap2_open = p->gap2_open;
    if (p->has_gap2_extend) a.gap2_extend = p->gap2_extend;
    return (int)alignment_mode_from_params(a);
}

// AllPairIterator::with_options(...).get_pairs(); ctx (with the sequences loaded) is needed for the tree strategy only
int awh_pair_list(aw_ctx* ctx, uint64_t n, const char* const* ids, int kind, double value, uint64_t kn, uint64_t kf, double rf, int kmer,
                  int exclude_self, uint64_t** out_pairs, uint64_t* out_n) {
    try {
        std::vector<Sequence> seqs(n);
        for (uint64_t i = 0; i < n; ++i) seqs[i].id = ids[i];
        SparsificationStrategy sp;
        sp.kind = (SparsificationStrategy::Kind)kind;
        sp.value = value;
        sp.k_nearest = kn;
        sp.k_farthest = kf;
        sp.random_fraction = rf;
        if (kmer) sp.kmer_size = (size_t)kmer;
        Context c(ctx, false);
        AllPairIterator it(c, seqs, AlignmentParams(), exclude_self != 0, true, sp);
        const auto& p = it.get_pairs();
        uint64_t* o = (uint64_t*)std::malloc(sizeof(uint64_t) * 2 * (p.size() ? p.size() : 1));
        for (size_t i = 0; i < p.size(); ++i) {
            o[2 * i] = p[i].first;
            o[2 * i + 1] = p[i].second;
        }
        *out_pairs = o;
        *out_n = p.size();
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

uint64_t* awh_build_knn_graph(const double* m, uint64_t n, uint64_t k, int farthest, uint64_t* out_n) {
    std::vector<std::vector<double>> dm(n, std::vector<double>(n));
    for (uint64_t i = 0; i < n; ++i)
        for (uint64_t j = 0; j < n; ++j) dm[i][j] = m[i * n + j];
    auto p = build_knn_graph(dm, (size_t)k, farthest != 0);
    uint64_t* o = (uint64_t*)std::malloc(sizeof(uint64_t) * 2 * (p.size() ? p.size() : 1));
    for (size_t i = 0; i < p.size(); ++i) {
        o[2 * i] = p[i].first;
        o[2 * i + 1] = p[i].second;
    }
    *out_n = p.size();
    return o;
}

// partition_pairs (multi-GPU sharding): out_part[i] = GPU of pair i
int awh_partition_pairs(const uint64_t* pairs, uint64_t npairs, const uint64_t* lens, uint64_t nseq, uint64_t nparts, uint32_t* out_part) {
    try {
        std::vector<Sequence> seqs(nseq);
        for (uint64_t i = 0; i < nseq; ++i) seqs[i].seq.resize(lens[i]);
        std::vector<std::pair<size_t, size_t>> p(npairs);
        for (uint64_t i = 0; i < npairs; ++i) p[i] = {(size_t)pairs[2 * i], (size_t)pairs[2 * i + 1]};
        const auto shards = partition_pairs(p, seqs, (size_t)nparts);
        for (size_t g = 0; g < shards.size(); ++g)
            for (size_t i : shards[g]) out_part[i] = (uint32_t)g;
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

// parse_ani_preset (src/main.rs:83-124): writes the score string into out (>= 32 bytes)
int awh_parse_ani_preset(const char* s, char* out) {
    try {
        const std::string r = parse_ani_preset(s);
        std::strncpy(out, r.c_str(), 31);
        out[31] = 0;
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

// read_fasta + the -k / -e prefix filters: returns the number of sequences, their ids joined by '\n' and their total length
int64_t awh_read_fasta(const char* path, const char* keep, const char* exclude, char** ids_out, uint64_t* total_len) {
    try {
        std::vector<Sequence> seqs = read_fasta(path);
        if (keep && *keep) filter_by_prefixes(seqs, keep, true);
        if (exclude && *exclude) filter_by_prefixes(seqs, exclude, false);
        std::string joined;
        uint64_t tot = 0;
        for (const auto& s : seqs) {
            joined += s.id;
            joined += '\n';
            tot += s.seq.size();
        }
        char* o = (char*)std::malloc(joined.size() + 1);
        std::memcpy(o, joined.c_str(), joined.size() + 1);
        *ids_out = o;
        *total_len = tot;
        return (int64_t)seqs.size();
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

// The whole host path on in-memory sequences over `n_gpus` devices (first_device ..): contexts, sequence upload, pair list
// (-p grammar), the streaming multi-GPU driver, PAF blocks to `out_path` (NULL/"" = discard).  This is what `allwave --gpus N`
// does after reading the FASTA; bench.py uses it for the strong-scaling run through the product path.
//   max_pairs > 0 truncates the pair list (deterministic prefix);  checksum != 0 adds an order-independent digest of the lines
//   out[0] pairs, out[1] PAF bytes, out[2] seconds (alignment: pair list ready -> last byte delivered), out[3] seconds (setup:
//   contexts + upload + pair list), out[4] max/mean GPU busy time, out[5] digest (sum of per-line FNV-1a hashes, as double bits)
int awh_run_job(uint64_t n, const char* const* ids, const uint8_t* const* seqs, const uint64_t* lens, const char* scores, const char* spars, int use_mash,
                int first_device, int n_gpus, uint64_t max_pairs, const char* out_path, int checksum, double* out) {
    try {
        std::vector<Sequence> S(n);
        for (uint64_t i = 0; i < n; ++i) {
            S[i].id = ids[i];
            S[i].seq.assign(seqs[i], seqs[i] + lens[i]);
        }
        const auto t0 = std::chrono::steady_clock::now();
        std::vector<std::unique_ptr<Context>> ctxs((size_t)std::max(1, n_gpus));
        {
            std::vector<std::thread> th;
            std::vector<std::exception_ptr> errs(ctxs.size());
            for (size_t g = 0; g < ctxs.size(); ++g)
                th.emplace_back([&, g] {
                    try {
                        ctxs[g].reset(new Context(first_device + (int)g));
                        ctxs[g]->load(S);
                    } catch (...) {
                        errs[g] = std::current_exception();
                    }
                });
            for (auto& t : th) t.join();
            for (auto& e : errs)
                if (e) std::rethrow_exception(e);
        }
        std::vector<Context*> others;
        for (size_t g = 1; g < ctxs.size(); ++g) others.push_back(ctxs[g].get());
        AllPairIterator it(*ctxs[0], S, parse_scores(scores), true, use_mash != 0, parse_sparsification(spars));
        if (max_pairs) it.truncate(max_pairs);
        FILE* f = (out_path && *out_path) ? std::fopen(out_path, "w") : nullptr;
        if (out_path && *out_path && !f) throw std::runtime_error(std::string("cannot open ") + out_path);
        const auto t1 = std::chrono::steady_clock::now();
        uint64_t bytes = 0, lines = 0, digest = 0;
        it.for_each_paf_block(
            [&](const char* text, size_t len, size_t n_lines) {
                bytes += len;
                lines += n_lines;
                if (f) std::fwrite(text, 1, len, f);
                if (checksum) {
                    uint64_t h = 1469598103934665603ull;
                    for (size_t i = 0; i < len; ++i) {
                        if (text[i] == '\n') {
                            digest += h;
                            h = 1469598103934665603ull;
                        } else {
                            h = (h ^ (uint8_t)text[i]) * 1099511628211ull;
                        }
                    }
                }
            },
            others);
        const auto t2 = std::chrono::steady_clock::now();
        if (f) std::fclose(f);
        out[0] = (double)lines;
        out[1] = (double)bytes;
        out[2] = std::chrono::duration<double>(t2 - t1).count();
        out[3] = std::chrono::duration<double>(t1 - t0).count();
        out[4] = it.last_imbalance();
        std::memcpy(&out[5], &digest, 8);
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

// callback-error cancellation (src/iterator.rs:235-251) through the C++ wrapper: the callback throws at its
// `fail_at`-th result; returns the number of results delivered before the run stopped, -1 if nothing was thrown back
int64_t awh_test_cancel(aw_ctx* ctx, uint64_t n, const char* const* ids, const uint64_t* lens, uint64_t fail_at, uint64_t chunk_pairs, char* msg_out /*>=128*/) {
    std::vector<Sequence> S(n);
    for (uint64_t i = 0; i < n; ++i) {
        S[i].id = ids[i];
        S[i].seq.resize(lens[i]);  // lengths only: the sequences are already loaded in ctx
    }
    Context c(ctx, false);
    AllPairIterator it(c, S, AlignmentParams(), true, true, SparsificationStrategy::none());
    it.set_chunk_pairs(chunk_pairs);
    uint64_t seen = 0;
    try {
        it.for_each_with_callback([&](const AlignmentResult&) {
            if (++seen == fail_at) throw std::runtime_error("callback failed on purpose");
        });
    } catch (const std::exception& e) {
        std::strncpy(msg_out, e.what(), 127);
        msg_out[127] = 0;
        return (int64_t)seen;
    }
    return -1;
}

// for_each_with_callback with the given aw_align_pairs flags (e.g. AW_FLAG_SCORE_ONLY) over all ordered pairs of the loaded
// sequences, default AlignmentParams, mash orientation.  Per result, 8 values in `rows` (room for `cap` results): query_idx,
// target_idx, score, is_reverse, query_end, target_end, cigar string length, PAF length.  Returns the number of results, -1 on error.
int64_t awh_test_for_each(aw_ctx* ctx, uint64_t n, const char* const* ids, const uint64_t* lens, uint32_t flags, int64_t* rows, uint64_t cap) {
    std::vector<Sequence> S(n);
    for (uint64_t i = 0; i < n; ++i) {
        S[i].id = ids[i];
        S[i].seq.resize(lens[i]);  // lengths only: the sequences are already loaded in ctx
    }
    try {
        Context c(ctx, false);
        AllPairIterator it(c, S, AlignmentParams(), true, true, SparsificationStrategy::none());
        uint64_t k = 0;
        it.for_each_with_callback(
            [&](const AlignmentResult& a) {
                if (k < cap) {
                    int64_t* r = rows + 8 * k;
                    r[0] = (int64_t)a.query_idx;
                    r[1] = (int64_t)a.target_idx;
                    r[2] = a.score;
                    r[3] = a.is_reverse ? 1 : 0;
                    r[4] = (int64_t)a.query_end;
                    r[5] = (int64_t)a.target_end;
                    r[6] = (int64_t)a.cigar.size();
                    r[7] = (int64_t)a.paf.size();
                }
                ++k;
            },
            flags);
        return (int64_t)k;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

// wfa::validate_cigar_alignment (src/wfa.rs:105-176): 0 = valid, else 1 with the reference's message in msg_out
int awh_validate_cigar(const uint8_t* cigar, uint64_t n, uint64_t query_len, uint64_t reference_len, char* msg_out /*>=160*/) {
    const std::string m = wfa::validate_cigar_alignment(cigar, (size_t)n, (size_t)query_len, (size_t)reference_len);
    if (msg_out) std::snprintf(msg_out, 160, "%s", m.c_str());
    return m.empty() ? 0 : 1;
}

// wfa::align_sequences (src/wfa.rs:178-258) through the C++ mirror: mode 0 edit, 1 affine, 2 two-piece affine.
// counts = {matches, mismatches, insertions, deletions, alignment_length}; the cigar string is malloc'ed (awh_free)
int awh_align_sequences(aw_ctx* ctx, const uint8_t* pattern, uint64_t plen, const uint8_t* text, uint64_t tlen, const int32_t pen[5], int mode, int32_t* score,
                        uint64_t counts[5], char** cigar_out) {
    try {
        Context c(ctx, false);
        const wfa::Penalties p{pen[0], pen[1], pen[2], pen[3], pen[4]};
        const wfa::Result r = wfa::align_sequences(c, std::vector<uint8_t>(pattern, pattern + plen), std::vector<uint8_t>(text, text + tlen), p,
                                                   mode == 0 ? wfa::Mode::EditDistance : mode == 1 ? wfa::Mode::SinglePieceAffine : wfa::Mode::TwoPieceAffine);
        *score = r.score;
        counts[0] = r.matches;
        counts[1] = r.mismatches;
        counts[2] = r.insertions;
        counts[3] = r.deletions;
        counts[4] = r.alignment_length;
        *cigar_out = (char*)std::malloc(r.cigar.size() + 1);
        std::memcpy(*cigar_out, r.cigar.c_str(), r.cigar.size() + 1);
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return 1;
    }
}

void awh_free(void* p) { std::free(p); }
}
