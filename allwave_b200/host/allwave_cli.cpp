// allwave_cli.cpp -- minimal driver with allwave's CLI surface for the alignment path
// (src/main.rs:32-80): -i FASTA[.gz] [-o PAF] [-s scores | -x ANI preset] [-p strategy] [-t N] [-k prefixes | -e prefixes]
// [--mash-matrix] [--wfa-orientation] [--cs[=short|long]] [--no-progress] [--gpu D] [--gpus N].  FASTA parsing and the PAF writer thread stay on
// the host; everything between the pair list and the ready-to-write PAF text runs on the GPU through liballwave_cuda.so.
#include <chrono>
#include <cstdio>
#include <iostream>
#include <memory>

#include "allwave.hpp"

// bounded single-consumer queue + writer thread (src/main.rs:347-367)
class PafWriter {
   public:
    explicit PafWriter(FILE* out) : out_(out), th_([this] { run(); }) {}
    ~PafWriter() { close(); }
    void push(const char* text, size_t len) {
        std::string blk(text, len);
        std::unique_lock<std::mutex> g(mu_);
        not_full_.wait(g, [&] { return bytes_ < kMaxBytes; });
        bytes_ += blk.size();
        q_.push_back(std::move(blk));
        not_empty_.notify_one();
    }
    void close() {
        {
            std::lock_guard<std::mutex> g(mu_);
            if (closed_) return;
            closed_ = true;
        }
        not_empty_.notify_one();
        th_.join();
        if (failed_) throw std::runtime_error("error while writing the PAF output");
    }

   private:
    void run() {
        for (;;) {
            std::string blk;
            {
                std::unique_lock<std::mutex> g(mu_);
                not_empty_.wait(g, [&] { return !q_.empty() || closed_; });
                if (q_.empty()) return;
                blk = std::move(q_.front());
                q_.pop_front();
                bytes_ -= blk.size();
            }
            not_full_.notify_one();
            if (std::fwrite(blk.data(), 1, blk.size(), out_) != blk.size()) failed_ = true;
        }
    }
    static constexpr size_t kMaxBytes = 1ull << 30;
    FILE* out_;
    std::mutex mu_;
    std::condition_variable not_empty_, not_full_;
    std::deque<std::string> q_;
    size_t bytes_ = 0;
    bool closed_ = false, failed_ = false;
    std::thread th_;
};

int main(int argc, char** argv) {
    std::string input, output, scores = "0,5,8,2,24,1", spars = "giant:0.99", preset, keep_prefixes, exclude_prefixes;
    bool wfa_orientation = false, progress = true, mash_matrix = false, scores_given = false;
    int device = 0, gpus = 1, threads = 1;
    uint32_t cs_flags = 0;  // --cs: minimap2's cs:Z: column on every PAF line (short form; --cs=long: long form)
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "error: %s needs a value\n", name);
                std::exit(2);
            }
            return argv[++i];
        };
        if (a == "-i" || a == "--input") input = need("-i");
        else if (a == "-o" || a == "--output") output = need("-o");
        else if (a == "-s" || a == "--scores") {
            scores = need("-s");
            scores_given = true;
        } else if (a == "-x" || a == "--preset") preset = need("-x");
        else if (a == "-k" || a == "--keep-prefixes") keep_prefixes = need("-k");
        else if (a == "-e" || a == "--exclude-prefixes") exclude_prefixes = need("-e");
        else if (a == "--mash-matrix") mash_matrix = true;
        else if (a == "-p" || a == "--sparsification") spars = need("-p");
        else if (a == "-t" || a == "--threads") threads = std::max(1, std::atoi(need("-t").c_str()));
        else if (a == "--gpu") device = std::atoi(need("--gpu").c_str());
        else if (a == "--gpus") gpus = std::max(1, std::atoi(need("--gpus").c_str()));  // devices device .. device+gpus-1, pairs sharded by predicted cost
        else if (a == "--wfa-orientation") wfa_orientation = true;
        else if (a == "--cs" || a == "--cs=short") cs_flags = AW_FLAG_CS;
        else if (a == "--cs=long") cs_flags = AW_FLAG_CS | AW_FLAG_CS_LONG;
        else if (a.rfind("--cs=", 0) == 0) {
            std::fprintf(stderr, "error: --cs takes 'short' or 'long', not '%s'\n", a.c_str() + 5);
            return 2;
        }
        else if (a == "--no-progress") progress = false;
        else {
            std::fprintf(stderr,
                         "usage: allwave -i FASTA[.gz] [-o PAF] [-s scores | -x ANI] [-p none|auto|random:f|giant:p|tree:n:f:r[:k]] [-k prefixes | -e prefixes]\n"
                         "               [--mash-matrix] [--wfa-orientation] [--cs[=short|long]] [--no-progress] [--gpu D] [--gpus N]\n");
            return 2;
        }
    }
    if (!preset.empty() && scores_given) {  // clap: conflicts_with = "scores"
        std::fprintf(stderr, "error: the argument '--preset <PRESET>' cannot be used with '--scores <SCORES>'\n");
        return 2;
    }
    if (!keep_prefixes.empty() && !exclude_prefixes.empty()) {
        std::fprintf(stderr, "error: the argument '--keep-prefixes <KEEP_PREFIXES>' cannot be used with '--exclude-prefixes <EXCLUDE_PREFIXES>'\n");
        return 2;
    }
    // -t: the reference's rayon pool size.  Accepted for command-line compatibility; the pairs run on the GPU(s), and the host
    // always uses one driver thread per GPU plus one writer thread whatever -t says.
    (void)threads;
    if (input.empty()) {
        std::fprintf(stderr, "error: -i/--input is required\n");
        return 2;
    }
    // ALLWAVE_TIMING=1: wall time of every start-up phase on stderr (where a short job's time goes)
    const bool timing = std::getenv("ALLWAVE_TIMING") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto mark = [&](const char* what) {
        if (timing) std::fprintf(stderr, "[timing] %8.3f s  %s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(), what);
    };
    try {
        using namespace allwave;
        const SparsificationStrategy sp = parse_sparsification(spars);
        std::vector<Sequence> seqs = read_fasta(input);
        mark("FASTA read");
        if (!keep_prefixes.empty()) {
            const size_t before = seqs.size(), removed = filter_by_prefixes(seqs, keep_prefixes, true);
            if (removed) std::fprintf(stderr, "Kept sequences with prefixes: %zu -> %zu (prefixes: %s)\n", before, seqs.size(), keep_prefixes.c_str());
            if (seqs.empty()) throw std::invalid_argument("No sequences match the specified keep prefixes");
        }
        if (!exclude_prefixes.empty()) {
            const size_t before = seqs.size(), removed = filter_by_prefixes(seqs, exclude_prefixes, false);
            if (removed) std::fprintf(stderr, "Excluded sequences with prefixes: %zu -> %zu (prefixes: %s)\n", before, seqs.size(), exclude_prefixes.c_str());
            if (seqs.empty()) throw std::invalid_argument("All sequences were excluded by the specified prefixes");
        }
        Context ctx(device);
        mark("device context created");
        ctx.load(seqs);
        mark("sequences packed and sketched on the device");
        if (mash_matrix) {  // src/main.rs:280-293: print the mash distance matrix and exit
            print_mash_matrix(ctx, seqs, sp.kind == SparsificationStrategy::TreeSampling ? sp.kmer_size.value_or(15) : 15, stdout);
            return 0;
        }
        if (!preset.empty()) {
            scores = parse_ani_preset(preset);
            std::fprintf(stderr, "Using ANI preset %s -> alignment scores: %s\n", preset.c_str(), scores.c_str());
        }
        const AlignmentParams params = parse_scores(scores);
        std::vector<std::unique_ptr<Context>> more;
        std::vector<Context*> others;
        {  // the other GPUs' contexts are created and loaded concurrently (CUDA context creation takes seconds per device)
            more.resize(gpus > 1 ? gpus - 1 : 0);
            std::vector<std::thread> th;
            std::vector<std::exception_ptr> errs(more.size());
            for (size_t g = 0; g < more.size(); ++g)
                th.emplace_back([&, g] {
                    try {
                        more[g].reset(new Context(device + 1 + (int)g));
                        more[g]->load(seqs);
                    } catch (...) {
                        errs[g] = std::current_exception();
                    }
                });
            for (auto& t : th) t.join();
            for (auto& e : errs)
                if (e) std::rethrow_exception(e);
            for (auto& m : more) others.push_back(m.get());
        }
        AllPairIterator it(ctx, seqs, params, true, !wfa_orientation, sp);
        mark("pair list built");
        FILE* out = output.empty() ? stdout : std::fopen(output.c_str(), "w");
        if (!out) throw std::runtime_error("cannot open " + output);
        const auto t0 = std::chrono::steady_clock::now();
        // the writer has its own thread fed through a bounded queue, like the reference's mpsc writer (src/main.rs:347-367):
        // file I/O overlaps the GPUs and the D2H copies; the GPU threads only move a block pointer
        PafWriter writer(out);
        size_t done = 0;
        it.for_each_paf_block(
            [&](const char* text, size_t len, size_t n_lines) {
                writer.push(text, len);
                done += n_lines;
            },
            others, cs_flags);
        mark("last PAF block delivered");
        writer.close();
        if (out != stdout) std::fclose(out);
        mark("output closed");
        const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (progress) std::fprintf(stderr, "[%.1fs] %zu/%zu (100.0%%) %.1f alignments/sec - Complete!\n", dt, done, it.pair_count(), done / std::max(dt, 1e-9));
    } catch (const std::exception& e) {
        std::fprintf(stderr, "Error: %s\n", e.what());
        return 1;
    }
    return 0;
}
