// aw_api.cu -- C-ABI implementation of liballwave_cuda.so (see include/allwave_cuda.h).
// Host plumbing only: sequence store upload, workspace sizing, kernel launches, the retry
// ladder for pairs whose device workspace was too small, result delivery.  All arithmetic of
// the path runs in the kernels of aw_wfa.cuh / aw_sketch.cuh; there is no CPU fallback.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "aw_common.cuh"
#include "aw_sketch.cuh"
#include "aw_wfa.cuh"
#include "aw_cs.cuh"

static thread_local char g_err[512] = "";
void aw_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

// ---- caching allocator: cudaMalloc / cudaFree / cudaHostAlloc synchronise the device and cost 0.1 - 100 ms each, and
// the host-facing calls (aw_load_sequences, aw_align_pairs) need the same few buffers on every call.  Released buffers
// are parked per device (device memory) or globally (pinned host memory) and handed out again best-fit.
struct BufCache {
    std::mutex mu;
    std::multimap<size_t, void*> free_dev[64];
    std::multimap<size_t, void*> free_pin;
    size_t parked_dev[64] = {0}, parked_pin = 0;
    static constexpr size_t kMaxParkedDev = 24ull << 30, kMaxParkedPin = 2ull << 30;
    static size_t round_up(size_t b) {
        const size_t g = b >= (1u << 20) ? (2u << 20) : (64u << 10);
        return ((b ? b : 1) + g - 1) / g * g;
    }
    void* take(std::multimap<size_t, void*>& m, size_t& parked, size_t want, size_t* got) {
        auto it = m.lower_bound(want);
        if (it == m.end() || it->first > 2 * want + (4u << 20)) return nullptr;
        void* p = it->second;
        *got = it->first;
        parked -= it->first;
        m.erase(it);
        return p;
    }
    void trim_dev(int dev) {
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : free_dev[dev]) cudaFree(kv.second);
        free_dev[dev].clear();
        parked_dev[dev] = 0;
    }
    void trim_pin() {
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : free_pin) cudaFreeHost(kv.second);
        free_pin.clear();
        parked_pin = 0;
    }
};
static BufCache g_cache;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int dev = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }  // early returns park the buffer instead of leaking it
    int ensure(size_t bytes) {
        if (bytes <= cap) return AW_OK;
        release();
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
        const size_t want = BufCache::round_up(bytes);
        {
            std::lock_guard<std::mutex> g(g_cache.mu);
            size_t got = 0;
            if (void* q = g_cache.take(g_cache.free_dev[dev], g_cache.parked_dev[dev], want, &got)) {
                p = q;
                cap = got;
                return AW_OK;
            }
        }
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {  // give the parked buffers back to the driver and try once more
            cudaGetLastError();
            g_cache.trim_dev(dev);
            e = cudaMalloc(&p, want);
        }
        if (e != cudaSuccess) {
            p = nullptr;
            aw_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            cudaGetLastError();
            return AW_ENOMEM;
        }
        cap = want;
        return AW_OK;
    }
    void release() {
        if (p) {
            std::lock_guard<std::mutex> g(g_cache.mu);
            if (g_cache.parked_dev[dev] + cap <= BufCache::kMaxParkedDev) {
                g_cache.free_dev[dev].emplace(cap, p);
                g_cache.parked_dev[dev] += cap;
            } else {
                cudaFree(p);
            }
        }
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(const PinBuf&) = delete;
    PinBuf& operator=(const PinBuf&) = delete;
    ~PinBuf() { release(); }
    int ensure(size_t bytes) {
        if (bytes <= cap) return AW_OK;
        release();
        const size_t want = BufCache::round_up(bytes + bytes / 4 + 4096);
        {
            std::lock_guard<std::mutex> g(g_cache.mu);
            size_t got = 0;
            if (void* q = g_cache.take(g_cache.free_pin, g_cache.parked_pin, want, &got)) {
                p = q;
                cap = got;
                return AW_OK;
            }
        }
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
        if (e != cudaSuccess) {
            p = nullptr;
            aw_set_error("cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e));
            cudaGetLastError();
            return AW_ENOMEM;
        }
        cap = want;
        return AW_OK;
    }
    void release() {
        if (p) {
            std::lock_guard<std::mutex> g(g_cache.mu);
            if (g_cache.parked_pin + cap <= BufCache::kMaxParkedPin) {
                g_cache.free_pin.emplace(cap, p);
                g_cache.parked_pin += cap;
            } else {
                cudaFreeHost(p);
            }
        }
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct SketchSet {
    DevBuf sk, n;
    uint32_t count = 0, size = 0;
};

}  // namespace

struct aw_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    // options
    int ctas_per_sm = 0;       // 0 = auto
    int threads_per_cta = 0;   // 0 = auto (32 for short pairs, 256 otherwise)
    int64_t max_w = 1 << 20;   // cap on allocated diagonals per wavefront (first attempt)
    int64_t hist_mb = 16;      // base-case history arena per CTA (first attempt)
    int64_t chunk_pairs = 65536;
    int ws16 = 1;              // 1 = int16 wavefront storage when every offset fits
    int64_t cluster_min_len = 200000;  // pairs at least this long (2-bit sequences, int32 rows) run one pair per thread-block cluster; 0 = never
    int cluster_always = 0;            // tests: use the cluster kernel whatever the batch size
    int64_t solo_len = 65536;          // ... and inside them sub-problems with plen + tlen below this are left to CTA 0 of the cluster
    int max_retry = 3;         // rungs of the retry ladder (0: a pair whose first-try workspace was too small fails)
    // streams: `stream` runs the kernels (they serialise: every launch fills the GPU), `up_stream` uploads the next batch's
    // pair list, `copy_stream` brings the previous batch's results back while the next kernel runs
    cudaStream_t up_stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev_sketch = nullptr;  // recorded after the stranded sketch build; every stream that reads the sketches waits on it
    aw_params orient_params = {0, 1, 1, 1, 0, 0, 0, 0};  // AlignmentParams::edit_distance(), src/iterator.rs:85
    // sequence store
    uint32_t n = 0;
    std::vector<uint64_t> lens;
    std::vector<AwSlot> h_slots;
    std::vector<std::string> ids;
    bool all_clean = true;
    uint64_t max_len = 0;
    DevBuf d_slots, d_ascii, d_packed, d_ids, d_id_off;
    // sketches: stranded (k=15,s=1000) over 2n slots; canonical by (k, size) over n sequences
    SketchSet stranded;
    bool have_stranded = false;
    std::map<std::pair<int, uint32_t>, SketchSet*> canonical;
    // grow-only per-launch workspace.  Two sets: the streaming driver alternates its two batches between them and between
    // two kernel streams, so that the first CTAs of batch k+1 start on the SMs that the tail of batch k leaves idle
    struct Workspace {
        DevBuf ws_main, ws_hist_meta, ws_runs, ws_blk, ws_seq2;
        size_t bytes() const { return ws_main.cap + ws_hist_meta.cap + ws_runs.cap + ws_blk.cap + ws_seq2.cap; }
    } wsp[2];
    cudaStream_t stream2 = nullptr;  // kernel stream of workspace set 1 (set 0 runs on `stream`)
};

// Layout of a batch's control block (aw_batch::d_ctl, and the one of each retry rung), zeroed before every launch: the
// arena cursors and work-list counters its alignment passes advance with atomics.  The --wfa-orientation passes run before
// the main pass and into their own results: each strand has its own next-pair counter, and both share one pair of arena
// cursors.  A next-pair counter is 32 bits wide, in the low word of its slot.
struct BatchCtl {
    unsigned long long text_cursor, bytes_cursor;  // main pass: bytes used in the PAF text and CIGAR byte arenas
    unsigned long long next_pair;                  // main pass: next entry of the work list
    unsigned long long orient_next_pair[2];        // orientation passes: next entry of the work list, per strand
    unsigned long long orient_text_cursor, orient_bytes_cursor;
    unsigned long long tag_cursor;                 // AW_FLAG_CS: bytes used in the tag arena
};

struct aw_batch {
    AwPen pen;
    int orient = AW_ORIENT_MASH;
    uint32_t flags = 0;   // as the caller gave them (AW_FLAG_CS_LONG adds AW_FLAG_CS)
    uint32_t kflags = 0;  // what the alignment passes are told: AW_FLAG_CS needs the CIGAR op bytes, and no kernel reads the CS bits
    uint64_t npairs = 0;
    std::vector<aw_pair> h_pairs;
    DevBuf d_pairs, d_isrev, d_order, d_out, d_text, d_bytes, d_ctl;
    DevBuf d_text2, d_off;              // AW_FLAG_PAF_BLOCKS / AW_FLAG_CS: the text arena again in pair order, and the per-pair offsets (n+1)
    DevBuf d_tags, d_cs_out;            // AW_FLAG_CS: the tag arena and where each pair's tag lies in it
    DevBuf d_out_f, d_out_r, d_strand;  // --wfa-orientation passes: per-strand results and a constant 0.. / 1.. strand array
    AwPen pen_orient;
    uint64_t text_cap = 0, bytes_cap = 0, text2_cap = 0, tag_cap = 0;
    bool has_order = false;
    uint64_t max_p = 0, max_t = 0;
    // host copies
    PinBuf h_out, h_text, h_bytes;
    // retry pass results
    std::vector<AwPairOut> r_out;
    std::vector<uint64_t> r_cs_len;  // AW_FLAG_CS: tag length of each r_out entry (its line in r_text carries the cs column)
    std::vector<uint32_t> r_idx;
    std::vector<char> r_text;
    std::vector<uint8_t> r_bytes;
    uint64_t stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t cyc[6] = {0, 0, 0, 0, 0, 0};
    bool launched = false;
    int slot = 0;                              // workspace set / kernel stream of the context this batch runs on
    cudaStream_t last_stream = nullptr;        // stream of the last launch
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // around the alignment kernel of the last launch
    cudaEvent_t ev_done = nullptr;             // after the last kernel of the launch (what fetch waits for)
};

struct aw_aligner {
    aw_ctx* ctx = nullptr;  // private context on the parent's device
    aw_params params;
    int memory_mode = AW_MEMORY_ULTRALOW;
    int scope = AW_SCOPE_ALIGNMENT;
    int32_t score = 0;
    std::vector<uint8_t> cigar;
};

// ------------------------------------------------------------------------------------------
extern "C" int aw_abi_version(void) { return AW_ABI_VERSION; }
extern "C" const char* aw_last_error(void) { return g_err; }
extern "C" const char* aw_strerror(int s) {
    switch (s) {
        case AW_OK: return "ok";
        case AW_EINVAL: return "invalid argument";
        case AW_ENODEVICE: return "no usable CUDA device";
        case AW_ECUDA: return "CUDA runtime error";
        case AW_ENOMEM: return "out of memory";
        case AW_EUNSUPPORTED: return "unsupported parameter";
        case AW_EWORKSPACE: return "device workspace exhausted";
        case AW_ECALLBACK: return "cancelled by callback";
        case AW_EALIGN: return "alignment failed";
        default: return "unknown status";
    }
}
extern "C" int aw_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int aw_create(int device, aw_ctx** out) {
    if (!out) return AW_EINVAL;
    *out = nullptr;
    int n = aw_device_count();
    if (n <= 0 || device < 0 || device >= n) {
        aw_set_error("no CUDA device %d (visible devices: %d); this library has no CPU fallback", device, n);
        return AW_ENODEVICE;
    }
    AW_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    AW_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        aw_set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return AW_ENODEVICE;
    }
    aw_ctx* c = new aw_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_sketch, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        aw_set_error("cudaStreamCreate: %s", cudaGetErrorString(e));
        delete c;
        return AW_ECUDA;
    }
    *out = c;
    return AW_OK;
}

static void free_sketches(aw_ctx* c) {
    c->stranded.sk.release();
    c->stranded.n.release();
    c->have_stranded = false;
    for (auto& kv : c->canonical) {
        kv.second->sk.release();
        kv.second->n.release();
        delete kv.second;
    }
    c->canonical.clear();
}

extern "C" void aw_destroy(aw_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();  // nothing of this context may still be running when its buffers are parked for reuse
    free_sketches(c);
    c->d_slots.release();
    c->d_ascii.release();
    c->d_packed.release();
    c->d_ids.release();
    c->d_id_off.release();
    for (auto& w : c->wsp) {
        w.ws_main.release();
        w.ws_hist_meta.release();
        w.ws_blk.release();
        w.ws_seq2.release();
        w.ws_runs.release();
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->up_stream) cudaStreamDestroy(c->up_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->ev_sketch) cudaEventDestroy(c->ev_sketch);
    delete c;
}

extern "C" void aw_trim_cache(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) n = 0;
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < n && d < 64; ++d) {
        cudaSetDevice(d);
        g_cache.trim_dev(d);
    }
    cudaSetDevice(cur);
    g_cache.trim_pin();
}

extern "C" int aw_set_option(aw_ctx* c, const char* key, int64_t value) {
    if (!c || !key) return AW_EINVAL;
    std::string k(key);
    if (k == "ctas_per_sm") c->ctas_per_sm = (int)value;
    else if (k == "threads_per_cta") {
#ifdef AW_NT_EXPERIMENT
        if (value != 0 && value != 32 && value != 128 && value != 256 && value != AW_NT_EXPERIMENT) return AW_EINVAL;
#else
        if (value != 0 && value != 32 && value != 128 && value != 256) return AW_EINVAL;
#endif
        c->threads_per_cta = (int)value;
    } else if (k == "max_wavefront_width") c->max_w = value;
    else if (k == "hist_mb") c->hist_mb = value;
    else if (k == "chunk_pairs") c->chunk_pairs = value > 0 ? value : 65536;
    else if (k == "band_engine") (void)value;  // accepted for compatibility: the experimental band engine of the first kernels is gone
    else if (k == "ws16") c->ws16 = value ? 1 : 0;
    else if (k == "cluster_min_len") c->cluster_min_len = value;
    else if (k == "cluster_always") c->cluster_always = value ? 1 : 0;
    else if (k == "solo_len") c->solo_len = std::max<int64_t>(0, value);
    else if (k == "max_retry_attempts") c->max_retry = (int)std::max<int64_t>(0, std::min<int64_t>(3, value));
    else return AW_EINVAL;
    return AW_OK;
}

extern "C" uint32_t aw_num_sequences(const aw_ctx* c) { return c ? c->n : 0; }

static int pen_from_params(const aw_params* p, AwPen* pen);
// AllPairIterator::with_orientation_params (src/iterator.rs:95-98)
extern "C" int aw_set_orientation_params(aw_ctx* c, const aw_params* p) {
    if (!c || !p) return AW_EINVAL;
    AwPen pen;
    int rc = pen_from_params(p, &pen);
    if (rc) return rc;
    c->orient_params = *p;
    return AW_OK;
}

extern "C" int aw_load_sequences(aw_ctx* c, uint32_t n, const uint8_t* const* seqs, const uint64_t* lens, const char* const* ids) {
    if (!c || (n && (!seqs || !lens))) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    AW_CUDA_CHECK(cudaStreamSynchronize(c->stream));  // nothing may still read the store that is about to be replaced
    AW_CUDA_CHECK(cudaStreamSynchronize(c->stream2));
    free_sketches(c);
    c->n = n;
    c->lens.assign(lens, lens + n);
    c->ids.resize(n);
    c->h_slots.assign((size_t)2 * n, AwSlot{0, 0, 0, 1});
    c->max_len = 0;
    // layout: every slot 16-byte aligned with 16 guard bytes / 4 guard words either side
    uint64_t a_off = 16, p_off = 4, raw_total = 0;
    std::vector<uint64_t> raw_off(n);
    for (uint32_t i = 0; i < n; ++i) {
        if (lens[i] > 0x07ffffffull) {
            aw_set_error("sequence %u is longer than 2^27-1 bases", i);
            return AW_EUNSUPPORTED;
        }
        raw_off[i] = raw_total;
        raw_total += lens[i];
        c->max_len = std::max<uint64_t>(c->max_len, lens[i]);
        for (int s = 0; s < 2; ++s) {
            AwSlot& sl = c->h_slots[2 * i + s];
            sl.ascii_off = a_off;
            sl.packed_off = p_off;
            sl.len = (uint32_t)lens[i];
            sl.clean = 1;
            a_off += ((lens[i] + 15) / 16) * 16 + 32;
            p_off += (lens[i] + 15) / 16 + 8;
        }
        c->ids[i] = ids && ids[i] ? ids[i] : "";
    }
    // ids
    std::vector<uint32_t> id_off(n + 1);
    std::string idcat;
    for (uint32_t i = 0; i < n; ++i) {
        id_off[i] = (uint32_t)idcat.size();
        idcat += c->ids[i];
    }
    id_off[n] = (uint32_t)idcat.size();
    int rc;
    if ((rc = c->d_slots.ensure(sizeof(AwSlot) * 2 * (size_t)std::max(1u, n)))) return rc;
    if ((rc = c->d_ascii.ensure(a_off + 16))) return rc;
    if ((rc = c->d_packed.ensure((p_off + 4) * 4))) return rc;
    if ((rc = c->d_ids.ensure(idcat.size() + 1))) return rc;
    if ((rc = c->d_id_off.ensure(4 * (size_t)(n + 1)))) return rc;
    AW_CUDA_CHECK(cudaMemsetAsync(c->d_ascii.p, 0, a_off + 16, c->stream));
    AW_CUDA_CHECK(cudaMemsetAsync(c->d_packed.p, 0, (p_off + 4) * 4, c->stream));
    if (n == 0) {
        AW_CUDA_CHECK(cudaStreamSynchronize(c->stream));
        return AW_OK;
    }
    // stage raw sequences through pinned memory
    PinBuf stage;
    DevBuf d_raw, d_raw_off;
    if ((rc = stage.ensure(raw_total + 16))) return rc;
    for (uint32_t i = 0; i < n; ++i) memcpy(stage.as<uint8_t>() + raw_off[i], seqs[i], lens[i]);
    if ((rc = d_raw.ensure(raw_total + 16)) || (rc = d_raw_off.ensure(8 * (size_t)n))) {
        stage.release();
        return rc;
    }
    cudaError_t e = cudaMemcpyAsync(d_raw.p, stage.p, raw_total, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_raw_off.p, raw_off.data(), 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_slots.p, c->h_slots.data(), sizeof(AwSlot) * 2 * (size_t)n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_ids.p, idcat.data(), idcat.size(), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_id_off.p, id_off.data(), 4 * (size_t)(n + 1), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        const uint64_t maxwords = (c->max_len + 15) / 16;
        dim3 grid((unsigned)std::max<uint64_t>(1, std::min<uint64_t>((maxwords + 127) / 128, 1024)), (unsigned)std::min<uint32_t>(n, 65535u));
        awk::aw_pack_kernel<<<grid, 128, 0, c->stream>>>(d_raw.as<uint8_t>(), d_raw_off.as<uint64_t>(), c->d_slots.as<AwSlot>(), n,
                                                         c->d_ascii.as<uint8_t>(), c->d_packed.as<uint32_t>());
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->h_slots.data(), c->d_slots.p, sizeof(AwSlot) * 2 * (size_t)n, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    stage.release();
    d_raw.release();
    d_raw_off.release();
    if (e != cudaSuccess) {
        aw_set_error("aw_load_sequences: %s", cudaGetErrorString(e));
        return AW_ECUDA;
    }
    c->all_clean = true;
    for (auto& s : c->h_slots) c->all_clean = c->all_clean && s.clean;
    return AW_OK;
}

// ---- sketches ------------------------------------------------------------------------------
static uint32_t next_pow2(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

static int build_sketches(aw_ctx* c, SketchSet& ss, bool canonical, int k, uint32_t size, cudaStream_t st) {
    const uint32_t count = canonical ? c->n : 2 * c->n;
    if (k < 1 || k > 31 || size == 0 || size > 4096) return AW_EINVAL;
    int rc;
    if ((rc = ss.sk.ensure(sizeof(uint64_t) * (size_t)std::max(1u, count) * size))) return rc;
    if ((rc = ss.n.ensure(sizeof(uint32_t) * (size_t)std::max(1u, count)))) return rc;
    ss.count = count;
    ss.size = size;
    if (count == 0) return AW_OK;
    const uint32_t cap = next_pow2(size);
    const size_t smem = sizeof(unsigned long long) * cap;
    if (canonical)
        awk::aw_sketch_kernel<true><<<count, awk::SK_NT, smem, st>>>(c->d_ascii.as<uint8_t>(), c->d_slots.as<AwSlot>(), 2, k, size, cap, ss.sk.as<uint64_t>(), ss.n.as<uint32_t>());
    else
        awk::aw_sketch_kernel<false><<<count, awk::SK_NT, smem, st>>>(c->d_ascii.as<uint8_t>(), c->d_slots.as<AwSlot>(), 1, k, size, cap, ss.sk.as<uint64_t>(), ss.n.as<uint32_t>());
    AW_CUDA_CHECK(cudaGetLastError());
    return AW_OK;
}

static int ensure_stranded(aw_ctx* c, cudaStream_t st, uint64_t* launches) {
    if (c->have_stranded) {
        // the sketches may have been built on another stream: order this one after the build
        AW_CUDA_CHECK(cudaStreamWaitEvent(st, c->ev_sketch, 0));
        return AW_OK;
    }
    int rc = build_sketches(c, c->stranded, false, AW_ORIENT_K, AW_SKETCH_SIZE, st);
    if (rc) return rc;
    AW_CUDA_CHECK(cudaEventRecord(c->ev_sketch, st));
    c->have_stranded = true;
    if (launches) ++*launches;
    return AW_OK;
}

static int ensure_canonical(aw_ctx* c, int k, uint32_t size, SketchSet** out) {
    auto key = std::make_pair(k, size);
    auto it = c->canonical.find(key);
    if (it != c->canonical.end()) {
        *out = it->second;
        return AW_OK;
    }
    SketchSet* ss = new SketchSet();
    int rc = build_sketches(c, *ss, true, k, size, c->stream);
    if (rc) {
        delete ss;
        return rc;
    }
    c->canonical[key] = ss;
    *out = ss;
    return AW_OK;
}

extern "C" int aw_get_sketch(aw_ctx* c, uint32_t idx, int reverse_complement, int canonical, int k, uint32_t sketch_size, uint64_t* out, uint32_t* out_n) {
    if (!c || !out || !out_n || idx >= c->n) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    SketchSet* ss = nullptr;
    uint32_t row;
    int rc;
    if (canonical) {
        if ((rc = ensure_canonical(c, k, sketch_size, &ss))) return rc;
        row = idx;
    } else {
        if (k != AW_ORIENT_K || sketch_size != AW_SKETCH_SIZE) return AW_EUNSUPPORTED;
        if ((rc = ensure_stranded(c, c->stream, nullptr))) return rc;
        ss = &c->stranded;
        row = 2 * idx + (reverse_complement ? 1 : 0);
    }
    AW_CUDA_CHECK(cudaMemcpyAsync(out_n, ss->n.as<uint32_t>() + row, 4, cudaMemcpyDeviceToHost, c->stream));
    AW_CUDA_CHECK(cudaMemcpyAsync(out, ss->sk.as<uint64_t>() + (size_t)row * ss->size, 8 * (size_t)ss->size, cudaMemcpyDeviceToHost, c->stream));
    AW_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return AW_OK;
}

extern "C" int aw_mash_jaccard_counts(aw_ctx* c, int k, uint32_t sketch_size, uint32_t* inter, uint32_t* uni) {
    if (!c || !inter || !uni) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    SketchSet* ss = nullptr;
    int rc = ensure_canonical(c, k, sketch_size, &ss);
    if (rc) return rc;
    const size_t nn = (size_t)c->n * c->n;
    if (nn == 0) return AW_OK;
    DevBuf di, du;
    if ((rc = di.ensure(4 * nn)) || (rc = du.ensure(4 * nn))) {
        di.release();
        return rc;
    }
    cudaError_t e = cudaMemsetAsync(di.p, 0, 4 * nn, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(du.p, 0, 4 * nn, c->stream);
    if (e == cudaSuccess) {
        awk::aw_jaccard_matrix_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(c->n, ss->sk.as<uint64_t>(), ss->n.as<uint32_t>(), ss->size, di.as<uint32_t>(), du.as<uint32_t>());
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(inter, di.p, 4 * nn, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(uni, du.p, 4 * nn, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    di.release();
    du.release();
    if (e != cudaSuccess) {
        aw_set_error("aw_mash_jaccard_counts: %s", cudaGetErrorString(e));
        return AW_ECUDA;
    }
    return AW_OK;
}

extern "C" int aw_orient_pairs(aw_ctx* c, const aw_pair* pairs, uint64_t npairs, uint8_t* out_is_reverse) {
    if (!c || (npairs && (!pairs || !out_is_reverse))) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    for (uint64_t i = 0; i < npairs; ++i)
        if (pairs[i].query_idx >= c->n || pairs[i].target_idx >= c->n) return AW_EINVAL;
    if (npairs == 0) return AW_OK;
    int rc = ensure_stranded(c, c->stream, nullptr);
    if (rc) return rc;
    DevBuf dp, dr;
    if ((rc = dp.ensure(sizeof(aw_pair) * npairs)) || (rc = dr.ensure(npairs))) {
        dp.release();
        return rc;
    }
    cudaError_t e = cudaMemcpyAsync(dp.p, pairs, sizeof(aw_pair) * npairs, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        awk::aw_orient_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(dp.as<aw_pair>(), npairs, c->stranded.sk.as<uint64_t>(), c->stranded.n.as<uint32_t>(), c->stranded.size, dr.as<uint8_t>());
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_is_reverse, dr.p, npairs, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    dp.release();
    dr.release();
    if (e != cudaSuccess) {
        aw_set_error("aw_orient_pairs: %s", cudaGetErrorString(e));
        return AW_ECUDA;
    }
    return AW_OK;
}

extern "C" int aw_estimate_divergence(aw_ctx* c, const aw_pair* pairs, uint64_t npairs, float* out) {
    if (!c || (npairs && (!pairs || !out))) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    for (uint64_t i = 0; i < npairs; ++i)
        if (pairs[i].query_idx >= c->n || pairs[i].target_idx >= c->n) return AW_EINVAL;
    if (npairs == 0) return AW_OK;
    int rc = ensure_stranded(c, c->stream, nullptr);
    if (rc) return rc;
    DevBuf dp, dd;
    if ((rc = dp.ensure(sizeof(aw_pair) * npairs)) || (rc = dd.ensure(4 * npairs))) return rc;
    cudaError_t e = cudaMemcpyAsync(dp.p, pairs, sizeof(aw_pair) * npairs, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        awk::aw_divergence_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(dp.as<aw_pair>(), npairs, c->stranded.sk.as<uint64_t>(), c->stranded.n.as<uint32_t>(),
                                                                   c->stranded.size, AW_ORIENT_K, dd.as<float>());
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dd.p, 4 * npairs, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        aw_set_error("aw_estimate_divergence: %s", cudaGetErrorString(e));
        return AW_ECUDA;
    }
    return AW_OK;
}

// ---- batches -------------------------------------------------------------------------------
// create_wfa_aligner + AlignmentMode::from_params (src/alignment.rs:263-289, src/types.rs:105-117)
static int pen_from_params(const aw_params* p, AwPen* pen) {
    memset(pen, 0, sizeof(*pen));
    if (p->match_score > 0) {
        aw_set_error("match_score must be negative or zero (WFA2: wavefront_penalties_set_*)");
        return AW_EUNSUPPORTED;
    }
    const bool two = p->has_gap2_open && p->has_gap2_extend;
    const bool edit = !two && p->gap_open == p->gap_extend && p->gap_open == p->mismatch_penalty;
    pen->x = p->mismatch_penalty;
    pen->o1 = edit ? p->mismatch_penalty : p->gap_open;
    pen->e1 = edit ? p->mismatch_penalty : p->gap_extend;
    pen->two_piece = two ? 1 : 0;
    if (two) {
        pen->o2 = p->gap2_open;
        pen->e2 = p->gap2_extend;
        if (pen->o2 < 0 || pen->e2 <= 0) return AW_EINVAL;
    }
    if (pen->x <= 0 || pen->o1 < 0 || pen->e1 <= 0) {
        aw_set_error("penalties must satisfy mismatch>0, gap_open>=0, gap_extend>0");
        return AW_EINVAL;
    }
    pen->sx = pen->x;
    pen->so1 = pen->o1;
    pen->se1 = pen->e1;
    pen->so2 = pen->o2;
    pen->se2 = pen->e2;
    pen->smatch = p->match_score;
    if (p->match_score < 0) {  // WFA2's penalty shifting (include/aw_wfa2_compat.h): the wavefronts run on x', o', e'
        const int m = p->match_score;
        pen->x = AW_SHIFT_MISMATCH(pen->x, m);
        pen->o1 = AW_SHIFT_GAP_OPEN(pen->o1, m);
        pen->e1 = AW_SHIFT_GAP_EXTEND(pen->e1, m);
        if (two) {
            pen->o2 = AW_SHIFT_GAP_OPEN(pen->o2, m);
            pen->e2 = AW_SHIFT_GAP_EXTEND(pen->e2, m);
        }
    }
    int sc = std::max(pen->x, pen->o1 + pen->e1);
    if (two) sc = std::max(sc, pen->o2 + pen->e2);
    pen->scope = sc + 1;
    if (pen->scope > 512) {
        aw_set_error("penalties too large (max_score_scope %d > 512)", pen->scope);
        return AW_EUNSUPPORTED;
    }
    return AW_OK;
}

extern "C" void aw_batch_destroy(aw_ctx* c, aw_batch* b) {
    if (!b) return;
    if (c) cudaSetDevice(c->device);
    if (b->launched) {  // never park buffers a kernel still uses (the buffers' destructors park them)
        if (b->ev_done) cudaEventSynchronize(b->ev_done);
        if (b->last_stream) cudaStreamSynchronize(b->last_stream);
    }
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->ev_done) cudaEventDestroy(b->ev_done);
    delete b;
}

// score-only results carry no CIGAR and no PAF text, and the cs:Z: tag is a PAF column
static int check_flags(uint32_t flags) {
    if ((flags & AW_FLAG_SCORE_ONLY) && (flags & (AW_FLAG_CIGAR_BYTES | AW_FLAG_PAF_BLOCKS))) {
        aw_set_error("AW_FLAG_SCORE_ONLY cannot be combined with AW_FLAG_CIGAR_BYTES or AW_FLAG_PAF_BLOCKS");
        return AW_EINVAL;
    }
    if ((flags & (AW_FLAG_CS | AW_FLAG_CS_LONG)) && (flags & (AW_FLAG_NO_PAF | AW_FLAG_SCORE_ONLY))) {
        aw_set_error("AW_FLAG_CS / AW_FLAG_CS_LONG cannot be combined with AW_FLAG_NO_PAF or AW_FLAG_SCORE_ONLY");
        return AW_EINVAL;
    }
    return AW_OK;
}

// the pair-order re-layout of the text arena: whole blocks for the block callback, and one contiguous line per pair with its
// cs column
static bool ordered_text(uint32_t flags) { return ((flags & AW_FLAG_PAF_BLOCKS) && !(flags & AW_FLAG_NO_PAF)) || (flags & AW_FLAG_CS); }

// (re)initialises a batch object for a new pair list; device / pinned buffers of an earlier use are kept (grow-only)
static int batch_init(aw_ctx* c, aw_batch* b, const aw_params* params, int orientation_mode, const aw_pair* pairs, uint64_t npairs, uint32_t flags) {
    int rc = pen_from_params(params, &b->pen);
    if (rc) return rc;
    if (orientation_mode == AW_ORIENT_WFA && (rc = pen_from_params(&c->orient_params, &b->pen_orient))) return rc;
    b->orient = orientation_mode;
    if (flags & AW_FLAG_SCORE_ONLY) flags |= AW_FLAG_NO_PAF;
    if (flags & AW_FLAG_CS_LONG) flags |= AW_FLAG_CS;
    b->flags = flags;
    b->kflags = (flags & ~(AW_FLAG_CS | AW_FLAG_CS_LONG)) | ((flags & AW_FLAG_CS) ? AW_FLAG_CIGAR_BYTES : 0u);
    b->npairs = npairs;
    b->launched = false;
    b->has_order = false;
    b->max_p = b->max_t = 0;
    b->h_pairs.assign(pairs, pairs + npairs);
    uint64_t sum_len = 0;
    bool varied = false;
    for (uint64_t i = 0; i < npairs; ++i) {
        if (pairs[i].query_idx >= c->n || pairs[i].target_idx >= c->n) {
            aw_set_error("pair %llu references a sequence index out of range", (unsigned long long)i);
            return AW_EINVAL;
        }
        const uint64_t pl = c->lens[pairs[i].query_idx], tl = c->lens[pairs[i].target_idx];
        b->max_p = std::max(b->max_p, pl);
        b->max_t = std::max(b->max_t, tl);
        sum_len += pl + tl;
        if (i && (pl + tl) != c->lens[pairs[0].query_idx] + c->lens[pairs[0].target_idx]) varied = true;
    }
    size_t idlen_max = 0;
    for (auto& s : c->ids) idlen_max = std::max(idlen_max, s.size());
    b->text_cap = (flags & AW_FLAG_SCORE_ONLY) ? 16
                  : (flags & AW_FLAG_NO_PAF)    ? sum_len / 2 + 64 * npairs + 1024
                                                : sum_len + (257 + 2 * idlen_max) * npairs + 1024;
    b->bytes_cap = (b->kflags & AW_FLAG_CIGAR_BYTES) ? sum_len + 16 : 16;
    b->tag_cap = (flags & AW_FLAG_CS) ? 2 * sum_len + 16 : 0;                   // a tag is at most 2 * (qlen + tlen) bytes (aw_cs.cuh)
    b->text2_cap = b->text_cap + ((flags & AW_FLAG_CS) ? 6 * npairs + b->tag_cap : 0);  // + "\tcs:Z:" and the tag per line
    const size_t np1 = (size_t)std::max<uint64_t>(1, npairs);
    if ((rc = b->d_pairs.ensure(sizeof(aw_pair) * np1)) || (rc = b->d_isrev.ensure(np1)) || (rc = b->d_out.ensure(sizeof(AwPairOut) * np1)) ||
        (rc = b->d_text.ensure(b->text_cap)) || (rc = b->d_bytes.ensure(b->bytes_cap)) || (rc = b->d_ctl.ensure(sizeof(BatchCtl))) ||
        (orientation_mode == AW_ORIENT_WFA &&
         ((rc = b->d_out_f.ensure(sizeof(AwPairOut) * np1)) || (rc = b->d_out_r.ensure(sizeof(AwPairOut) * np1)) || (rc = b->d_strand.ensure(2 * np1)))))
        return rc;
    if (ordered_text(flags) && ((rc = b->d_text2.ensure(b->text2_cap)) || (rc = b->d_off.ensure(8 * (np1 + 1))))) return rc;
    if ((flags & AW_FLAG_CS) && ((rc = b->d_tags.ensure(b->tag_cap)) || (rc = b->d_cs_out.ensure(sizeof(AwCsOut) * np1)))) return rc;
    // uploads go through their own stream, so that a batch can be prepared while the previous one is still running
    cudaStream_t us = c->up_stream;
    cudaError_t e = cudaMemcpyAsync(b->d_pairs.p, pairs, sizeof(aw_pair) * npairs, cudaMemcpyHostToDevice, us);
    if (e == cudaSuccess) e = cudaMemsetAsync(b->d_isrev.p, 0, np1, us);
    if (e == cudaSuccess && orientation_mode == AW_ORIENT_WFA) e = cudaMemsetAsync(b->d_strand.p, 0, np1, us);
    if (e == cudaSuccess && orientation_mode == AW_ORIENT_WFA) e = cudaMemsetAsync(b->d_strand.as<uint8_t>() + np1, 1, np1, us);
    // (one-warp kernels for reads up to 1 kb keep the given order: their costs are within a small factor of each other and the
    // sort + upload would cost more than it saves)
    if (e == cudaSuccess && varied && std::max(b->max_p, b->max_t) > 1024) {
        // heaviest pairs first: greedy balance of the persistent CTAs.  Predicted cost = wavefront cells ~ (expected score)^2
        // with the score estimated from length x divergence (mash distance of the stranded sketches) + length difference
        std::vector<uint32_t> order(npairs);
        std::vector<double> cost(npairs);
        std::vector<float> div;
        if (orientation_mode == AW_ORIENT_MASH) {  // the sketches are (or will be) there anyway: estimate every pair's divergence
            DevBuf dd;
            if ((rc = ensure_stranded(c, us, nullptr)) || (rc = dd.ensure(4 * np1))) return rc;
            div.resize(npairs);
            awk::aw_divergence_kernel<<<c->sm_count * 8, 256, 0, us>>>(b->d_pairs.as<aw_pair>(), npairs, c->stranded.sk.as<uint64_t>(),
                                                                c->stranded.n.as<uint32_t>(), c->stranded.size, AW_ORIENT_K, dd.as<float>());
            e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaMemcpyAsync(div.data(), dd.p, 4 * (size_t)npairs, cudaMemcpyDeviceToHost, us);
            if (e == cudaSuccess) e = cudaStreamSynchronize(us);
            if (e != cudaSuccess) {
                aw_set_error("aw_batch_create: %s", cudaGetErrorString(e));
                return AW_ECUDA;
            }
        }
        for (uint64_t i = 0; i < npairs; ++i) {
            order[i] = (uint32_t)i;
            const double pl = (double)c->lens[pairs[i].query_idx], tl = (double)c->lens[pairs[i].target_idx];
            const double d = div.empty() ? 0.05 : std::min(0.5, std::max(1e-3, (double)div[i]));
            const double sc = std::max(pl, tl) * d + std::fabs(pl - tl);
            cost[i] = sc * sc + pl + tl;
        }
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t bb) { return cost[a] > cost[bb]; });
        if ((rc = b->d_order.ensure(4 * np1))) return rc;
        e = cudaMemcpyAsync(b->d_order.p, order.data(), 4 * (size_t)npairs, cudaMemcpyHostToDevice, us);
        if (e == cudaSuccess) e = cudaStreamSynchronize(us);  // `order` dies with this scope
        b->has_order = true;
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(us);
    if (e != cudaSuccess) {
        aw_set_error("aw_batch_create: %s", cudaGetErrorString(e));
        return AW_ECUDA;
    }
    return AW_OK;
}

extern "C" int aw_batch_create(aw_ctx* c, const aw_params* params, int orientation_mode, const aw_pair* pairs, uint64_t npairs, uint32_t flags,
                               aw_batch** out) {
    if (!c || !params || !out || (npairs && !pairs)) return AW_EINVAL;
    *out = nullptr;
    if (npairs > 0xfffffff0ull) return AW_EINVAL;
    if (orientation_mode != AW_ORIENT_MASH && orientation_mode != AW_ORIENT_FORWARD && orientation_mode != AW_ORIENT_WFA) return AW_EINVAL;
    if (int rc = check_flags(flags)) return rc;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    aw_batch* b = new aw_batch();
    int rc = batch_init(c, b, params, orientation_mode, pairs, npairs, flags);
    if (rc) {
        aw_batch_destroy(c, b);
        return rc;
    }
    *out = b;
    return AW_OK;
}

namespace {

// Mb-scale pairs: CTAs per pair (thread-block cluster; 8 is the largest portable cluster size)
#ifndef AW_CLUSTER_SIZE
#define AW_CLUSTER_SIZE 8  // (16 needs the non-portable cluster size opt-in)
#endif
#ifndef AW_CLUSTER_NT
#define AW_CLUSTER_NT 512  // threads per CTA of the cluster kernels: 4 pairs of 1 Mb take 23.8 s with 512, 35.5 s with 256
#endif

struct LaunchCfg {
    int nt, grid;
    int cluster;  // CTAs per pair: 1, or the cluster size of the Mb-scale kernels (grid = clusters * cluster)
    int W;
    unsigned long long ws_ints, hist_ints, runs_cap;
    bool ws16;
    int hist_max_scores;
    int blk_cap;
    unsigned long long seq2_cap;
};

template <int NT, int BITS, bool TWO, class WS, int CL = 1, bool SCORE = false>
cudaError_t launch_align(const awk::KParams& P, int grid, size_t smem, cudaStream_t st) {
    auto kern = SCORE ? awk::aw_score_kernel<NT, BITS, TWO, WS, CL> : awk::aw_align_kernel<NT, BITS, TWO, WS, CL>;
    // static + dynamic shared memory together decide whether the opt-in is needed (the kernels carry up to 28 KB of static
    // shared memory); query the static part once per instantiation
    static size_t static_smem = ~(size_t)0;
    static int max_optin = 0;
    if (static_smem == ~(size_t)0) {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kern);
        if (e != cudaSuccess) return e;
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        static_smem = fa.sharedSizeBytes;
    }
    // int16 2-bit kernels read the staged sequences through a 32 KB address window (ld16s): the CTA must own all of it
    if (NT >= 64 && BITS == 2 && sizeof(WS) == 2 && static_smem + smem < awk::SEQ2_WINDOW) smem = awk::SEQ2_WINDOW - static_smem;
    if (const char* pad = getenv("AW_SMEM_PAD")) smem += (size_t)atoi(pad);  // tuning aid: what does a larger shared-memory footprint cost?
    if (static_smem + smem > (size_t)max_optin) return cudaErrorInvalidConfiguration;
    if (static_smem + smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    if (CL > 1) {  // one pair per thread-block cluster
        if (CL > 8) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return e;
        }
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3((unsigned)grid);
        lc.blockDim = dim3(NT);
        lc.dynamicSmemBytes = smem;
        lc.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = CL;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        lc.attrs = at;
        lc.numAttrs = 1;
        // the CTAs are persistent: launching more clusters than can be resident at once buys nothing
        int max_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&max_clusters, kern, &lc) == cudaSuccess && max_clusters > 0 && grid / CL > max_clusters)
            lc.gridDim = dim3((unsigned)(max_clusters * CL));
        else
            cudaGetLastError();
        return cudaLaunchKernelEx(&lc, kern, P);
    }
    kern<<<grid, NT, smem, st>>>(P);
    return cudaGetLastError();
}

cudaError_t dispatch_align(const awk::KParams& P, int nt, int bits, bool two, bool ws16, int grid, cudaStream_t st, int cluster = 1) {
    const int scope = P.pen.scope;
    // SlotMeta rings: forward + reverse, plus one per warp for the warp-parallel leaves of the chunked kernels (aw_wfa.cuh RM_N)
    const int rm_n = (AW_LEAFPAR && nt >= 64 && bits == 2 && cluster == 1) ? 2 + nt / 32 : 2;
    size_t smem = sizeof(awk::SlotMeta) * rm_n * (scope + 1) + sizeof(int) * 10 * scope + sizeof(unsigned long long) * nt + sizeof(int) * (10 * scope + 4);
    // AW_FLAG_SCORE_ONLY: the score-only twin of every kernel (the orientation passes clear the flag: they need X+I+D)
    const bool score = (P.flags & AW_FLAG_SCORE_ONLY) != 0;
    if (cluster == AW_CLUSTER_SIZE && nt == AW_CLUSTER_NT && bits == 2 && !ws16) {
        if (two)
            return score ? launch_align<AW_CLUSTER_NT, 2, true, int, AW_CLUSTER_SIZE, true>(P, grid, smem, st)
                         : launch_align<AW_CLUSTER_NT, 2, true, int, AW_CLUSTER_SIZE>(P, grid, smem, st);
#ifndef AW_FAST_BUILD
        return score ? launch_align<AW_CLUSTER_NT, 2, false, int, AW_CLUSTER_SIZE, true>(P, grid, smem, st)
                     : launch_align<AW_CLUSTER_NT, 2, false, int, AW_CLUSTER_SIZE>(P, grid, smem, st);
#endif
    }
    if (cluster != 1) return cudaErrorInvalidConfiguration;
#define AW_CASE(NT_, BITS_, TWO_, WS_, W16_)                         \
    if (nt == NT_ && bits == BITS_ && two == TWO_ && ws16 == W16_) \
        return score ? launch_align<NT_, BITS_, TWO_, WS_, 1, true>(P, grid, smem, st) : launch_align<NT_, BITS_, TWO_, WS_>(P, grid, smem, st);
#ifndef AW_FAST_BUILD  // dev builds (-DAW_FAST_BUILD) keep only the two-piece 2-bit int16 kernels
    AW_CASE(32, 2, true, int, false)
    AW_CASE(32, 2, false, int, false)
    AW_CASE(32, 8, true, int, false)
    AW_CASE(32, 8, false, int, false)
    AW_CASE(256, 2, true, int, false)
    AW_CASE(256, 2, false, int, false)
    AW_CASE(256, 8, true, int, false)
    AW_CASE(256, 8, false, int, false)
    AW_CASE(256, 2, false, short, true)
    AW_CASE(256, 8, true, short, true)
    AW_CASE(256, 8, false, short, true)
    AW_CASE(128, 2, false, short, true)
    AW_CASE(128, 2, false, int, false)
#endif
    AW_CASE(256, 2, true, short, true)
    AW_CASE(128, 2, true, short, true)
#ifdef AW_NT_EXPERIMENT  // tuning builds: another CTA size for the int16 two-piece kernel (set_option threads_per_cta)
    AW_CASE(AW_NT_EXPERIMENT, 2, true, short, true)
#endif
    AW_CASE(128, 2, true, int, false)
#undef AW_CASE
    return cudaErrorInvalidValue;
}

// sizes the per-CTA workspace for one launch; attempt 0 is the fast first try, later attempts
// remove the wavefront-width cap and grow the history arena (retry ladder)
int plan_launch(aw_ctx* c, const AwPen& pen, uint64_t npairs, uint64_t max_p, uint64_t max_t, int attempt, LaunchCfg* cfg, int slot = 0) {
    aw_ctx::Workspace& w = c->wsp[slot];
    cudaStream_t kst = slot ? c->stream2 : c->stream;
    const int ncomp = pen.two_piece ? 5 : 3;
    const uint64_t maxlen = std::max(max_p, max_t);
    // int16 storage: every offset (incl. out-of-bounds I/D drift, <= 2*tlen+plen) must stay below 32000
    // ... and a (drifted) null must stay separable from every real antidiagonal: 3 * (plen + tlen) < 63000 (aw_wfa.cuh, wf_cells_v)
    const bool fits16 = c->ws16 && (2 * max_t + max_p < 32000) && (2 * max_p + max_t < 32000) && (3 * (max_p + max_t) < 63000);
    // pairs up to 1 kb: one warp per pair; 2-bit pairs up to 50 kb: 128 threads (2 warps per direction, 4 CTAs per SM
    // measured best on C2); everything else: 256 threads
    // (20 kb pairs, int32 rows: 571 pairs/s with 128 threads vs 501 with 256); Mb-scale pairs keep 256 threads per pair
    int nt = c->threads_per_cta ? c->threads_per_cta : (maxlen <= 1024 ? 32 : ((c->all_clean && (fits16 || maxlen <= 50000)) ? 128 : 256));
    // Mb-scale pairs: one pair per cluster of AW_CLUSTER_SIZE 256-thread CTAs (few pairs in flight, each on 2048 threads)
    // ... when the batch is small: a cluster finishes one pair ~3x sooner than a single CTA but moves ~2.5x fewer cells per SM,
    // so with enough pairs to occupy every CTA slot the one-CTA-per-pair kernel is the faster regime (profiles/README.md)
    const uint64_t cluster_slots = std::max<uint64_t>(1, (uint64_t)c->sm_count * AW_CTAS_PER_SM(AW_CLUSTER_NT) / AW_CLUSTER_SIZE);
    const bool use_cluster = c->cluster_min_len > 0 && c->all_clean && !fits16 && (int64_t)maxlen >= c->cluster_min_len && !c->threads_per_cta &&
                             (npairs <= 2 * cluster_slots || c->cluster_always);
    if (use_cluster) nt = AW_CLUSTER_NT;
    int per_sm = c->ctas_per_sm ? c->ctas_per_sm : (nt == 32 ? 16 : AW_CTAS_PER_SM(nt));
    uint64_t full_w = (max_p + max_t + 3 + 16 + 15) & ~15ull;  // rows are 16-element aligned (vectorised int16 loop)
    uint64_t W = full_w;
    uint64_t hist_ints = (uint64_t)c->hist_mb * (1u << 20) / 4;
    if (nt == 32 && attempt == 0) hist_ints = std::min<uint64_t>(hist_ints, 1u << 18);
    for (int a = 0; a < attempt; ++a) hist_ints *= 8;
    int hist_max_scores = attempt == 0 ? (nt == 32 ? 1024 : 4096) : (attempt == 1 ? 32768 : 262144);
    uint64_t runs_cap = max_p + max_t + 4;
    if (nt == 128 && !c->all_clean) nt = 256;  // the 128-thread kernels exist for the chunked 2-bit path only
    // the warp-parallel leaves split the second half of the run buffer into nt / 32 parts, so a leaf gets 1 / (nt / 32) of
    // the pair's runs: a divergent pair whose leaf needs more fails its first try, and the retry rungs give every part room
    // for the whole pair
    if (attempt > 0 && !use_cluster) runs_cap *= nt / 32;
    const bool ws16 = fits16 && nt >= 64;
    const uint64_t epi = ws16 ? 2 : 1;  // elements per int
    // + the all-NULL row and the compact I/D rings of the int16 path (aw_wfa.cuh: null_base, cmp_base)
    const uint64_t cmp_rows = 2ull * (2 * (pen.e1 + 1) + (pen.two_piece ? 2 * (pen.e2 + 1) : 0));
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return AW_ECUDA;
    size_t parked = 0;
    {
        std::lock_guard<std::mutex> g(g_cache.mu);
        parked = g_cache.parked_dev[c->device >= 0 && c->device < 64 ? c->device : 0];
    }
    const uint64_t budget = (uint64_t)((double)(free_b + parked + w.bytes()) * 0.85);
    // workspace slots = pairs in flight: one per CTA, or one per cluster
    const uint64_t want_grid = std::min<uint64_t>(use_cluster ? std::max<uint64_t>(1, (uint64_t)c->sm_count * per_sm / AW_CLUSTER_SIZE) : (uint64_t)c->sm_count * per_sm,
                                                  std::max<uint64_t>(1, npairs));
    if (attempt == 0) {
        // first try: as many diagonals per wavefront as let every resident CTA have its own workspace (a wavefront
        // is at most 2*score+1 wide, far below plen+tlen for similar sequences); pairs that need more report
        // AW_EWORKSPACE and are re-run with the full width on fewer CTAs
        const uint64_t rows = 2ull * (pen.scope + 1) * ncomp + 1 + cmp_rows;
        const uint64_t fixed = hist_ints * 4 + (uint64_t)hist_max_scores * awk::HIST_META_INTS * 4 + runs_cap * 8 + (full_w / 16 + 8) * 16;
        const uint64_t share = budget / want_grid;
        uint64_t w_fit = share > fixed ? (share - fixed) / (rows * (ws16 ? 2 : 4)) : 0;
        w_fit = std::max<uint64_t>(w_fit & ~15ull, std::min<uint64_t>(full_w, 65536));
        W = std::min(W, w_fit);
        if (W > (uint64_t)c->max_w) W = std::max<uint64_t>(32, (uint64_t)c->max_w & ~15ull);
    }
    uint64_t ring_ints = ((2ull * (pen.scope + 1) * ncomp + 1 + cmp_rows) * W + epi - 1) / epi;
    if (ring_ints >= 0x7f000000ull) {
        aw_set_error("wavefront ring of %llu ints per CTA exceeds the 32-bit workspace index", (unsigned long long)ring_ints);
        return AW_EUNSUPPORTED;
    }
    hist_ints = std::min<uint64_t>(hist_ints, 0x7ff00000ull - ring_ints);
    hist_ints &= ~7ull;
    ring_ints = (ring_ints + 7) & ~7ull;
    uint64_t ws_ints = ring_ints + hist_ints;
    uint64_t per_cta = ws_ints * 4 + (uint64_t)hist_max_scores * awk::HIST_META_INTS * 4 + runs_cap * 8 + (full_w / 16 + 8) * 16;
    uint64_t grid = want_grid;
    while (grid > 1 && grid * per_cta > budget) grid = grid / 2;
    if (grid * per_cta > budget) {
        aw_set_error("device workspace for one pair (%llu MB) does not fit in free memory", (unsigned long long)(per_cta >> 20));
        return AW_ENOMEM;
    }
    cfg->nt = nt;
    cfg->cluster = use_cluster ? AW_CLUSTER_SIZE : 1;
    cfg->grid = (int)grid * cfg->cluster;
    cfg->W = (int)std::min<uint64_t>(W, 0x7ffffff0ull);
    cfg->ws_ints = ws_ints;
    cfg->hist_ints = hist_ints * epi;  // capacity in workspace elements
    cfg->ws16 = ws16;
    cfg->runs_cap = runs_cap;
    cfg->hist_max_scores = hist_max_scores;
    cfg->blk_cap = (int)(W / (awk::VBLOCK_CHUNKS * 4) + 2);  // blocks of >= 30 x 4 diagonals
    // pairs too long for the shared-memory staging keep their 4 word-pair arrays (pattern, text, both reversed) per CTA
    cfg->seq2_cap = (!ws16 && nt >= 64 && c->all_clean) ? 2 * ((max_p / 16 + 2) + (max_t / 16 + 2)) : 0;
    // growing a workspace re-allocates it: a kernel of an earlier batch that is still running must not lose its buffers
    const std::pair<DevBuf*, uint64_t> need[] = {
        {&w.ws_main, grid * ws_ints * 4},
        {&w.ws_blk, grid * 2ull * (pen.scope + 1) * (uint64_t)cfg->blk_cap * 2 * 4},
        {&w.ws_seq2, grid * cfg->seq2_cap * 8 + 16},
        {&w.ws_hist_meta, grid * (uint64_t)hist_max_scores * awk::HIST_META_INTS * 4},
        {&w.ws_runs, grid * runs_cap * 8},
    };
    for (const auto& n : need)
        if (n.second > n.first->cap) {
            if (cudaStreamSynchronize(kst) != cudaSuccess) return AW_ECUDA;
            break;
        }
    for (const auto& n : need)
        if (int rc = n.first->ensure(n.second)) return rc;
    return AW_OK;
}

// launches one alignment pass of batch b on the workspace set of the batch: the pairs order[0 .. npairs) (0 .. npairs
// without an order) with the strands is_reverse, results into out, PAF text and CIGAR bytes into the two arenas
cudaError_t launch_pass(aw_ctx* c, aw_batch* b, const AwPen& pen, const LaunchCfg& cfg, uint32_t flags, const uint8_t* is_reverse,
                        const uint32_t* order, uint64_t npairs, AwPairOut* out, char* text, uint64_t text_cap, uint8_t* bytes, uint64_t bytes_cap,
                        unsigned long long* text_cursor, unsigned long long* bytes_cursor, unsigned long long* next_pair, cudaStream_t st) {
    awk::KParams P;
    memset(&P, 0, sizeof(P));
    P.slots = c->d_slots.as<AwSlot>();
    P.packed = c->d_packed.as<uint32_t>();
    P.ascii = c->d_ascii.as<uint8_t>();
    P.ids = c->d_ids.as<char>();
    P.id_off = c->d_id_off.as<uint32_t>();
    P.pairs = b->d_pairs.as<aw_pair>();
    P.is_reverse = is_reverse;
    P.order = order;
    P.npairs = (uint32_t)npairs;
    P.next_pair = reinterpret_cast<unsigned int*>(next_pair);
    P.pen = pen;
    P.flags = flags;
    const aw_ctx::Workspace& w = c->wsp[b->slot];
    P.ws = w.ws_main.as<int>();
    P.ws_ints_per_cta = cfg.ws_ints;
    P.W = cfg.W;
    P.hist_ints = (int)std::min<unsigned long long>(cfg.hist_ints, 0x7fffffffull);
    P.ws_hist_meta = w.ws_hist_meta.as<int>();
    P.ws_blk = w.ws_blk.as<int>();
    P.blk_cap = cfg.blk_cap;
    P.ws_seq2 = w.ws_seq2.as<uint2>();
    P.seq2_cap = cfg.seq2_cap;
    P.hist_max_scores = cfg.hist_max_scores;
    P.ws_runs = w.ws_runs.as<uint32_t>();
    P.runs_cap = cfg.runs_cap;
    P.out = out;
    P.text = text;
    P.text_cursor = text_cursor;
    P.text_cap = text_cap;
    P.bytes = bytes;
    P.bytes_cursor = bytes_cursor;
    P.bytes_cap = bytes_cap;
    P.solo_len = (int)std::min<int64_t>(c->solo_len, 0x7fffffff);
    return dispatch_align(P, cfg.nt, c->all_clean ? 2 : 8, pen.two_piece != 0, cfg.ws16, cfg.grid, st, cfg.cluster);
}

// determine_orientation_wfa's two alignments: the pairs order[0 .. npairs) with the orientation penalties, forward and
// reverse-complemented query, counts only (flags without AW_FLAG_SCORE_ONLY: the pick needs X+I+D), into d_out_f / d_out_r
cudaError_t launch_orientation(aw_ctx* c, aw_batch* b, const LaunchCfg& cfo, const uint32_t* order, uint64_t npairs, BatchCtl* ctl, cudaStream_t st) {
    const size_t np1 = (size_t)std::max<uint64_t>(1, b->npairs);
    for (int s = 0; s < 2; ++s) {
        cudaError_t e = launch_pass(c, b, b->pen_orient, cfo, AW_KFLAG_COUNT_ONLY | AW_FLAG_NO_PAF, b->d_strand.as<uint8_t>() + s * np1, order, npairs,
                                    (s == 0 ? b->d_out_f : b->d_out_r).as<AwPairOut>(), b->d_text.as<char>(), b->text_cap, b->d_bytes.as<uint8_t>(),
                                    b->bytes_cap, &ctl->orient_text_cursor, &ctl->orient_bytes_cursor, &ctl->orient_next_pair[s], st);
        if (e != cudaSuccess) return e;
        ++b->stats[0];
    }
    return cudaSuccess;
}

// the cs:Z: tags of the pairs order[0 .. npairs) (0 .. npairs without an order) of an alignment pass: results `out`, CIGAR op
// bytes `ops`; tags into the arena `tags` at the cursor, their places into cs_out
cudaError_t launch_cs(aw_ctx* c, aw_batch* b, const AwPairOut* out, const uint32_t* order, uint64_t npairs, const uint8_t* ops, char* tags,
                      unsigned long long* tag_cursor, AwCsOut* cs_out, cudaStream_t st) {
    const unsigned grid = (unsigned)std::min<uint64_t>(npairs, 1u << 20);
    const int long_form = (b->flags & AW_FLAG_CS_LONG) ? 1 : 0;
    if (b->max_p + b->max_t <= awk::CS_SHORT_LEN)
        awk::aw_cs_kernel<awk::CS_NT_SHORT><<<grid, awk::CS_NT_SHORT, 0, st>>>(out, order, (uint32_t)npairs, b->d_pairs.as<aw_pair>(), c->d_slots.as<AwSlot>(),
                                                                             c->d_ascii.as<uint8_t>(), ops, long_form, tags, tag_cursor, cs_out);
    else
        awk::aw_cs_kernel<awk::CS_NT><<<grid, awk::CS_NT, 0, st>>>(out, order, (uint32_t)npairs, b->d_pairs.as<aw_pair>(), c->d_slots.as<AwSlot>(),
                                                                 c->d_ascii.as<uint8_t>(), ops, long_form, tags, tag_cursor, cs_out);
    return cudaGetLastError();
}

}  // namespace

extern "C" int aw_batch_launch(aw_ctx* c, aw_batch* b, void* stream) {
    if (!c || !b) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : (b->slot ? c->stream2 : c->stream);
    b->last_stream = st;
    memset(b->stats, 0, sizeof(b->stats));
    memset(b->cyc, 0, sizeof(b->cyc));
    b->r_out.clear();
    b->r_cs_len.clear();
    b->r_idx.clear();
    b->r_text.clear();
    b->r_bytes.clear();
    b->launched = true;
    if (b->npairs == 0) return AW_OK;
    int rc;
    if (b->orient == AW_ORIENT_MASH) {
        if ((rc = ensure_stranded(c, st, &b->stats[0]))) return rc;
        awk::aw_orient_kernel<<<c->sm_count * 8, 256, 0, st>>>(b->d_pairs.as<aw_pair>(), b->npairs, c->stranded.sk.as<uint64_t>(), c->stranded.n.as<uint32_t>(),
                                                               c->stranded.size, b->d_isrev.as<uint8_t>());
        AW_CUDA_CHECK(cudaGetLastError());
        ++b->stats[0];
    }
    LaunchCfg cfg;
    if ((rc = plan_launch(c, b->pen, b->npairs, b->max_p, b->max_t, 0, &cfg, b->slot))) return rc;
    AW_CUDA_CHECK(cudaMemsetAsync(b->d_ctl.p, 0, sizeof(BatchCtl), st));
    BatchCtl* ctl = b->d_ctl.as<BatchCtl>();
    const uint32_t* order = b->has_order ? b->d_order.as<uint32_t>() : nullptr;
    if (b->orient == AW_ORIENT_WFA) {
        // determine_orientation_wfa: two full alignments with the orientation penalties, forward and
        // reverse-complemented query, statistics only; then pick the strand with fewer X+I+D columns
        LaunchCfg cfo;
        if ((rc = plan_launch(c, b->pen_orient, b->npairs, b->max_p, b->max_t, 0, &cfo, b->slot))) return rc;  // never larger than the main plan
        cudaError_t eo = launch_orientation(c, b, cfo, order, b->npairs, ctl, st);
        if (eo != cudaSuccess) {
            aw_set_error("orientation kernel launch: %s", cudaGetErrorString(eo));
            return AW_ECUDA;
        }
        awk::aw_wfa_orient_pick_kernel<<<c->sm_count * 4, 256, 0, st>>>(b->d_out_f.as<AwPairOut>(), b->d_out_r.as<AwPairOut>(), b->npairs, b->d_isrev.as<uint8_t>());
        AW_CUDA_CHECK(cudaGetLastError());
        ++b->stats[0];
    }
    if (!b->ev0) {
        AW_CUDA_CHECK(cudaEventCreate(&b->ev0));
        AW_CUDA_CHECK(cudaEventCreate(&b->ev1));
        AW_CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_done, cudaEventDisableTiming));
    }
    AW_CUDA_CHECK(cudaEventRecord(b->ev0, st));
    cudaError_t e = launch_pass(c, b, b->pen, cfg, b->kflags, b->d_isrev.as<uint8_t>(), order, b->npairs, b->d_out.as<AwPairOut>(), b->d_text.as<char>(),
                                b->text_cap, b->d_bytes.as<uint8_t>(), b->bytes_cap, &ctl->text_cursor, &ctl->bytes_cursor, &ctl->next_pair, st);
    if (e != cudaSuccess) {
        aw_set_error("align kernel launch (nt=%d grid=%d): %s", cfg.nt, cfg.grid, cudaGetErrorString(e));
        return AW_ECUDA;
    }
    AW_CUDA_CHECK(cudaEventRecord(b->ev1, st));
    const bool cs = (b->flags & AW_FLAG_CS) != 0;
    if (cs) {
        AW_CUDA_CHECK(launch_cs(c, b, b->d_out.as<AwPairOut>(), nullptr, b->npairs, b->d_bytes.as<uint8_t>(), b->d_tags.as<char>(), &ctl->tag_cursor,
                                b->d_cs_out.as<AwCsOut>(), st));
        ++b->stats[0];
    }
    if (ordered_text(b->flags)) {
        const AwCsOut* cs_out = cs ? b->d_cs_out.as<AwCsOut>() : nullptr;
        const unsigned nl = (b->flags & AW_FLAG_PAF_BLOCKS) ? 1u : 0u;
        awk::aw_text_scan_kernel<<<1, 1024, 0, st>>>(b->d_out.as<AwPairOut>(), cs_out, nl, (uint32_t)b->npairs, b->d_off.as<unsigned long long>());
        awk::aw_text_gather_kernel<<<c->sm_count * 8, 256, 0, st>>>(b->d_out.as<AwPairOut>(), b->d_off.as<unsigned long long>(), (uint32_t)b->npairs,
                                                                  b->d_text.as<char>(), cs_out, b->d_tags.as<char>(), nl, b->d_text2.as<char>());
        AW_CUDA_CHECK(cudaGetLastError());
        b->stats[0] += 2;
    }
    AW_CUDA_CHECK(cudaEventRecord(b->ev_done, st));
    ++b->stats[0];
    return AW_OK;
}

// One rung of a retry ladder: re-runs the pairs `todo` of batch b with the workspace plan_launch gives their longest query
// and target at `attempt`.  launch(cfg, order, ctl, stream) queues the rung's passes over the uploaded work list `order`
// with the zeroed control block `ctl` and returns an AW_ status.  The rung then waits for them and copies each result array
// of `outs` back (all npairs entries), and the control block into *h_ctl when that is given.
template <class Launch>
static int retry_rung(aw_ctx* c, aw_batch* b, const AwPen& pen, const std::vector<uint32_t>& todo, int attempt, const char* what, Launch launch,
                      std::initializer_list<std::pair<const DevBuf*, std::vector<AwPairOut>*>> outs, BatchCtl* h_ctl = nullptr) {
    cudaStream_t kst = b->slot ? c->stream2 : c->stream;
    uint64_t max_p = 0, max_t = 0;
    for (uint32_t i : todo) {
        max_p = std::max(max_p, c->lens[b->h_pairs[i].query_idx]);
        max_t = std::max(max_t, c->lens[b->h_pairs[i].target_idx]);
    }
    LaunchCfg cfg;
    int rc = plan_launch(c, pen, todo.size(), max_p, max_t, attempt, &cfg, b->slot);
    if (rc) return rc;
    DevBuf d_order, d_ctl;
    if ((rc = d_order.ensure(4 * todo.size())) || (rc = d_ctl.ensure(sizeof(BatchCtl)))) return rc;
    cudaError_t e = cudaMemcpy(d_order.p, todo.data(), 4 * todo.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_ctl.p, 0, sizeof(BatchCtl));
    if (e == cudaSuccess) {
        if ((rc = launch(cfg, d_order.as<uint32_t>(), d_ctl.as<BatchCtl>(), kst))) return rc;
        e = cudaStreamSynchronize(kst);
    }
    for (const auto& o : outs) {
        o.second->resize(b->npairs);
        if (e == cudaSuccess) e = cudaMemcpy(o.second->data(), o.first->p, sizeof(AwPairOut) * b->npairs, cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess && h_ctl) e = cudaMemcpy(h_ctl, d_ctl.p, sizeof(BatchCtl), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        aw_set_error("%s: %s", what, cudaGetErrorString(e));
        return AW_ECUDA;
    }
    return AW_OK;
}

// --wfa-orientation, pairs whose first-try orientation passes ran out of workspace (strand 2 = undecided): both count-only
// passes go through the same ladder as the alignment itself, then the strand is picked like determine_orientation_wfa
// (src/alignment.rs:157-175: a pass that still fails after the ladder counts as usize::MAX)
static int retry_orientation(aw_ctx* c, aw_batch* b, const AwPairOut* h_out) {
    std::vector<uint32_t> todo;
    for (uint64_t i = 0; i < b->npairs; ++i)
        if (h_out[i].status == AW_EWORKSPACE && h_out[i].is_reverse > 1) todo.push_back((uint32_t)i);
    if (todo.empty()) return AW_OK;
    std::vector<AwPairOut> of, orv;
    std::vector<uint8_t> strand(b->npairs, 0);
    std::vector<uint8_t> have_f(b->npairs, 0), have_r(b->npairs, 0);
    std::vector<unsigned long long> ed_f(b->npairs, ~0ull), ed_r(b->npairs, ~0ull);
    // at least one rung, also with max_retry_attempts = 0 (where retry_failed runs none)
    for (int attempt = 1; attempt <= std::max(1, c->max_retry) && !todo.empty(); ++attempt) {
        auto launch = [&](const LaunchCfg& cfo, const uint32_t* order, BatchCtl* ctl, cudaStream_t kst) -> int {
            const cudaError_t e = launch_orientation(c, b, cfo, order, todo.size(), ctl, kst);
            if (e != cudaSuccess) aw_set_error("orientation retry: %s", cudaGetErrorString(e));
            return e == cudaSuccess ? AW_OK : AW_ECUDA;
        };
        if (int rc = retry_rung(c, b, b->pen_orient, todo, attempt, "orientation retry", launch, {{&b->d_out_f, &of}, {&b->d_out_r, &orv}})) return rc;
        std::vector<uint32_t> still;
        const bool last = attempt >= std::max(1, c->max_retry);
        for (uint32_t i : todo) {
            if (!have_f[i] && (of[i].status != AW_EWORKSPACE || last)) {
                have_f[i] = 1;
                ed_f[i] = of[i].status == AW_OK ? of[i].n_x + of[i].n_i + of[i].n_d : ~0ull;
            }
            if (!have_r[i] && (orv[i].status != AW_EWORKSPACE || last)) {
                have_r[i] = 1;
                ed_r[i] = orv[i].status == AW_OK ? orv[i].n_x + orv[i].n_i + orv[i].n_d : ~0ull;
            }
            if (have_f[i] && have_r[i]) strand[i] = ed_f[i] <= ed_r[i] ? 0 : 1;
            else still.push_back(i);
        }
        todo.swap(still);
    }
    // publish the decided strands (everything else in d_isrev is untouched)
    for (uint64_t i = 0; i < b->npairs; ++i)
        if (h_out[i].status == AW_EWORKSPACE && h_out[i].is_reverse > 1) {
            cudaError_t e = cudaMemcpy(b->d_isrev.as<uint8_t>() + i, &strand[i], 1, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) {
                aw_set_error("orientation retry: %s", cudaGetErrorString(e));
                return AW_ECUDA;
            }
        }
    return AW_OK;
}

// re-runs the pairs that reported AW_EWORKSPACE with a larger workspace (synchronous, rare)
static int retry_failed(aw_ctx* c, aw_batch* b, const AwPairOut* h_out) {
    std::vector<uint32_t> failed;
    for (uint64_t i = 0; i < b->npairs; ++i)
        if (h_out[i].status == AW_EWORKSPACE) failed.push_back((uint32_t)i);
    if (failed.empty()) return AW_OK;
    b->stats[1] = failed.size();
    // a later batch may already be queued on this batch's kernel stream with the current workspace: let it finish before the
    // workspace is re-planned (and possibly re-allocated) for the retry
    AW_CUDA_CHECK(cudaStreamSynchronize(b->slot ? c->stream2 : c->stream));
    if (b->orient == AW_ORIENT_WFA) {
        int rc = retry_orientation(c, b, h_out);
        if (rc) return rc;
    }
    const unsigned nl = (b->flags & AW_FLAG_PAF_BLOCKS) ? 1u : 0u;
    const bool cs = (b->flags & AW_FLAG_CS) != 0;
    for (int attempt = 1; attempt <= 3 && !failed.empty(); ++attempt) {
        const bool give_up = attempt > c->max_retry;  // ladder disabled or exhausted: report the pairs as failed
        if (give_up) {
            for (uint32_t i : failed) {
                AwPairOut o = h_out[i];
                o.status = AW_EALIGN;
                b->r_idx.push_back(i);
                b->r_out.push_back(o);
                b->r_cs_len.push_back(0);
            }
            failed.clear();
            break;
        }
        uint64_t sum_len = 0;
        size_t idlen_max = 0;
        for (uint32_t i : failed) {
            sum_len += c->lens[b->h_pairs[i].query_idx] + c->lens[b->h_pairs[i].target_idx];
            idlen_max = std::max(idlen_max, c->ids[b->h_pairs[i].query_idx].size() + c->ids[b->h_pairs[i].target_idx].size());
        }
        const uint64_t text_cap = 12 * sum_len + (256 + idlen_max) * failed.size() + 1024;
        const uint64_t bytes_cap = (b->kflags & AW_FLAG_CIGAR_BYTES) ? sum_len + 16 : 16;
        const uint64_t tag_cap = cs ? 2 * sum_len + 16 : 0;
        DevBuf d_out, d_text, d_bytes, d_tags, d_cs_out;
        auto launch = [&](const LaunchCfg& cfg, const uint32_t* order, BatchCtl* ctl, cudaStream_t kst) -> int {
            int rc;
            if ((rc = d_out.ensure(sizeof(AwPairOut) * b->npairs)) || (rc = d_text.ensure(text_cap)) || (rc = d_bytes.ensure(bytes_cap))) return rc;
            if (cs && ((rc = d_tags.ensure(tag_cap)) || (rc = d_cs_out.ensure(sizeof(AwCsOut) * b->npairs)))) return rc;
            cudaError_t e = launch_pass(c, b, b->pen, cfg, b->kflags, b->d_isrev.as<uint8_t>(), order, failed.size(), d_out.as<AwPairOut>(),
                                        d_text.as<char>(), text_cap, d_bytes.as<uint8_t>(), bytes_cap, &ctl->text_cursor, &ctl->bytes_cursor,
                                        &ctl->next_pair, kst);
            ++b->stats[0];
            if (e == cudaSuccess && cs) {
                e = launch_cs(c, b, d_out.as<AwPairOut>(), order, failed.size(), d_bytes.as<uint8_t>(), d_tags.as<char>(), &ctl->tag_cursor,
                              d_cs_out.as<AwCsOut>(), kst);
                ++b->stats[0];
            }
            if (e != cudaSuccess) aw_set_error("retry launch: %s", cudaGetErrorString(e));
            return e == cudaSuccess ? AW_OK : AW_ECUDA;
        };
        std::vector<AwPairOut> outs;
        BatchCtl ctl;
        if (int rc = retry_rung(c, b, b->pen, failed, attempt, "retry launch", launch, {{&d_out, &outs}}, &ctl)) return rc;
        std::vector<char> text(std::min<uint64_t>(ctl.text_cursor, text_cap));
        std::vector<uint8_t> bytes((b->flags & AW_FLAG_CIGAR_BYTES) ? std::min<uint64_t>(ctl.bytes_cursor, bytes_cap) : 0);
        std::vector<char> tags(cs ? std::min<uint64_t>(ctl.tag_cursor, tag_cap) : 0);
        std::vector<AwCsOut> cs_out(cs ? b->npairs : 0);
        if (!text.empty()) AW_CUDA_CHECK(cudaMemcpy(text.data(), d_text.p, text.size(), cudaMemcpyDeviceToHost));
        if (!bytes.empty()) AW_CUDA_CHECK(cudaMemcpy(bytes.data(), d_bytes.p, bytes.size(), cudaMemcpyDeviceToHost));
        if (!tags.empty()) AW_CUDA_CHECK(cudaMemcpy(tags.data(), d_tags.p, tags.size(), cudaMemcpyDeviceToHost));
        if (cs) AW_CUDA_CHECK(cudaMemcpy(cs_out.data(), d_cs_out.p, sizeof(AwCsOut) * b->npairs, cudaMemcpyDeviceToHost));
        std::vector<uint32_t> still;
        for (uint32_t i : failed) {
            AwPairOut o = outs[i];
            if (o.status == AW_EWORKSPACE && attempt < 3) {
                still.push_back(i);
                continue;
            }
            uint64_t cs_len = 0;
            if (o.status == AW_OK) {
                const uint64_t toff = b->r_text.size(), boff = b->r_bytes.size();
                // the line, then the cs column, then the newline of block mode
                b->r_text.insert(b->r_text.end(), text.begin() + o.paf_off, text.begin() + o.paf_off + o.paf_len);
                if (cs) {
                    static const char col[] = "\tcs:Z:";
                    cs_len = cs_out[i].len;
                    b->r_text.insert(b->r_text.end(), col, col + 6);
                    b->r_text.insert(b->r_text.end(), tags.begin() + cs_out[i].off, tags.begin() + cs_out[i].off + cs_len);
                }
                if (o.paf_len && nl) b->r_text.push_back('\n');
                const uint64_t nb = (b->flags & AW_FLAG_CIGAR_BYTES) ? o.n_m + o.n_x + o.n_i + o.n_d : 0;
                if (nb) b->r_bytes.insert(b->r_bytes.end(), bytes.begin() + o.bytes_off, bytes.begin() + o.bytes_off + nb);
                o.paf_off = toff;
                o.bytes_off = boff;
            }
            b->r_idx.push_back(i);
            b->r_out.push_back(o);
            b->r_cs_len.push_back(cs_len);
        }
        failed.swap(still);
    }
    return AW_OK;
}

// adds a pair's work counters to the batch's stats: CIGAR runs and alignment columns (a score-only result has no op counts),
// computed cells and wavefront steps, and with `cycles` the device-clock breakdown
static void count_pair(aw_batch* b, const AwPairOut& o, bool cycles) {
    if (!(b->flags & AW_FLAG_SCORE_ONLY)) {
        b->stats[3] += o.nruns;
        b->stats[4] += std::max(o.n_m + o.n_x + o.n_d, o.n_m + o.n_x + o.n_i);
    }
    b->stats[6] += o.cells;
    b->stats[7] += o.steps;
    if (cycles)
        for (int q = 0; q < 6; ++q) b->cyc[q] += o.cyc[q];
}

// joins the batch's launch (an event, not a device-wide sync: another batch of the same context may be running), copies the
// results back on the context's copy stream and delivers them
static int fetch_impl(aw_ctx* c, aw_batch* b, aw_result_cb cb, aw_paf_block_cb block_cb, void* user) {
    if (b->npairs == 0) return AW_OK;
    AW_CUDA_CHECK(cudaEventSynchronize(b->ev_done));
    cudaStream_t cs = c->copy_stream;
    const bool with_cs = (b->flags & AW_FLAG_CS) != 0;
    int rc;
    // pinned: the results, the control block, and with AW_FLAG_CS the ordered arena's size and every pair's tag place
    if ((rc = b->h_out.ensure(sizeof(AwPairOut) * b->npairs + sizeof(BatchCtl) + 8 + (with_cs ? sizeof(AwCsOut) * b->npairs : 0)))) return rc;
    BatchCtl* h_ctl = reinterpret_cast<BatchCtl*>(b->h_out.as<char>() + sizeof(AwPairOut) * b->npairs);
    unsigned long long* h_ordered_len = reinterpret_cast<unsigned long long*>(h_ctl + 1);
    const AwCsOut* h_cs = reinterpret_cast<const AwCsOut*>(h_ordered_len + 1);
    AW_CUDA_CHECK(cudaMemcpyAsync(h_ctl, b->d_ctl.p, sizeof(BatchCtl), cudaMemcpyDeviceToHost, cs));
    AW_CUDA_CHECK(cudaMemcpyAsync(b->h_out.p, b->d_out.p, sizeof(AwPairOut) * b->npairs, cudaMemcpyDeviceToHost, cs));
    if (with_cs) {
        AW_CUDA_CHECK(cudaMemcpyAsync(h_ordered_len, b->d_off.as<unsigned long long>() + b->npairs, 8, cudaMemcpyDeviceToHost, cs));
        AW_CUDA_CHECK(cudaMemcpyAsync((void*)h_cs, b->d_cs_out.p, sizeof(AwCsOut) * b->npairs, cudaMemcpyDeviceToHost, cs));
    }
    AW_CUDA_CHECK(cudaStreamSynchronize(cs));
    const uint64_t text_used = with_cs ? std::min<uint64_t>(*h_ordered_len, b->text2_cap) : std::min<uint64_t>(h_ctl->text_cursor, b->text_cap);
    const uint64_t bytes_used = std::min<uint64_t>(h_ctl->bytes_cursor, b->bytes_cap);
    if ((rc = b->h_text.ensure(text_used + 1)) || (rc = b->h_bytes.ensure(bytes_used + 1))) return rc;
    // block mode and AW_FLAG_CS: the arena was re-laid out in pair order on the device (every line followed by '\n' in block
    // mode, and by its cs column with AW_FLAG_CS)
    const bool ordered = ordered_text(b->flags);
    if (text_used) AW_CUDA_CHECK(cudaMemcpyAsync(b->h_text.p, ordered ? b->d_text2.p : b->d_text.p, text_used, cudaMemcpyDeviceToHost, cs));
    if (bytes_used && (b->flags & AW_FLAG_CIGAR_BYTES)) AW_CUDA_CHECK(cudaMemcpyAsync(b->h_bytes.p, b->d_bytes.p, bytes_used, cudaMemcpyDeviceToHost, cs));
    AW_CUDA_CHECK(cudaStreamSynchronize(cs));
    const AwPairOut* outs = b->h_out.as<AwPairOut>();
    if ((rc = retry_failed(c, b, outs))) return rc;
    std::vector<int64_t> retry_of(b->r_idx.empty() ? 0 : b->npairs, -1);
    for (size_t j = 0; j < b->r_idx.size(); ++j) retry_of[b->r_idx[j]] = (int64_t)j;
    b->stats[2] = text_used + b->r_text.size();
    const bool blocks = block_cb && (b->flags & AW_FLAG_PAF_BLOCKS) && !(b->flags & AW_FLAG_NO_PAF);
    const unsigned nl = (b->flags & AW_FLAG_PAF_BLOCKS) ? 1u : 0u;
    const bool all_first_try = b->r_idx.empty();
    // the whole arena is one gap-free block of newline-terminated lines when every pair succeeded at the first try
    if (blocks && all_first_try && text_used && block_cb(b->h_text.as<char>(), text_used, b->npairs, user) != 0) return AW_ECALLBACK;
    std::string sentinel;
    if (blocks && all_first_try && !cb) {  // nothing per pair is wanted: only the counters
        for (uint64_t i = 0; i < b->npairs; ++i) count_pair(b, outs[i], false);
        return AW_OK;
    }
    uint64_t ordered_off = 0;  // running offset of pair i's line in the ordered arena
    static const char cs_col[] = "\tcs:Z:";
    for (uint64_t i = 0; i < b->npairs; ++i) {
        const AwPairOut* o = &outs[i];
        const char* text = b->h_text.as<char>();
        const uint8_t* bytes = b->h_bytes.as<uint8_t>();
        uint64_t paf_off = o->paf_off;
        uint64_t cs_len = with_cs ? h_cs[i].len : 0;
        if (ordered) {
            paf_off = ordered_off;
            if (o->status == AW_OK && o->paf_len) ordered_off += o->paf_len + nl + (with_cs ? 6 + cs_len : 0);
        }
        if (!retry_of.empty() && retry_of[i] >= 0) {
            o = &b->r_out[retry_of[i]];
            text = b->r_text.data();
            bytes = b->r_bytes.data();
            paf_off = o->paf_off;
            cs_len = with_cs ? b->r_cs_len[retry_of[i]] : 0;
        }
        aw_result r;
        memset(&r, 0, sizeof(r));
        r.query_idx = b->h_pairs[i].query_idx;
        r.target_idx = b->h_pairs[i].target_idx;
        r.is_reverse = (uint8_t)(o->is_reverse == 1);
        if (o->status == AW_OK && (b->flags & AW_FLAG_SCORE_ONLY)) {
            // End2End covers both sequences; there are no op counts, CIGAR or text to derive anything else from
            r.status = AW_OK;
            r.score = o->score;
            r.query_end = c->lens[r.query_idx];
            r.target_end = c->lens[r.target_idx];
            count_pair(b, *o, true);
        } else if (o->status == AW_OK) {
            r.status = AW_OK;
            r.score = o->score;
            r.query_end = o->n_m + o->n_x + o->n_d;
            r.target_end = o->n_m + o->n_x + o->n_i;
            r.num_matches = o->n_m;
            r.alignment_length = o->n_m + o->n_x;
            r.paf = (b->flags & AW_FLAG_NO_PAF) ? nullptr : text + paf_off;
            r.paf_len = (b->flags & AW_FLAG_NO_PAF) ? 0 : o->paf_len + (with_cs ? 6 + cs_len : 0);
            r.cg = text + paf_off + o->cg_off;
            r.cg_len = o->paf_len - o->cg_off;
            if (with_cs) {
                r.cs = text + paf_off + o->paf_len + 6;
                r.cs_len = cs_len;
            }
            if (b->flags & AW_FLAG_CIGAR_BYTES) {
                r.cigar_bytes = bytes + o->bytes_off;
                r.cigar_len = o->n_m + o->n_x + o->n_i + o->n_d;
            }
            count_pair(b, *o, true);
            if (blocks && !all_first_try && block_cb(r.paf, r.paf_len + nl, 1, user) != 0) return AW_ECALLBACK;
        } else {
            // the reference's failure sentinel (src/alignment.rs:49-64) still becomes a PAF line
            r.status = AW_EALIGN;
            r.score = INT32_MAX;
            ++b->stats[5];
            if (!(b->flags & AW_FLAG_NO_PAF)) {
                char buf[128];
                sentinel = c->ids[r.query_idx];
                snprintf(buf, sizeof(buf), "\t%llu\t0\t0\t%c\t", (unsigned long long)c->lens[r.query_idx], r.is_reverse ? '-' : '+');
                sentinel += buf;
                sentinel += c->ids[r.target_idx];
                snprintf(buf, sizeof(buf), "\t%llu\t0\t0\t0\t0\t60\tgi:f:0.000000\tcg:Z:", (unsigned long long)c->lens[r.target_idx]);
                sentinel += buf;
                const size_t cg_end = sentinel.size();
                if (with_cs) sentinel += cs_col;
                if (nl) sentinel += '\n';
                r.paf = sentinel.data();
                r.paf_len = sentinel.size() - nl;
                r.cg = r.paf + cg_end;
                if (with_cs) r.cs = r.paf + r.paf_len;
                if (blocks && block_cb(r.paf, r.paf_len + nl, 1, user) != 0) return AW_ECALLBACK;
            }
        }
        if (cb && cb(&r, user) != 0) return AW_ECALLBACK;
    }
    return AW_OK;
}

extern "C" int aw_batch_fetch(aw_ctx* c, aw_batch* b, aw_result_cb cb, void* user) {
    if (!c || !b || !b->launched) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    return fetch_impl(c, b, cb, nullptr, user);
}

extern "C" int aw_batch_kernel_ms(aw_ctx* c, aw_batch* b, float* out_ms) {
    if (!c || !b || !out_ms || !b->ev0) return AW_EINVAL;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    AW_CUDA_CHECK(cudaEventSynchronize(b->ev1));
    AW_CUDA_CHECK(cudaEventElapsedTime(out_ms, b->ev0, b->ev1));
    return AW_OK;
}

extern "C" int aw_batch_debug_cycles(aw_ctx* c, aw_batch* b, uint64_t out[6]) {
    if (!c || !b || !out) return AW_EINVAL;
    memcpy(out, b->cyc, sizeof(b->cyc));
    return AW_OK;
}

extern "C" int aw_batch_stats(aw_ctx* c, aw_batch* b, uint64_t out[8]) {
    if (!c || !b || !out) return AW_EINVAL;
    memcpy(out, b->stats, sizeof(b->stats));
    return AW_OK;
}

// The streaming driver: two batch objects alternate.  While batch k's kernel runs on c->stream, batch k+1's pair list is
// uploaded (up_stream) and its kernels are queued behind it; batch k is then joined by its event, copied back on copy_stream
// and delivered while batch k+1 computes.  Nothing here synchronises the device.
extern "C" int aw_align_stream(aw_ctx* c, const aw_params* params, int orientation_mode, uint32_t flags, aw_chunk_source next, void* next_user,
                               aw_result_cb cb, aw_paf_block_cb block_cb, void* user) {
    if (!c || !params || !next) return AW_EINVAL;
    if (orientation_mode != AW_ORIENT_MASH && orientation_mode != AW_ORIENT_FORWARD && orientation_mode != AW_ORIENT_WFA) return AW_EINVAL;
    if (int rc = check_flags(flags)) return rc;
    AW_CUDA_CHECK(cudaSetDevice(c->device));
    aw_batch* slot[2] = {new aw_batch(), new aw_batch()};
    bool busy[2] = {false, false};
    int rc = AW_OK;
    // second workspace set + kernel stream for the odd batches, unless one set already takes a large share of the device
    // (Mb-scale pairs): then both batches share set 0 and simply queue behind each other
    bool two_sets = true;
    auto feed = [&](int s) -> int {  // pulls the next chunk into slot s and queues its kernels; busy[s] says whether there was one
        const aw_pair* pairs = nullptr;
        const uint64_t n = next(next_user, &pairs);
        if (n == 0) return AW_OK;
        if (!pairs || n > 0xfffffff0ull) return AW_EINVAL;
        int r = batch_init(c, slot[s], params, orientation_mode, pairs, n, flags);
        slot[s]->slot = (two_sets && s == 1) ? 1 : 0;
        if (r == AW_OK) r = aw_batch_launch(c, slot[s], nullptr);
        if (s == 0 && two_sets) {
            size_t free_b = 0, total_b = 0;
            if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || c->wsp[0].bytes() > total_b / 5) two_sets = false;
        }
        busy[s] = (r == AW_OK);
        return r;
    };
    rc = feed(0);
    for (int k = 0; rc == AW_OK && busy[k & 1]; ++k) {
        rc = feed((k + 1) & 1);
        if (rc != AW_OK) break;
        rc = fetch_impl(c, slot[k & 1], cb, block_cb, user);
        busy[k & 1] = false;
    }
    for (int s = 0; s < 2; ++s) aw_batch_destroy(c, slot[s]);  // waits for a batch that is still in flight (cancelled run)
    return rc;
}

namespace {
struct ArraySource {
    const aw_pair* pairs;
    uint64_t n, pos, chunk;
    static uint64_t next(void* user, const aw_pair** out) {
        ArraySource* a = static_cast<ArraySource*>(user);
        if (a->pos >= a->n) return 0;
        const uint64_t cnt = std::min<uint64_t>(a->chunk, a->n - a->pos);
        *out = a->pairs + a->pos;
        a->pos += cnt;
        return cnt;
    }
};
}  // namespace

extern "C" int aw_align_pairs(aw_ctx* c, const aw_params* params, int orientation_mode, const aw_pair* pairs, uint64_t npairs, uint32_t flags,
                              aw_result_cb cb, void* user) {
    if (!c || !params || (npairs && !pairs)) return AW_EINVAL;
    if (int rc = check_flags(flags)) return rc;
    if (npairs == 0) {  // still validates the parameters like a real call
        AwPen pen;
        return pen_from_params(params, &pen);
    }
    ArraySource src{pairs, npairs, 0, (uint64_t)c->chunk_pairs};
    return aw_align_stream(c, params, orientation_mode, flags & ~AW_FLAG_PAF_BLOCKS, &ArraySource::next, &src, cb, nullptr, user);
}

// ---- lib_wfa2::AffineWavefronts-shaped API -------------------------------------------------
static int aligner_new(aw_ctx* parent, const aw_params& p, int memory_mode, aw_aligner** out) {
    if (!parent || !out) return AW_EINVAL;
    *out = nullptr;
    AwPen pen;
    int rc = pen_from_params(&p, &pen);
    if (rc) return rc;
    aw_aligner* a = new aw_aligner();
    rc = aw_create(parent->device, &a->ctx);
    if (rc) {
        delete a;
        return rc;
    }
    a->params = p;
    a->memory_mode = memory_mode;
    *out = a;
    return AW_OK;
}
extern "C" int aw_aligner_new_affine(aw_ctx* ctx, int32_t match_, int32_t mismatch, int32_t gap_opening, int32_t gap_extension, int memory_mode,
                                     aw_aligner** out) {
    aw_params p;
    memset(&p, 0, sizeof(p));
    p.match_score = match_;
    p.mismatch_penalty = mismatch;
    p.gap_open = gap_opening;
    p.gap_extend = gap_extension;
    // with_penalties_and_memory_mode always builds a gap-affine aligner: keep o,e distinct from the
    // "edit" shortcut only in name -- the constructor is numerically identical (SURVEY fact 6)
    return aligner_new(ctx, p, memory_mode, out);
}
extern "C" int aw_aligner_new_affine2p(aw_ctx* ctx, int32_t match_, int32_t mismatch, int32_t gap_opening1, int32_t gap_extension1,
                                       int32_t gap_opening2, int32_t gap_extension2, int memory_mode, aw_aligner** out) {
    aw_params p;
    memset(&p, 0, sizeof(p));
    p.match_score = match_;
    p.mismatch_penalty = mismatch;
    p.gap_open = gap_opening1;
    p.gap_extend = gap_extension1;
    p.gap2_open = gap_opening2;
    p.gap2_extend = gap_extension2;
    p.has_gap2_open = p.has_gap2_extend = 1;
    return aligner_new(ctx, p, memory_mode, out);
}
extern "C" int aw_aligner_set_alignment_scope(aw_aligner* a, int scope) {
    if (!a) return AW_EINVAL;
    if (scope != AW_SCOPE_ALIGNMENT && scope != AW_SCOPE_SCORE) return AW_EUNSUPPORTED;
    a->scope = scope;
    return AW_OK;
}
extern "C" int aw_aligner_set_alignment_span(aw_aligner* a, int span) { return !a ? AW_EINVAL : (span == AW_SPAN_END2END ? AW_OK : AW_EUNSUPPORTED); }
extern "C" int aw_aligner_set_heuristic(aw_aligner* a, int h) { return !a ? AW_EINVAL : (h == AW_HEURISTIC_NONE ? AW_OK : AW_EUNSUPPORTED); }
extern "C" int aw_aligner_get_memory_mode(const aw_aligner* a) { return a ? a->memory_mode : AW_EINVAL; }

static int aligner_cb(const aw_result* r, void* user) {
    aw_aligner* a = (aw_aligner*)user;
    a->score = r->score;
    a->cigar.assign(r->cigar_bytes, r->cigar_bytes + r->cigar_len);
    return r->status == AW_OK ? 0 : 1;
}
extern "C" int aw_aligner_align(aw_aligner* a, const uint8_t* pattern, int32_t plen, const uint8_t* text, int32_t tlen) {
    if (!a || plen < 0 || tlen < 0 || (plen && !pattern) || (tlen && !text)) return AW_ALIGN_UNDEFINED;
    const uint8_t* seqs[2] = {pattern, text};
    const uint64_t lens[2] = {(uint64_t)plen, (uint64_t)tlen};
    const char* ids[2] = {"pattern", "text"};
    a->cigar.clear();
    a->score = INT32_MAX;
    if (aw_load_sequences(a->ctx, 2, seqs, lens, ids) != AW_OK) return AW_ALIGN_OOM;
    aw_pair pr = {0, 1};
    const uint32_t flags = a->scope == AW_SCOPE_SCORE ? AW_FLAG_SCORE_ONLY : AW_FLAG_CIGAR_BYTES | AW_FLAG_NO_PAF;
    int rc = aw_align_pairs(a->ctx, &a->params, AW_ORIENT_FORWARD, &pr, 1, flags, aligner_cb, a);
    if (rc == AW_OK) return AW_ALIGN_COMPLETED;
    return rc == AW_ENOMEM ? AW_ALIGN_OOM : AW_ALIGN_UNDEFINED;
}
extern "C" int32_t aw_aligner_score(const aw_aligner* a) { return a ? a->score : INT32_MAX; }
extern "C" const uint8_t* aw_aligner_cigar(const aw_aligner* a, uint64_t* len) {
    if (!a) return nullptr;
    if (len) *len = a->cigar.size();
    return a->cigar.data();
}
extern "C" void aw_aligner_delete(aw_aligner* a) {
    if (!a) return;
    aw_destroy(a->ctx);
    delete a;
}
