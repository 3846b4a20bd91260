// aw_sketch.cuh -- K1 (pack + reverse complement), K2 (SipHash-1-3 k-mer hashing + bottom-s
// selection), K3 (sketch Jaccard -> orientation bit / all-pairs counts).
// Restates /root/reference/src/alignment.rs:69-154,178-190 and src/mash.rs:40-135 on the GPU.
#pragma once
#include "aw_common.cuh"

namespace awk {

// ---- K1 ------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t rc_byte(uint8_t b) {  // reverse_complement, src/alignment.rs:181-188
    switch (b) {
        case 'A': case 'a': return 'T';
        case 'T': case 't': return 'A';
        case 'C': case 'c': return 'G';
        case 'G': case 'g': return 'C';
        default: return 'N';
    }
}
__device__ __forceinline__ int code2(uint8_t b, bool& clean) {
    switch (b) {
        case 'A': return 0;
        case 'C': return 1;
        case 'G': return 2;
        case 'T': return 3;
        default: clean = false; return 0;
    }
}

// one thread = one packed word (16 bases) of the forward slot and of the reverse-complement slot
__global__ void aw_pack_kernel(const uint8_t* __restrict__ raw, const uint64_t* __restrict__ raw_off, AwSlot* slots, uint32_t n,
                               uint8_t* ascii, uint32_t* packed) {
    for (uint32_t i = blockIdx.y; i < n; i += gridDim.y) {
        const AwSlot f = slots[2 * i], r = slots[2 * i + 1];
        const uint32_t len = f.len, nwords = (len + 15) / 16;
        const uint8_t* src = raw + raw_off[i];
        bool clean_f = true, clean_r = true;
        for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x) {
            uint32_t wf = 0, wr = 0;
            for (int j = 0; j < 16; ++j) {
                const uint32_t pos = 16 * w + j;
                if (pos >= len) break;
                const uint8_t b = src[pos];
                ascii[f.ascii_off + pos] = b;
                wf |= (uint32_t)code2(b, clean_f) << (2 * j);
                const uint8_t c = rc_byte(src[len - 1 - pos]);
                ascii[r.ascii_off + pos] = c;
                wr |= (uint32_t)code2(c, clean_r) << (2 * j);
            }
            packed[f.packed_off + w] = wf;
            packed[r.packed_off + w] = wr;
        }
        if (!clean_f) slots[2 * i].clean = 0;
        if (!clean_r) slots[2 * i + 1].clean = 0;
    }
}

// ---- K2 ------------------------------------------------------------------------------------
#define AW_SIPROUND(v0, v1, v2, v3)                \
    do {                                           \
        v0 += v1; v1 = (v1 << 13) | (v1 >> 51); v1 ^= v0; v0 = (v0 << 32) | (v0 >> 32); \
        v2 += v3; v3 = (v3 << 16) | (v3 >> 48); v3 ^= v2;                              \
        v0 += v3; v3 = (v3 << 21) | (v3 >> 43); v3 ^= v0;                              \
        v2 += v1; v1 = (v1 << 17) | (v1 >> 47); v1 ^= v2; v2 = (v2 << 32) | (v2 >> 32); \
    } while (0)

// Rust DefaultHasher over <[u8] as Hash>: SipHash-1-3, zero keys, stream = len(u64 LE) || bytes
// (SURVEY Appendix B).  `kmer` holds the k bytes (k <= 32).
__device__ __forceinline__ uint64_t hash_kmer_bytes(const uint8_t* kmer, int k) {
    uint64_t v0 = 0x736f6d6570736575ULL, v1 = 0x646f72616e646f6dULL, v2 = 0x6c7967656e657261ULL, v3 = 0x7465646279746573ULL;
    uint64_t m = (uint64_t)k;  // length prefix word
    v3 ^= m;
    AW_SIPROUND(v0, v1, v2, v3);
    v0 ^= m;
    int i = 0;
    for (; i + 8 <= k; i += 8) {
        m = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) m |= (uint64_t)kmer[i + j] << (8 * j);
        v3 ^= m;
        AW_SIPROUND(v0, v1, v2, v3);
        v0 ^= m;
    }
    uint64_t b = (uint64_t)((k + 8) & 0xff) << 56;
    for (int j = 0; i + j < k; ++j) b |= (uint64_t)kmer[i + j] << (8 * j);
    v3 ^= b;
    AW_SIPROUND(v0, v1, v2, v3);
    v0 ^= b;
    v2 ^= 0xff;
    AW_SIPROUND(v0, v1, v2, v3);
    AW_SIPROUND(v0, v1, v2, v3);
    AW_SIPROUND(v0, v1, v2, v3);
    return v0 ^ v1 ^ v2 ^ v3;
}

__device__ __forceinline__ bool is_dna(uint8_t b) {
    b &= 0xDF;  // to upper for letters
    return b == 'A' || b == 'C' || b == 'G' || b == 'T';
}

// hash of the k-mer starting at seq[i]; returns false when the k-mer holds a non-ACGT byte.
// CANON: min(H(kmer), H(reverse_complement_kmer(kmer))) as src/mash.rs:95-101
template <bool CANON>
__device__ __forceinline__ bool kmer_hash_at(const uint8_t* __restrict__ seq, uint32_t i, int k, uint64_t& h) {
    uint8_t buf[32];
    bool ok = true;
    for (int j = 0; j < k; ++j) {
        const uint8_t b = seq[i + j];
        buf[j] = b;
        ok = ok && is_dna(b);
    }
    if (!ok) return false;
    h = hash_kmer_bytes(buf, k);
    if (CANON) {
        uint8_t rc[32];
        for (int j = 0; j < k; ++j) {
            const uint8_t u = buf[k - 1 - j] & 0xDF;
            rc[j] = u == 'A' ? 'T' : u == 'T' ? 'A' : u == 'C' ? 'G' : 'C';
        }
        const uint64_t hr = hash_kmer_bytes(rc, k);
        h = hr < h ? hr : h;
    }
    return true;
}

constexpr int SK_NT = 256;
constexpr int SK_BITS = 11;
constexpr int SK_BINS = 1 << SK_BITS;

// One CTA per sketch.  Exact bottom-`sketch_size` with duplicates (sort_unstable + truncate,
// src/alignment.rs:118-121): MSB-first radix select finds the value of rank sketch_size, then
// the strictly smaller hashes are gathered, sorted in shared memory, and padded with copies
// of the rank value.
template <bool CANON>
__global__ void __launch_bounds__(SK_NT) aw_sketch_kernel(const uint8_t* __restrict__ ascii, const AwSlot* __restrict__ slots, uint32_t slot_stride,
                                                          int k, uint32_t sketch_size, uint32_t sort_cap, uint64_t* __restrict__ out, uint32_t* __restrict__ out_n) {
    extern __shared__ unsigned long long sk_smem[];  // [sort_cap]
    __shared__ unsigned hist[SK_BINS];
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned s_need, s_total, s_cnt;
    const int tid = threadIdx.x;
    const uint32_t sk = blockIdx.x;
    const AwSlot sl = slots[(size_t)sk * slot_stride];
    const uint8_t* seq = ascii + sl.ascii_off;
    const uint32_t len = sl.len;
    uint64_t* dst = out + (size_t)sk * sketch_size;
    if (len < (uint32_t)k) {
        if (tid == 0) out_n[sk] = 0;
        return;
    }
    const uint32_t nk = len - (uint32_t)k + 1;
    if (tid == 0) {
        s_prefix = 0;
        s_need = sketch_size;
    }
    int prefix_bits = 0;
    bool take_all = false;
    while (prefix_bits < 64) {
        const int bits = min(SK_BITS, 64 - prefix_bits);
        for (int b = tid; b < SK_BINS; b += SK_NT) hist[b] = 0;
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        for (uint32_t i = tid; i < nk; i += SK_NT) {
            uint64_t h;
            if (!kmer_hash_at<CANON>(seq, i, k, h)) continue;
            if (prefix_bits == 0 || (h >> (64 - prefix_bits)) == prefix) atomicAdd(&hist[(h >> (64 - prefix_bits - bits)) & ((1u << bits) - 1)], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned need = s_need, cum = 0;
            int d = 0;
            const int nb = 1 << bits;
            for (; d < nb; ++d) {
                if (cum + hist[d] >= need) break;
                cum += hist[d];
            }
            if (d == nb) {  // fewer than sketch_size valid k-mers (only possible in the first pass)
                s_total = cum;
                s_need = 0;
            } else {
                s_need = need - cum;
                s_prefix = (prefix << bits) | (unsigned long long)d;
                s_total = 0xffffffffu;
            }
        }
        __syncthreads();
        if (s_need == 0) {
            take_all = true;
            break;
        }
        prefix_bits += bits;
    }
    const unsigned long long tstar = s_prefix;
    const unsigned n_eq = take_all ? 0 : s_need;                          // copies of the rank value
    const unsigned n_lt = take_all ? s_total : sketch_size - s_need;      // strictly smaller hashes
    if (tid == 0) s_cnt = 0;
    for (uint32_t i = tid; i < sort_cap; i += SK_NT) sk_smem[i] = ~0ull;
    __syncthreads();
    for (uint32_t i = tid; i < nk; i += SK_NT) {
        uint64_t h;
        if (!kmer_hash_at<CANON>(seq, i, k, h)) continue;
        if (take_all || h < tstar) {
            const unsigned idx = atomicAdd(&s_cnt, 1u);
            if (idx < sort_cap) sk_smem[idx] = h;
        }
    }
    __syncthreads();
    // bitonic sort of sort_cap (power of two) entries
    for (uint32_t size = 2; size <= sort_cap; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t i = tid; i < sort_cap / 2; i += SK_NT) {
                const uint32_t lo = (i / stride) * (stride * 2) + (i % stride);
                const uint32_t hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long a = sk_smem[lo], b = sk_smem[hi];
                if ((a > b) == up) {
                    sk_smem[lo] = b;
                    sk_smem[hi] = a;
                }
            }
            __syncthreads();
        }
    }
    for (uint32_t i = tid; i < n_lt; i += SK_NT) dst[i] = sk_smem[i];
    for (uint32_t i = tid; i < n_eq; i += SK_NT) dst[n_lt + i] = tstar;
    if (tid == 0) out_n[sk] = n_lt + n_eq;
}

// ---- K3 ------------------------------------------------------------------------------------
// HashSet semantics on ascending lists with duplicates: distinct counts + intersection by
// binary search; one warp per call, result valid in every lane.
__device__ __forceinline__ void warp_jaccard_counts(const uint64_t* __restrict__ a, uint32_t na, const uint64_t* __restrict__ b, uint32_t nb,
                                                    uint32_t& inter, uint32_t& uni) {
    const int lane = threadIdx.x & 31;
    uint32_t da = 0, db = 0, in = 0;
    for (uint32_t i = lane; i < na; i += 32) {
        const uint64_t x = a[i];
        if (i > 0 && a[i - 1] == x) continue;
        ++da;
        uint32_t lo = 0, hi = nb;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (b[mid] < x) lo = mid + 1;
            else hi = mid;
        }
        if (lo < nb && b[lo] == x) ++in;
    }
    for (uint32_t i = lane; i < nb; i += 32)
        if (i == 0 || b[i - 1] != b[i]) ++db;
    da = __reduce_add_sync(0xffffffffu, da);
    db = __reduce_add_sync(0xffffffffu, db);
    in = __reduce_add_sync(0xffffffffu, in);
    inter = in;
    uni = da + db - in;
}

// determine_orientation_mash (src/alignment.rs:69-94): stranded sketches live at slot index
// (2*i = forward, 2*i+1 = reverse complement); is_reverse = !(fwd_jaccard >= rev_jaccard)
__global__ void aw_orient_kernel(const aw_pair* __restrict__ pairs, uint64_t npairs, const uint64_t* __restrict__ sk, const uint32_t* __restrict__ sk_n,
                                 uint32_t sketch_size, uint8_t* __restrict__ is_reverse) {
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t p = warp; p < npairs; p += nwarps) {
        const uint32_t q = pairs[p].query_idx, t = pairs[p].target_idx;
        const uint64_t* T = sk + (size_t)(2 * t) * sketch_size;
        const uint64_t* F = sk + (size_t)(2 * q) * sketch_size;
        const uint64_t* R = sk + (size_t)(2 * q + 1) * sketch_size;
        uint32_t fi, fu, ri, ru;
        warp_jaccard_counts(F, sk_n[2 * q], T, sk_n[2 * t], fi, fu);
        warp_jaccard_counts(R, sk_n[2 * q + 1], T, sk_n[2 * t], ri, ru);
        const double fj = fu == 0 ? 0.0 : (double)fi / (double)fu;
        const double rj = ru == 0 ? 0.0 : (double)ri / (double)ru;
        if ((threadIdx.x & 31) == 0) is_reverse[p] = (fj >= rj) ? 0 : 1;
    }
}

// Per-pair divergence estimate for cost-ordered scheduling (BASELINE north_star: "greedy partitioner balanced by predicted
// cost (length times divergence)"): mash distance -1/k ln(2j/(1+j)) of the better of the two stranded Jaccards, i.e. of the
// strand determine_orientation_mash will pick.  Scheduling only: never enters a result.
__global__ void aw_divergence_kernel(const aw_pair* __restrict__ pairs, uint64_t npairs, const uint64_t* __restrict__ sk, const uint32_t* __restrict__ sk_n,
                                     uint32_t sketch_size, int k, float* __restrict__ out) {
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t p = warp; p < npairs; p += nwarps) {
        const uint32_t q = pairs[p].query_idx, t = pairs[p].target_idx;
        const uint64_t* T = sk + (size_t)(2 * t) * sketch_size;
        uint32_t fi, fu, ri, ru;
        warp_jaccard_counts(sk + (size_t)(2 * q) * sketch_size, sk_n[2 * q], T, sk_n[2 * t], fi, fu);
        warp_jaccard_counts(sk + (size_t)(2 * q + 1) * sketch_size, sk_n[2 * q + 1], T, sk_n[2 * t], ri, ru);
        const double fj = fu == 0 ? 0.0 : (double)fi / (double)fu, rj = ru == 0 ? 0.0 : (double)ri / (double)ru;
        const double j = fj >= rj ? fj : rj;
        double d = 1.0;
        if (j > 0.0) d = -log(2.0 * j / (1.0 + j)) / (double)k;
        if ((threadIdx.x & 31) == 0) out[p] = (float)fmin(fmax(d, 0.0), 1.0);
    }
}

// determine_orientation_wfa (src/alignment.rs:157-175): compare the X+I+D column counts of the two
// orientation alignments; fwd <= rev keeps the forward strand; a failed alignment counts as usize::MAX
__global__ void aw_wfa_orient_pick_kernel(const AwPairOut* __restrict__ fwd, const AwPairOut* __restrict__ rev, uint64_t npairs, uint8_t* __restrict__ is_reverse) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < npairs; i += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long f = fwd[i].status == AW_OK ? fwd[i].n_x + fwd[i].n_i + fwd[i].n_d : ~0ull;
        const unsigned long long r = rev[i].status == AW_OK ? rev[i].n_x + rev[i].n_i + rev[i].n_d : ~0ull;
        // a pass that ran out of first-try workspace has not failed: the strand stays undecided (2) and the host re-runs
        // both passes through the retry ladder before the pair is aligned (the reference completes both alignments)
        const bool undecided = fwd[i].status == AW_EWORKSPACE || rev[i].status == AW_EWORKSPACE;
        is_reverse[i] = undecided ? 2 : ((f <= r) ? 0 : 1);
    }
}

// ---- ordered PAF text (AW_FLAG_PAF_BLOCKS, AW_FLAG_CS): the alignment kernel appends lines to the text arena in completion
// order; these two kernels lay them out again in PAIR order (the order the reference's writer sees with one worker thread,
// src/main.rs:347-374), so a whole batch leaves the GPU as one ready-to-write block of lines.  A line is followed by '\n'
// when nl is 1, and with cs (AW_FLAG_CS) it gains the column "\tcs:Z:" + the pair's tag before that.
__device__ __forceinline__ unsigned long long ordered_line_len(const AwPairOut& o, const AwCsOut* cs, uint32_t i, unsigned nl) {
    if (o.status != AW_OK || o.paf_len == 0) return 0;
    return o.paf_len + nl + (cs ? 6 + cs[i].len : 0);
}
// off[i] = byte offset of pair i's line in the ordered arena, off[n] = total; one block, exclusive scan of the line lengths
__global__ void aw_text_scan_kernel(const AwPairOut* __restrict__ out, const AwCsOut* __restrict__ cs, unsigned nl, uint32_t n,
                                    unsigned long long* __restrict__ off) {
    __shared__ unsigned long long part[1024];
    const uint32_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint32_t b = min(n, threadIdx.x * per), e = min(n, b + per);
    unsigned long long sum = 0;
    for (uint32_t i = b; i < e; ++i) sum += ordered_line_len(out[i], cs, i, nl);
    part[threadIdx.x] = sum;
    __syncthreads();
    for (unsigned d = 1; d < blockDim.x; d <<= 1) {
        const unsigned long long t = threadIdx.x >= d ? part[threadIdx.x - d] : 0ull;
        __syncthreads();
        part[threadIdx.x] += t;
        __syncthreads();
    }
    unsigned long long run = part[threadIdx.x] - sum;
    for (uint32_t i = b; i < e; ++i) {
        off[i] = run;
        run += ordered_line_len(out[i], cs, i, nl);
    }
    if (threadIdx.x == blockDim.x - 1) off[n] = part[threadIdx.x];
}
// one warp per pair: copy the line (+ the cs column from the tag arena) (+ '\n') to its slot of the ordered arena
__global__ void aw_text_gather_kernel(const AwPairOut* __restrict__ out, const unsigned long long* __restrict__ off, uint32_t n, const char* __restrict__ src,
                                      const AwCsOut* __restrict__ cs, const char* __restrict__ tags, unsigned nl, char* __restrict__ dst) {
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const unsigned lane = threadIdx.x & 31;
    for (uint64_t p = warp; p < n; p += nwarps) {
        if (out[p].status != AW_OK || out[p].paf_len == 0) continue;
        const char* s = src + out[p].paf_off;
        char* d = dst + off[p];
        const unsigned len = out[p].paf_len;
        for (unsigned i = lane; i < len; i += 32) d[i] = s[i];
        d += len;
        if (cs) {
            const char col[6] = {'\t', 'c', 's', ':', 'Z', ':'};
            if (lane < 6) d[lane] = col[lane];
            const char* t = tags + cs[p].off;
            const unsigned long long tl = cs[p].len;
            for (unsigned long long i = lane; i < tl; i += 32) d[6 + i] = t[i];
            d += 6 + tl;
        }
        if (nl && lane == 0) *d = '\n';
    }
}

// all-pairs canonical Jaccard counts, i<j (src/mash.rs:156-162); one warp per (i,j)
__global__ void aw_jaccard_matrix_kernel(uint32_t n, const uint64_t* __restrict__ sk, const uint32_t* __restrict__ sk_n, uint32_t sketch_size,
                                         uint32_t* __restrict__ inter, uint32_t* __restrict__ uni) {
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t total = (uint64_t)n * n;
    for (uint64_t c = warp; c < total; c += nwarps) {
        const uint32_t i = (uint32_t)(c / n), j = (uint32_t)(c % n);
        if (i >= j) continue;
        uint32_t in, un;
        warp_jaccard_counts(sk + (size_t)i * sketch_size, sk_n[i], sk + (size_t)j * sketch_size, sk_n[j], in, un);
        if ((threadIdx.x & 31) == 0) {
            inter[(size_t)i * n + j] = in;
            uni[(size_t)i * n + j] = un;
            inter[(size_t)j * n + i] = in;
            uni[(size_t)j * n + i] = un;
        }
    }
}

}  // namespace awk
