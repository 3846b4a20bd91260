// aw_cs.cuh -- minimap2's cs:Z: difference string (AW_FLAG_CS / AW_FLAG_CS_LONG), built after the alignment passes from each
// pair's CIGAR op bytes (WFA2 letters M X I D, one per column) and the ASCII copies of the target (slot 2t) and of the
// oriented query (slot 2q + is_reverse, the sequence the CIGAR refers to).
//
// Tokens, left to right along the CIGAR: a run of M -> ":N" (short) or "=" + the target bases upper-cased (long); every X
// column -> "*" + target base + query base; a run of WFA2 D (query bases only, PAF 'I') -> "+" + the query bases; a run of
// WFA2 I (target bases only, PAF 'D') -> "-" + the target bases.  Bases of "*", "+" and "-" are lower-cased; only A-Z
// change case, every other byte is written as it is.  A tag is at most 2 * (qlen + tlen) bytes: no token writes more than
// two bytes per base it consumes (":1" for one match, "+a" for one inserted base, "*ac" for two bases).
//
// Kept apart from the alignment kernel on purpose: aw_align_kernel is sensitive to its instruction-cache footprint and
// register pressure, and this pass needs neither its registers nor its shared memory.
#pragma once
#include "aw_common.cuh"
#include "aw_wfa.cuh"

namespace awk {

// threads per pair: one warp while the batch's pairs are short (a few columns per thread of a full CTA would leave the pass
// dominated by its block scans), a full CTA otherwise
constexpr int CS_NT_SHORT = 32, CS_NT = 256;
constexpr unsigned long long CS_SHORT_LEN = 4096;  // plen + tlen of the batch's longest pair up to which CS_NT_SHORT is used

__device__ __forceinline__ char cs_lower(uint8_t b) { return (char)((b >= 'A' && b <= 'Z') ? b + 32 : b); }
__device__ __forceinline__ char cs_upper(uint8_t b) { return (char)((b >= 'a' && b <= 'z') ? b - 32 : b); }

// The bytes of the tokens that START in columns [a, b) of one pair (a token that starts earlier belongs to an earlier
// thread, even where its bases lie in this chunk); with WRITE they are written to dst.  nb: the first token boundary at or
// after b (ncols when there is none), where a run of M that reaches b ends; t, q: target and query position of column a.
template <bool WRITE>
__device__ unsigned long long cs_chunk(const uint8_t* __restrict__ ops, unsigned long long a, unsigned long long b, unsigned long long nb,
                                       bool long_form, const uint8_t* __restrict__ T, const uint8_t* __restrict__ Q, unsigned long long t,
                                       unsigned long long q, char* __restrict__ dst) {
    unsigned long long n = 0;
    uint8_t prev = a ? ops[a - 1] : 0;
    for (unsigned long long c = a; c < b; ++c) {
        const uint8_t op = ops[c];
        const bool start = op != prev;  // (an X column is a token of its own whatever precedes it)
        prev = op;
        if (op == 'X') {
            if (WRITE) {
                dst[n] = '*';
                dst[n + 1] = cs_lower(T[t]);
                dst[n + 2] = cs_lower(Q[q]);
            }
            n += 3;
            ++t;
            ++q;
        } else if (op == 'M') {
            if (long_form) {
                if (start) {
                    if (WRITE) dst[n] = '=';
                    ++n;
                }
                if (WRITE) dst[n] = cs_upper(T[t]);
                ++n;
            } else if (start) {
                unsigned long long e = c + 1;
                while (e < b && ops[e] == 'M') ++e;
                if (e == b) e = nb;
                if (WRITE) {
                    dst[n] = ':';
                    put_u64(dst + n + 1, e - c);
                }
                n += 1 + ndigits(e - c);
            }
            ++t;
            ++q;
        } else if (op == 'I') {  // WFA2 I: a target base the query lacks
            if (start) {
                if (WRITE) dst[n] = '-';
                ++n;
            }
            if (WRITE) dst[n] = cs_lower(T[t]);
            ++n;
            ++t;
        } else {  // WFA2 D: a query base the target lacks
            if (start) {
                if (WRITE) dst[n] = '+';
                ++n;
            }
            if (WRITE) dst[n] = cs_lower(Q[q]);
            ++n;
            ++q;
        }
    }
    return n;
}

// min of v over the threads above this one (none when there is none); sbuf: NT entries of shared memory
template <int NT>
__device__ __forceinline__ unsigned long long block_min_above(unsigned long long v, unsigned long long none, unsigned long long* sbuf) {
    const int tid = threadIdx.x;
    cta_sync<NT>();
    sbuf[tid] = v;
    cta_sync<NT>();
    for (int d = 1; d < NT; d <<= 1) {
        const unsigned long long o = tid + d < NT ? sbuf[tid + d] : none;
        cta_sync<NT>();
        sbuf[tid] = min(sbuf[tid], o);
        cta_sync<NT>();
    }
    return tid + 1 < NT ? sbuf[tid + 1] : none;
}

// One CTA of NT threads per pair: the pairs order[0 .. n) (0 .. n without an order) whose alignment succeeded.  The CTA
// splits the pair's columns into one contiguous chunk per thread; block scans give each thread the target / query position of its chunk, the
// end of a run of matches that crosses its chunk's end, and the output offset of its tokens.  The tag goes to the tag arena
// at a cursor-allocated offset, recorded in cs_out[pair] (failed pairs get an empty record).
template <int NT>
__global__ void __launch_bounds__(NT) aw_cs_kernel(const AwPairOut* __restrict__ out, const uint32_t* __restrict__ order, uint32_t n,
                                                     const aw_pair* __restrict__ pairs, const AwSlot* __restrict__ slots,
                                                     const uint8_t* __restrict__ ascii, const uint8_t* __restrict__ ops, int long_form,
                                                     char* __restrict__ tags, unsigned long long* tag_cursor, AwCsOut* __restrict__ cs_out) {
    __shared__ unsigned long long sbuf[NT];
    __shared__ unsigned long long s_base;
    const unsigned tid = threadIdx.x;
    for (uint32_t j = blockIdx.x; j < n; j += gridDim.x) {
        const uint32_t i = order ? order[j] : j;
        const AwPairOut& o = out[i];
        if (o.status != AW_OK) {
            if (tid == 0) cs_out[i] = AwCsOut{0, 0};
            continue;
        }
        const unsigned long long ncols = o.n_m + o.n_x + o.n_i + o.n_d;
        const uint8_t* op = ops + o.bytes_off;
        const uint8_t* T = ascii + slots[2ull * pairs[i].target_idx].ascii_off;
        const uint8_t* Q = ascii + slots[2ull * pairs[i].query_idx + (o.is_reverse == 1)].ascii_off;
        const unsigned long long chunk = (ncols + NT - 1) / NT;
        const unsigned long long a = min(ncols, tid * chunk), b = min(ncols, a + chunk);
        // first token boundary of the chunk, and the bases the chunk consumes (target << 32 | query: both < 2^27)
        unsigned long long first = ncols, tq = 0;
        for (unsigned long long c = a; c < b; ++c) {
            const uint8_t x = op[c];
            if (first == ncols && (c == 0 || x == 'X' || x != op[c - 1])) first = c;
            tq += (x != 'D' ? 1ull << 32 : 0ull) + (x != 'I' ? 1ull : 0ull);
        }
        const unsigned long long nb = block_min_above<NT>(first, ncols, sbuf);
        unsigned long long total;
        const unsigned long long pos = block_excl_scan<NT>(tq, sbuf, &total);
        const unsigned long long t0 = pos >> 32, q0 = pos & 0xffffffffull;
        const unsigned long long mine = cs_chunk<false>(op, a, b, nb, long_form != 0, T, Q, t0, q0, nullptr);
        const unsigned long long off = block_excl_scan<NT>(mine, sbuf, &total);
        if (tid == 0) {
            s_base = atomicAdd(tag_cursor, total);
            cs_out[i] = AwCsOut{s_base, total};
        }
        cta_sync<NT>();
        cs_chunk<true>(op, a, b, nb, long_form != 0, T, Q, t0, q0, tags + s_base + off);
        cta_sync<NT>();  // s_base and sbuf are reused by the next pair
    }
}

}  // namespace awk
