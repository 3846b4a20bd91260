// aw_wfa.cuh -- the alignment hot path as one persistent sm_100a kernel per pair class:
//   K4 wavefront compute (gap-affine / gap-affine-2p M,I1,D1,I2,D2 recurrences)
//   K5 match extend (XOR + popc/clz longest common prefix on 2-bit packed or byte words)
//   K6 biWFA breakpoint search (forward/reverse wavefronts, overlap test, DFS recursion stack)
//   K7 base case: full-history unidirectional WFA + WFA2-ordered backtrace
//   K8 CIGAR run-length encoding, op statistics, score, PAF text
// One CTA owns one pair at a time and pulls pairs from a global work counter.  Replaces lib_wfa2's
// AffineWavefronts::align as driven by /root/reference/src/alignment.rs:201-261 and the CIGAR/PAF passes of
// src/alignment.rs:292-376 + src/lib.rs:71-112.  Tie-break constants: include/aw_wfa2_compat.h.
//
// Two wavefront-step engines share the driver (aw_align_kernel):
//   * chunked (VEC: 2-bit sequences, NT >= 64; int16 or int32 rows): v_launch / wf_cells_v / v_finish -- every thread owns
//     16 bytes of consecutive diagonals, packed int16x2 recurrences, arithmetic trim, block maxima for the overlap test;
//   * scalar (byte sequences or the one-warp NT=32 kernels): launch_dir / wf_cells / finish_dir -- one diagonal per thread
//     per iteration with explicit edge tracking.
// DESIGN.md section 4 describes both and lists the measured experiments behind the compile-time flags below.
#pragma once
#include <limits.h>

#include "aw_common.cuh"

namespace awk {

#define AW_KFLAG_COUNT_ONLY 0x100u  // internal: statistics only (orientation passes), no text output
#ifndef AW_PREFETCH_STEPS
#define AW_PREFETCH_STEPS 0  // chunked path: L2 prefetch distance (score steps) for the old M rows; 0 = off (measured: no gain on C2)
#endif
#ifndef AW_COMPACT_ID_RINGS
// int16 path: 1 = far from the overlap phase, I/D rows rotate through small rings (extension distance + 1 rows) so that they
// are overwritten while still in L2.  Measured on C2 (592 pairs in flight): HBM writes -28 % but no speed-up (the M rings
// alone overflow L2), and the extra addressing costs ~10 %, so it is off by default.
#define AW_COMPACT_ID_RINGS 0
#endif
#ifndef AW_L1_PREFETCH
#define AW_L1_PREFETCH 0  // chunked path: after a step, prefetch into L1 the row chunks the next step will read (measured: -3 % on C2, off)
#endif
#ifndef AW_PREFETCH_NEXT_ITER
#define AW_PREFETCH_NEXT_ITER 1  // chunked path: prefetch (L1) the rows of a warp's next iteration while it computes the current one
#endif
#ifndef AW_PF_DIST32
#define AW_PF_DIST32 1  // int32 rows: prefetch distance (warp iterations) of the row loads, into L2 (measured on 296 x 100 kb pairs: 1: 17.0 s, 4: 17.6 s, 8: 18.6 s, 16: 18.8 s)
#endif
#ifndef AW_LOAD_CG
#define AW_LOAD_CG 0  // chunked path: 1 = row loads bypass L1 (ld.global.cg)
#endif
#ifndef AW_CYCLE_COUNTERS
#define AW_CYCLE_COUNTERS 0  // (build with -DAW_CYCLE_COUNTERS=1 for tools/perf_probe.py) per-phase device-clock breakdown in AwPairOut::cyc (aw_batch_debug_cycles); 0 frees ~14 registers
#endif
#ifndef AW_LEAFPAR
#define AW_LEAFPAR 1  // warp-parallel leaves (see LEAFPAR in aw_align_kernel); 0 = every base case on the whole CTA (tuning builds)
#endif
#ifndef AW_REGS
#define AW_REGS 128  // register budget per thread of the CTA-per-pair kernels: resident CTAs per SM = 65536 / (NT * AW_REGS)
#endif
#define AW_CTAS_PER_SM(NT) ((NT) == 32 ? 1 : (65536 / ((NT) * AW_REGS)))
constexpr int NRED = 20;       // reduction slots, see RED_* below
constexpr int MAX_STACK = 96;  // DFS depth bound of the biWFA recursion
constexpr int HIST_META_INTS = 16;
constexpr int EDGE_ZONE = 64;  // I/D in-bounds tracking is only done this close to a wavefront end
constexpr int SEQ_SMEM_WORDS = 2048;  // 8 KB of shared memory for the pair's packed sequences (guards included)
// int16 wavefront storage: every negative value means "null".  Packed kernels let null values drift
// upwards by +1 per insertion step, at most once per diagonal, so NULL16 + (plen + tlen) stays negative
// (plan_launch only selects int16 when 2*tlen+plen and 2*plen+tlen are below 32000).
constexpr short NULL16 = -32000;
constexpr uint32_t NULL16X2 = 0x83008300u;
enum { IN_MX = 0, IN_MO1, IN_I1E, IN_D1E, IN_MO2, IN_I2E, IN_D2E };
enum { ST_OK = 0, ST_END_REACHED = 1, ST_FAIL_WORKSPACE = 2 };
// red[] layout: per component c: RED_HI+c = max in-bounds k, RED_LO+c = max(-k); then the two
// antidiagonal bounds and the value at the end cell
// chunked path only: RED_OOB = the row holds a non-null out-of-bounds cell, RED_CLO/RED_CHI = computed range of the row
// (published by the planning warp), RED_FAIL = the row does not fit the workspace
enum { RED_HI = 0, RED_LO = 5, RED_AKM = 10, RED_AKALL = 11, RED_END = 12, RED_OOB = 13, RED_CLO = 14, RED_CHI = 15, RED_FAIL = 16 };

struct SlotMeta {
    int lo[5], hi[5];   // trimmed range per component; empty iff lo > hi
    int akM;            // max antidiagonal 2*off-k over valid extended M cells (INT_MIN if none)
    int akAll;          // upper bound of 2*off-k over every component's non-null cells
    int off;            // workspace element offset of (component 0, k = 0) of this wavefront
    int cstride;        // elements between consecutive components
    int wlo, whi;       // int16 rows: diagonals that read back correctly without masking (NULL outside the trimmed range)
    int coff[5];        // int16 rows: element offset of (component c, k = 0), indexed by AW_COMP_*
    int full;           // int16 ring rows: 1 = the I/D components sit in the full ring (readable for `scope` steps), 0 = compact ring
    int bk0, nblk;      // int16 ring rows: first diagonal of block 0 and number of blocks of the per-block maxima
};

struct In {
    int off;     // element k lives at ws[off + k]
    int lo, hi;  // trimmed range; empty iff lo > hi
};

struct SubProblem {
    int pb, pe, tb, te;  // half-open ranges in the pair's pattern / text
    int cb, ce;          // begin / end component
    int rem;             // score_remaining
};

struct Breakpoint {
    int score, score_f, score_r, k_f, off_f, comp;
};

struct KParams {
    // sequence store
    const AwSlot* slots;
    const uint32_t* packed;
    const uint8_t* ascii;
    const char* ids;
    const uint32_t* id_off;  // n+1 offsets into ids
    // work list
    const aw_pair* pairs;
    const uint8_t* is_reverse;  // per pair, from the orientation stage
    const uint32_t* order;      // processing order (heaviest first) or NULL
    uint32_t npairs;
    unsigned int* next_pair;
    AwPen pen;
    uint32_t flags;
    // per-CTA workspace: [ring: 2 x (scope+1) x ncomp x W ints][history arena: hist_ints]
    int* ws;
    unsigned long long ws_ints_per_cta;
    int W;                   // allocated diagonals per ring wavefront
    int hist_ints;           // history arena size (ints)
    uint2* ws_seq2;          // chunked path, pairs too long for shared memory: [cta][seq2_cap] staged sequence word pairs
    unsigned long long seq2_cap;
    int* ws_blk;             // int16 path: [cta][2 directions][scope+1 slots][blk_cap][2] per-block (akM, akAll) maxima
    int blk_cap;
    int* ws_hist_meta;       // [cta][hist_max_scores][HIST_META_INTS]
    int hist_max_scores;
    uint32_t* ws_runs;       // [cta][2][runs_cap]: pair runs, then leaf scratch
    unsigned long long runs_cap;
    // outputs
    AwPairOut* out;          // [npairs]
    char* text;
    unsigned long long* text_cursor;
    unsigned long long text_cap;
    uint8_t* bytes;
    unsigned long long* bytes_cursor;
    unsigned long long bytes_cap;
    int solo_len;            // cluster kernels: sub-problems with plen + tlen below this run on CTA 0 of the cluster alone
};

// ------------------------------------------------------------------------------------------
// Thread-block cluster helpers (Mb-scale pairs: one pair per cluster, see aw_align_kernel).  barrier.cluster with
// release / acquire semantics orders global and distributed-shared-memory accesses of all CTAs of the cluster.
__device__ __forceinline__ unsigned cluster_ctarank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// reads the int at the same shared-memory address in CTA `rank` of the cluster (DSMEM)
__device__ __forceinline__ int ld_dsmem_int(const int* p, unsigned rank) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(p);
    unsigned ra;
    int v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
    asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(ra) : "memory");
    return v;
}

template <int NT>
__device__ __forceinline__ void cta_sync() {
    if (NT == 32) __syncwarp();
    else __syncthreads();
}

template <int NT>
__device__ __forceinline__ void red_max(int* red, int idx, int v) {
    v = __reduce_max_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v != INT_MIN) {
        if (NT == 32) red[idx] = v;
        else atomicMax(&red[idx], v);
    }
}

// ---- K5: longest common prefix on packed words -------------------------------------------
// BITS = 2 (2-bit packed, 16 symbols / word) or 8 (ASCII, 4 symbols / word).  Guard words
// either side of every sequence make the over-reads legal; the result is clamped to maxlen.
//@region lcp/extend helpers
template <int BITS>
__device__ __forceinline__ uint32_t load_fwd(const uint32_t* __restrict__ w, int pos) {
    constexpr int SPW = 32 / BITS;
    const unsigned idx = (unsigned)pos / SPW;  // pos >= 0
    const int sh = ((unsigned)pos % SPW) * BITS;
    return __funnelshift_r(w[idx], w[idx + 1], sh);
}
// symbols pos, pos-1, ... with `pos` in the most significant bits
template <int BITS>
__device__ __forceinline__ uint32_t load_rev(const uint32_t* __restrict__ w, int pos) {
    constexpr int SPW = 32 / BITS;
    const unsigned idx = (unsigned)pos / SPW;
    const int sh = (((unsigned)pos % SPW) + 1) * BITS;  // in [BITS, 32]
    return __funnelshift_rc(w[(int)idx - 1], w[idx], sh);
}
template <int BITS>
__device__ __forceinline__ int lcp_fwd(const uint32_t* __restrict__ pw, int pv, const uint32_t* __restrict__ tw, int th, int maxlen) {
    constexpr int SPW = 32 / BITS;
    int n = 0;
    while (n < maxlen) {
        const uint32_t x = load_fwd<BITS>(pw, pv + n) ^ load_fwd<BITS>(tw, th + n);
        if (x) {
            n += (__ffs(x) - 1) / BITS;
            break;
        }
        n += SPW;
    }
    return min(n, maxlen);
}
template <int BITS>
__device__ __forceinline__ int lcp_rev(const uint32_t* __restrict__ pw, int pv, const uint32_t* __restrict__ tw, int th, int maxlen) {
    constexpr int SPW = 32 / BITS;
    int n = 0;
    while (n < maxlen) {
        const uint32_t x = load_rev<BITS>(pw, pv - n) ^ load_rev<BITS>(tw, th - n);
        if (x) {
            n += __clz(x) / BITS;
            break;
        }
        n += SPW;
    }
    return min(n, maxlen);
}

// one aligner's view of the sub-problem sequences (wavefront_sequences_set_bounds): the reverse
// aligner reads both sub-ranges back to front
struct SeqView {
    const uint32_t* pw;
    const uint32_t* tw;
    int p0, t0;  // absolute symbol of v=0 / h=0 (forward: range begin; reverse: range end - 1)
    int plen, tlen;
    bool rev;
};
template <int BITS>
__device__ __forceinline__ int extend_cell(const SeqView& s, int k, int off) {
    const int v = off - k, h = off;
    const int maxlen = min(s.plen - v, s.tlen - h);
    if (maxlen <= 0) return off;
    const int n = s.rev ? lcp_rev<BITS>(s.pw, s.p0 - v, s.tw, s.t0 - h, maxlen) : lcp_fwd<BITS>(s.pw, s.p0 + v, s.tw, s.t0 + h, maxlen);
    return off + n;
}

// first (branch-free) round of the match extension: up to one word of symbols.  `more` is set
// when the whole word matched and symbols remain (the caller continues with lcp_fwd/lcp_rev).
template <int BITS>
__device__ __forceinline__ void extend_first(const SeqView& s, int k, int off, int& n, bool& more) {
    constexpr int SPW = 32 / BITS;
    int v = off - k, h = off;
    const int maxlen = min(s.plen - v, s.tlen - h);
    if (maxlen <= 0) v = h = 0;  // nothing to compare: keep the (unused) loads inside the sequences
    uint32_t x;
    int cnt;
    if (s.rev) {
        x = load_rev<BITS>(s.pw, s.p0 - v) ^ load_rev<BITS>(s.tw, s.t0 - h);
        cnt = __clz(x) / BITS;  // clz(0) = 32 -> SPW
    } else {
        x = load_fwd<BITS>(s.pw, s.p0 + v) ^ load_fwd<BITS>(s.tw, s.t0 + h);
        cnt = x ? (__ffs(x) - 1) / BITS : SPW;
    }
    n = max(0, min(cnt, maxlen));
    more = (x == 0) && (maxlen > SPW);
}
template <int BITS>
__device__ __forceinline__ int extend_rest(const SeqView& s, int k, int off) {  // off already advanced by one word
    constexpr int SPW = 32 / BITS;
    const int v = off - k, h = off;
    const int maxlen = min(s.plen - v, s.tlen - h);
    if (maxlen <= 0) return off;
    const int n = s.rev ? lcp_rev<BITS>(s.pw, s.p0 - v, s.tw, s.t0 - h, maxlen) : lcp_fwd<BITS>(s.pw, s.p0 + v, s.tw, s.t0 + h, maxlen);
    (void)SPW;
    return off + n;
}

// workspace element type: int (any length) or short (offsets < 32000; halves the L2/HBM footprint).
// Every negative offset means "null", so the int16 form stores one canonical negative value.
template <class WS>
__device__ __forceinline__ WS to_ws(int v);
template <>
__device__ __forceinline__ int to_ws<int>(int v) { return v; }
template <>
__device__ __forceinline__ short to_ws<short>(int v) { return (short)(v < 0 ? (int)NULL16 : v); }

//@region wf_cells scalar
struct StepOut {
    int lo[5], hi[5];
    int akM, akAll;
    int endval;
    bool ambiguous;  // an I/D trim end fell outside the tracked edge zones (needs an exact rescan)
};

// ---- K4+K5: compute wavefront s from its inputs, extend M, and accumulate the block-wide
// reductions (trim ends, antidiagonal bounds, end-cell value) into `red`.  No barrier here.
// Restates wavefront_compute_affine2p_idm + wavefront_extend_matches_packed_end2end(_max)
// (SURVEY A.2, A.3).  `red` must hold INT_MIN on entry.
template <int NT, int BITS, bool TWO, class WS>
__device__ __forceinline__ void wf_cells(WS* __restrict__ ws, const In (&in)[7], const int (&out)[5], int lo, int hi, const SeqView& sv, int k_end,
                                         int comp_end, int* red) {
    const int tid = threadIdx.x;
    const unsigned tlen = (unsigned)sv.tlen, plen = (unsigned)sv.plen;
    // interior cells whose every input (k-1, k, k+1) is inside every input's range need no checks
    int fast_lo = INT_MIN, fast_hi = INT_MAX;
    {
        bool all_present = true;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            if (!TWO && i >= IN_MO2) continue;
            all_present = all_present && (in[i].lo <= in[i].hi);
            fast_lo = max(fast_lo, in[i].lo + 1);
            fast_hi = min(fast_hi, in[i].hi - 1);
        }
        if (!all_present) {
            fast_lo = 1;
            fast_hi = 0;
        }
    }
    const bool narrow = (hi - lo) < 2 * EDGE_ZONE;
    int akM = INT_MIN, akAll = INT_MIN;
    // in-bounds ends of one component inside an edge row: one ballot, the leader lane publishes both ends
    auto edge_track = [&](int c, bool inb, int krow) {
        const unsigned amask = __activemask();
        const unsigned mask = __ballot_sync(amask, inb);
        if (mask != 0 && (int)(tid & 31) == __ffs(amask) - 1) {
            atomicMax(&red[RED_HI + c], krow + 31 - __clz(mask));
            atomicMax(&red[RED_LO + c], -(krow + __ffs(mask) - 1));
        }
    };
    // one running base pointer (ws + k) plus a 32-bit element offset per input / output array
    const int k0 = lo + tid;
    WS* pk = ws + k0;
    const int o_mx = in[IN_MX].off, o_mo1 = in[IN_MO1].off, o_i1e = in[IN_I1E].off, o_d1e = in[IN_D1E].off;
    const int o_mo2 = in[IN_MO2].off, o_i2e = in[IN_I2E].off, o_d2e = in[IN_D2E].off;
    const int w_m = out[AW_COMP_M], w_i1 = out[AW_COMP_I1], w_d1 = out[AW_COMP_D1], w_i2 = out[AW_COMP_I2], w_d2 = out[AW_COMP_D2];
    // one cell: recurrences, bounds, extend, stores, trim / antidiagonal tracking
    auto cell = [&](int k, int j, int mo1l, int mo1r, int i1l, int d1r, int mo2l, int mo2r, int i2l, int d2r, int mx) {
        const int i1 = max(mo1l, i1l) + 1;
        const int d1 = max(mo1r, d1r);
        int i2 = AW_NULLV, d2 = AW_NULLV, ins = i1, del = d1;
        if (TWO) {
            i2 = max(mo2l, i2l) + 1;
            d2 = max(mo2r, d2r);
            ins = max(i1, i2);
            del = max(d1, d2);
        }
        int m = max(del, max(mx + 1, ins));
        if (m >= 0) akAll = max(akAll, 2 * m - k);  // m (pre-null) dominates every component at k
        if ((unsigned)m > tlen || (unsigned)(m - k) > plen) m = AW_NULLV;
        if (m >= 0) {
            m = extend_cell<BITS>(sv, k, m);
            akM = max(akM, 2 * m - k);
        }
        (void)j;
        pk[w_m] = to_ws<WS>(m);
        pk[w_i1] = to_ws<WS>(i1);
        pk[w_d1] = to_ws<WS>(d1);
        if (TWO) {
            pk[w_i2] = to_ws<WS>(i2);
            pk[w_d2] = to_ws<WS>(d2);
        }
        // wavefront_compute_trim_ends keeps [first, last] in-bounds cell of every component: only rows
        // (32 consecutive diagonals of one warp) that touch an edge zone can hold those ends
        const int krow = k - (int)(tid & 31);
        if (narrow || krow - lo < EDGE_ZONE || hi - (krow + 31) < EDGE_ZONE) {
            edge_track(AW_COMP_M, m >= 0, krow);
            edge_track(AW_COMP_I1, (unsigned)i1 <= tlen && (unsigned)(i1 - k) <= plen, krow);
            edge_track(AW_COMP_D1, (unsigned)d1 <= tlen && (unsigned)(d1 - k) <= plen, krow);
            if (TWO) {
                edge_track(AW_COMP_I2, (unsigned)i2 <= tlen && (unsigned)(i2 - k) <= plen, krow);
                edge_track(AW_COMP_D2, (unsigned)d2 <= tlen && (unsigned)(d2 - k) <= plen, krow);
            }
        }
        if (k == k_end) red[RED_END] = (comp_end == AW_COMP_M) ? m : (comp_end == AW_COMP_I1) ? i1 : (comp_end == AW_COMP_D1) ? d1 : (comp_end == AW_COMP_I2) ? i2 : d2;
    };
    int k = k0;
    for (; k <= hi; k += NT) {
        int mo1l, mo1r, i1l, d1r, mo2l = AW_NULLV, mo2r = AW_NULLV, i2l = AW_NULLV, d2r = AW_NULLV, mx;
        if (k >= fast_lo && k <= fast_hi) {  // interior: immediate-offset loads, no checks
            mo1l = pk[o_mo1 - 1];
            mo1r = pk[o_mo1 + 1];
            i1l = pk[o_i1e - 1];
            d1r = pk[o_d1e + 1];
            if (TWO) {
                mo2l = pk[o_mo2 - 1];
                mo2r = pk[o_mo2 + 1];
                i2l = pk[o_i2e - 1];
                d2r = pk[o_d2e + 1];
            }
            mx = pk[o_mx];
        } else {
            auto ck = [&](const In& w, int o, int d) -> int { return (k + d >= w.lo && k + d <= w.hi) ? (int)pk[o + d] : AW_NULLV; };
            mo1l = ck(in[IN_MO1], o_mo1, -1);
            mo1r = ck(in[IN_MO1], o_mo1, 1);
            i1l = ck(in[IN_I1E], o_i1e, -1);
            d1r = ck(in[IN_D1E], o_d1e, 1);
            if (TWO) {
                mo2l = ck(in[IN_MO2], o_mo2, -1);
                mo2r = ck(in[IN_MO2], o_mo2, 1);
                i2l = ck(in[IN_I2E], o_i2e, -1);
                d2r = ck(in[IN_D2E], o_d2e, 1);
            }
            mx = ck(in[IN_MX], o_mx, 0);
        }
        cell(k, 0, mo1l, mo1r, i1l, d1r, mo2l, mo2r, i2l, d2r, mx);
        pk += NT;
    }
    red_max<NT>(red, RED_AKM, akM);
    red_max<NT>(red, RED_AKALL, akAll);
}

// ---- match extension of the int16 path: 2-bit sequences staged in shared memory as overlapping word
// pairs, entry i = (w[i], w[i+1]), so one 8-byte load + one funnel shift yields the 16 symbols that start
// at any position.  The reverse aligner reads reversed copies (wavefront_sequences_init_* keeps reversed
// copies too), so there is only a forward code path.
constexpr int SEQ2_ENTRIES = 2720;  // uint2 entries for 2 x (pattern + text): plen + tlen <= 21696 symbols
__device__ __forceinline__ uint32_t load16(const uint2* __restrict__ s2, int pos) {
    // entry pos/16 at byte offset (pos >> 1) & ~7; the funnel shift uses the low 5 bits of its amount = 2 * (pos % 16)
    const uint2 e = *reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(s2) + (((unsigned)pos >> 1) & ~7u));
    return __funnelshift_r(e.x, e.y, pos << 1);
}
// The same 16-symbol window from an array staged in SHARED memory, addressed by q = 2 * position + 4 * (byte address of the
// array in the CTA's shared window): byte address = (q >> 2) & ~7, funnel shift = q mod 32.  The address is confined to the
// first 32 KB of the window, so any q (null or out-of-bounds cells) reads legal memory; the caller discards such results.
constexpr unsigned SEQ2_WINDOW = 32768;
__device__ __forceinline__ uint32_t ld16s(int q) {
    const uint32_t a = ((uint32_t)q >> 2) & (SEQ2_WINDOW - 8);
    uint32_t lo, hi;
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(a));
    return __funnelshift_r(lo, hi, q);
}
// matching symbols from (pp, tp), at most maxlen
__device__ __forceinline__ int lcp2(const uint2* __restrict__ p2, const uint2* __restrict__ t2, int pp, int tp, int maxlen) {
    int n = 0;
    while (n < maxlen) {
        const uint32_t x = load16(p2, pp + n) ^ load16(t2, tp + n);
        if (x) {
            n += __clz(__brev(x)) >> 1;
            break;
        }
        n += 16;
    }
    return min(n, maxlen);
}

//@region wf_cells_v
// ---- K4+K5, int16 storage: every thread owns CPT consecutive diagonals ("chunk") --------------
// Rows are chunk-aligned in memory, so one 16-byte (CPT=8) or 8-byte (CPT=4) load fetches an input
// row for the whole chunk; the recurrences run on packed int16x2 words (VIMNMX/VIADD.16x2), the
// k-1 / k+1 neighbours come from the adjacent lanes by shuffle (lanes 0 and 31 of a warp are halo
// lanes that only load), and only the match extension is scalar.
//
// Reads outside an input's trimmed [lo,hi] must see OFFSET_NULL (wavefront_compute_init_ends).
// Every stored row therefore carries a NULL-filled margin of VMARGIN diagonals either side of its
// computed range, and its SlotMeta says which diagonals [wlo,whi] read back correctly without
// masking; absent inputs point at an all-NULL row.  A chunk inside every input's [wlo,whi] takes
// plain vector loads, the rest mask element by element.
//
// wavefront_compute_trim_ends without per-cell tracking: as long as no cell of the row is a
// non-null offset outside the sequences ("oob"; M's pre-null value dominates every component at
// its diagonal, so testing that one value covers all five), the trimmed range of every output
// component follows arithmetically from the inputs' trimmed ranges (their end cells are in bounds,
// hence non-null).  Rows that do hold such a cell raise RED_OOB and are trimmed exactly by
// wf_rescan after the barrier.
constexpr int VMARGIN = 48;
// Every warp iteration of the cell loop (VBLOCK diagonals) also records its own maxima of the two antidiagonal bounds
// (akM, akAll).  The overlap test uses them to skip (candidate, block) pairs that cannot contain a meeting point, which
// is almost all of them: the wavefronts only touch near the optimal path.
constexpr int VBLOCK_CHUNKS = 30;  // = chunks owned per warp iteration
constexpr int VBIG = 1 << 28;

// Element traits of the chunked loop: int16 rows hold two cells per 32-bit word (packed VIMNMX / VIADD.16x2
// arithmetic), int32 rows one.  A chunk is always 16 bytes: 8 int16 cells or 4 int32 cells.
template <class WS>
struct VecT;
template <>
struct VecT<short> {
    static constexpr int CPW = 2;  // cells per word
    static constexpr uint32_t NULLW = NULL16X2;
    static constexpr int NULLV = NULL16;
    static __device__ __forceinline__ uint32_t vmax(uint32_t a, uint32_t b) { return __vmaxs2(a, b); }
    static __device__ __forceinline__ uint32_t inc(uint32_t a) { return a + 0x00010001u; }  // nulls never hold 0xffff: no carry between halves
    static __device__ __forceinline__ uint32_t mstep(uint32_t mx, uint32_t i1) { return __viaddmax_s16x2(mx, 0x00010001u, i1); }  // max(mx + 1, i1)
    static __device__ __forceinline__ uint32_t vmax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_s16x2(a, b, c); }
    // words of a row shifted by one cell: `lo` supplies the cell that moves in from the left / `hi` from the right
    static __device__ __forceinline__ uint32_t shl1(uint32_t lo, uint32_t cur) { return __byte_perm(lo, cur, 0x5432); }
    static __device__ __forceinline__ uint32_t shr1(uint32_t cur, uint32_t hi) { return __byte_perm(cur, hi, 0x5432); }
    static __device__ __forceinline__ int get(const uint32_t* v, int j) { return (j & 1) ? (int)v[j >> 1] >> 16 : (int)(short)(v[j >> 1] & 0xffffu); }
};
template <>
struct VecT<int> {
    static constexpr int CPW = 1;
    static constexpr uint32_t NULLW = (uint32_t)AW_NULLV;
    static constexpr int NULLV = AW_NULLV;
    static __device__ __forceinline__ uint32_t vmax(uint32_t a, uint32_t b) { return (uint32_t)max((int)a, (int)b); }
    static __device__ __forceinline__ uint32_t inc(uint32_t a) { return a + 1u; }
    static __device__ __forceinline__ uint32_t mstep(uint32_t mx, uint32_t i1) { return (uint32_t)max((int)mx + 1, (int)i1); }
    static __device__ __forceinline__ uint32_t vmax3(uint32_t a, uint32_t b, uint32_t c) { return (uint32_t)max((int)a, max((int)b, (int)c)); }
    static __device__ __forceinline__ uint32_t shl1(uint32_t lo, uint32_t) { return lo; }
    static __device__ __forceinline__ uint32_t shr1(uint32_t, uint32_t hi) { return hi; }
    static __device__ __forceinline__ int get(const uint32_t* v, int j) { return (int)v[j]; }
};

template <class WS>
__device__ __forceinline__ void ld_vec(const WS* __restrict__ p, uint32_t (&v)[4]) {
#if AW_LOAD_CG
    uint4 t;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(t.x), "=r"(t.y), "=r"(t.z), "=r"(t.w) : "l"(p));
#else
    const uint4 t = *reinterpret_cast<const uint4*>(p);
#endif
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <class WS>
__device__ __forceinline__ void st_vec(WS* __restrict__ p, const uint32_t (&v)[4]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(v[0], v[1], v[2], v[3]);
}
// input row at diagonals [kc, kc+CPT): NULL outside the row's trimmed range [lo,hi]
template <class WS>
__device__ __forceinline__ void load_row(const WS* __restrict__ ws, int off, int lo, int hi, int kc, uint32_t (&v)[4]) {
    using T = VecT<WS>;
    constexpr int CPT = 4 * T::CPW;
    const int k1 = kc + CPT - 1;
    if (k1 < lo || kc > hi) {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = T::NULLW;
        return;
    }
    ld_vec<WS>(ws + off + kc, v);
    if (kc < lo || k1 > hi) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if constexpr (T::CPW == 2) {
                const int k = kc + 2 * i;
                const bool a = (k >= lo && k <= hi), b = (k + 1 >= lo && k + 1 <= hi);
                v[i] = (a ? (v[i] & 0xffffu) : (T::NULLW & 0xffffu)) | (b ? (v[i] & 0xffff0000u) : (T::NULLW & 0xffff0000u));
            } else {
                const int k = kc + i;
                if (k < lo || k > hi) v[i] = T::NULLW;
            }
        }
    }
}

// Called by the `gnw` warps of a group (gwarp = this warp's index in the group).
//   in_off  : lane i < 7 holds the element offset (k = 0) of input i (IN_*); the NULL row when absent
//   dsc     : warp-private shared memory, dsc[i] / dsc[8+i] = trimmed lo / hi of input i (empty: lo > hi)
//   ocoff   : shared memory, element offset (k = 0) of every output component (SlotMeta::coff)
//   [lo,hi] : computed range; [fast_lo,fast_hi] : diagonals every input reads back unmasked
//   [wlo,whi]: what this row must leave readable (computed chunks + NULL margin, clipped to the allocation)
template <int BITS, bool TWO, class WS>
__device__ __noinline__ void wf_cells_v(WS* __restrict__ ws, int in_off, const int* dsc, const int* ocoff, int lo, int hi, int fast_lo, int fast_hi,
                                        int wlo, int whi, const uint2* __restrict__ s_p2, const uint2* __restrict__ s_t2, int s_p0, int s_t0, int s_plen,
                                        int s_tlen, int k_end, int comp_end, int* red, int gwarp, int gnw, int pf_off, int* __restrict__ blk) {
    static_assert(BITS == 2, "the chunked path reads 2-bit sequences");
    using T = VecT<WS>;
    constexpr int CPT = 4 * T::CPW;
    constexpr bool SSEQ = sizeof(WS) == 2;  // int16 rows <=> the sequences are staged in shared memory (SEQ_SMEM)
    // ld16s() takes 2 * position + 4 * (shared-window byte address of the staged array)
    int cq_p = SSEQ ? 2 * s_p0 + 4 * (int)__cvta_generic_to_shared(s_p2) : 0;
    int cq_t = SSEQ ? 2 * s_t0 + 4 * (int)__cvta_generic_to_shared(s_t2) : 0;
    asm volatile("" : "+r"(cq_p), "+r"(cq_t));  // opaque: keeps ptxas from re-deriving them per cell (3 instructions instead of 1)
    const int ak_null = -(s_tlen + 8);
    // pf_off: lanes IN_MO1 / IN_MO2 hold the element offset of the M row those inputs will be two steps from now
    // (or -1): rows that old have usually left L2, so their lines are requested now (prefetch.global.L2)
    int pf1 = -1, pf2 = -1;
    if (AW_PREFETCH_STEPS > 0) {
        pf1 = __shfl_sync(0xffffffffu, pf_off, IN_MO1);
        if (TWO) pf2 = __shfl_sync(0xffffffffu, pf_off, IN_MO2);
    }
    constexpr int VW = 4;
    constexpr int SH = (CPT == 8) ? 3 : 2;
    constexpr int OWN = VBLOCK_CHUNKS;  // chunks owned per warp iteration (lanes 1..30)
    const int lane = threadIdx.x & 31;
    // Row addressing.  int16 rows: offsets are kept in BYTES and added to the workspace base as one unsigned 32-bit value
    // (IADD + 64-bit add = 3 instructions per access instead of 4 with sign extension and scaling; a CTA's int16 workspace is
    // below 4 GB).  int32 rows (Mb-scale pairs) keep element offsets and 64-bit pointer arithmetic.
    constexpr int OS = SSEQ ? 2 : 1;
    auto at = [&](int kc_, int o) -> WS* {
        if constexpr (SSEQ) return reinterpret_cast<WS*>(reinterpret_cast<char*>(ws) + (uint32_t)(((uint32_t)kc_ << 1) + (uint32_t)o));
        else return ws + kc_ + o;
    };
    const int o_mx = OS * __shfl_sync(0xffffffffu, in_off, IN_MX), o_mo1 = OS * __shfl_sync(0xffffffffu, in_off, IN_MO1);
    const int o_i1e = OS * __shfl_sync(0xffffffffu, in_off, IN_I1E), o_d1e = OS * __shfl_sync(0xffffffffu, in_off, IN_D1E);
    int o_mo2 = 0, o_i2e = 0, o_d2e = 0;
    if (TWO) {
        o_mo2 = OS * __shfl_sync(0xffffffffu, in_off, IN_MO2);
        o_i2e = OS * __shfl_sync(0xffffffffu, in_off, IN_I2E);
        o_d2e = OS * __shfl_sync(0xffffffffu, in_off, IN_D2E);
    }
    const int c_lo = lo >> SH, c_hi = hi >> SH;  // arithmetic shift = floor
    const int o_m = OS * ocoff[AW_COMP_M], o_i1 = OS * ocoff[AW_COMP_I1], o_i2 = OS * ocoff[AW_COMP_I2], o_d1 = OS * ocoff[AW_COMP_D1], o_d2 = OS * ocoff[AW_COMP_D2];
    int akM = INT_MIN, akAll = INT_MIN;
    bool oob = false;
    int bidx = gwarp;
    for (int cw = c_lo + gwarp * OWN; cw <= c_hi; cw += gnw * OWN, bidx += gnw) {
        int akM_b = INT_MIN, akAll_b = INT_MIN;
        // lanes past the right halo chunk (c_hi + 1) feed nobody: they shadow the halo lane (same addresses, one request per
        // warp) instead of taking a branch of their own with 20 NULL-initialised registers
        const int c = min(cw - 1 + lane, c_hi + 1);
        const int kc = c << SH;
        const bool own = (lane >= 1) && (lane <= OWN) && (cw - 1 + lane <= c_hi);
        const bool fast = (kc >= fast_lo) && (kc + CPT - 1 <= fast_hi);
        uint32_t mx[VW], tI1[VW], tD1[VW], tI2[VW], tD2[VW];
        {
            uint32_t mo[VW], ie[VW], de[VW], mo2[VW], ie2[VW], de2[VW];
            if (fast) {
                if (AW_PREFETCH_STEPS > 0) {
                    if (pf1 >= 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kc, OS * pf1)));
                    if (pf2 >= 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kc, OS * pf2)));
                }
                ld_vec<WS>(at(kc, o_mx), mx);
                ld_vec<WS>(at(kc, o_mo1), mo);
                ld_vec<WS>(at(kc, o_i1e), ie);
                ld_vec<WS>(at(kc, o_d1e), de);
                if (TWO) {
                    ld_vec<WS>(at(kc, o_mo2), mo2);
                    ld_vec<WS>(at(kc, o_i2e), ie2);
                    ld_vec<WS>(at(kc, o_d2e), de2);
                }
                // this warp's later iterations read the same rows further on: request those lines now so that only the first
                // iteration(s) of a step wait for L2 / HBM.  int16 rows (kb-scale pairs, a few iterations per step): the next
                // iteration, into L1.  int32 rows (Mb-scale pairs stream rows of megabytes through HBM, hundreds of iterations per
                // warp and step): AW_PF_DIST32 iterations ahead, into L2 (L1 is too small to hold that many lines per warp).
                constexpr int PFD = SSEQ ? 1 : AW_PF_DIST32;
                if (AW_PREFETCH_NEXT_ITER && cw + PFD * gnw * OWN <= c_hi) {
                    const int kn = kc + PFD * gnw * OWN * CPT;
                    if constexpr (SSEQ) {
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_mx)));
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_mo1)));
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_i1e)));
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_d1e)));
                        if (TWO) {
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_mo2)));
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_i2e)));
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(at(kn, o_d2e)));
                        }
                    } else {
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_mx)));
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_mo1)));
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_i1e)));
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_d1e)));
                        if (TWO) {
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_mo2)));
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_i2e)));
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(at(kn, o_d2e)));
                        }
                    }
                }
            } else {
                load_row<WS>(ws, o_mx / OS, dsc[IN_MX], dsc[8 + IN_MX], kc, mx);
                load_row<WS>(ws, o_mo1 / OS, dsc[IN_MO1], dsc[8 + IN_MO1], kc, mo);
                load_row<WS>(ws, o_i1e / OS, dsc[IN_I1E], dsc[8 + IN_I1E], kc, ie);
                load_row<WS>(ws, o_d1e / OS, dsc[IN_D1E], dsc[8 + IN_D1E], kc, de);
                if (TWO) {
                    load_row<WS>(ws, o_mo2 / OS, dsc[IN_MO2], dsc[8 + IN_MO2], kc, mo2);
                    load_row<WS>(ws, o_i2e / OS, dsc[IN_I2E], dsc[8 + IN_I2E], kc, ie2);
                    load_row<WS>(ws, o_d2e / OS, dsc[IN_D2E], dsc[8 + IN_D2E], kc, de2);
                }
            }
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                tI1[i] = T::vmax(mo[i], ie[i]);
                tD1[i] = T::vmax(mo[i], de[i]);
                if (TWO) {
                    tI2[i] = T::vmax(mo2[i], ie2[i]);
                    tD2[i] = T::vmax(mo2[i], de2[i]);
                }
            }
        }
        // neighbours: element kc-1 of the insertion sources, element kc+CPT of the deletion sources
        const uint32_t pI1 = __shfl_up_sync(0xffffffffu, tI1[VW - 1], 1);
        const uint32_t nD1 = __shfl_down_sync(0xffffffffu, tD1[0], 1);
        uint32_t pI2 = 0, nD2 = 0;
        if (TWO) {
            pI2 = __shfl_up_sync(0xffffffffu, tI2[VW - 1], 1);
            nD2 = __shfl_down_sync(0xffffffffu, tD2[0], 1);
        }
        if (own) {
            uint32_t vI1[VW], vD1[VW], vI2[VW], vD2[VW], vM[VW];
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                vI1[i] = T::inc(T::shl1(i == 0 ? pI1 : tI1[i - 1], tI1[i]));
                vD1[i] = T::shr1(tD1[i], i == VW - 1 ? nD1 : tD1[i + 1]);
                uint32_t m = T::mstep(mx[i], vI1[i]);
                if (TWO) {
                    vI2[i] = T::inc(T::shl1(i == 0 ? pI2 : tI2[i - 1], tI2[i]));
                    vD2[i] = T::shr1(tD2[i], i == VW - 1 ? nD2 : tD2[i + 1]);
                    m = T::vmax3(m, vI2[i], vD1[i]);
                    m = T::vmax(m, vD2[i]);
                } else {
                    m = T::vmax(m, vD1[i]);
                }
                vM[i] = m;
            }
            st_vec<WS>(at(kc, o_i1), vI1);
            st_vec<WS>(at(kc, o_d1), vD1);
            if (TWO) {
                st_vec<WS>(at(kc, o_i2), vI2);
                st_vec<WS>(at(kc, o_d2), vD2);
            }
            if (comp_end != AW_COMP_M && k_end >= kc && k_end < kc + CPT) {
                // select the VALUES, never a pointer to one of the register arrays: a pointer select forces all four
                // arrays into local memory on every iteration (16 STL per chunk, 2.4x the kernel's global stores in r01)
                const int j = k_end - kc;
                uint32_t src[VW];
#pragma unroll
                for (int i = 0; i < VW; ++i) {
                    uint32_t w = vI1[i];
                    if (comp_end == AW_COMP_D1) w = vD1[i];
                    if (TWO && comp_end == AW_COMP_I2) w = vI2[i];
                    if (TWO && comp_end == AW_COMP_D2) w = vD2[i];
                    src[i] = w;
                }
                int val = T::get(src, 0);
#pragma unroll
                for (int q = 1; q < CPT; ++q)
                    if (j == q) val = T::get(src, q);
                red[RED_END] = val;
            }
            // Per-cell scalar part, written with masks instead of conditionals: ptxas turns `valid ? .. : ..` blocks into
            // one branch region per cell (BSSY/BSYNC), which serialises the CPT independent chains; pure ALU code lets it
            // interleave them.
            int mm[CPT];
            unsigned more = 0;
            int oobm = 0;
            if constexpr (SSEQ) {
                // int16 rows + sequences in shared memory.  ~33 instructions per cell instead of 58:
                //  * the two sequence reads are not masked for invalid cells: the address is confined to the first 32 KB of the
                //    CTA's shared window (which holds the staged sequences, see the kernel prologue), so a null or out-of-bounds
                //    cell reads harmless garbage that the validity select discards;
                //  * nulls are <= NULL16 + drift, so 2*m - k of a null cell is far below every real antidiagonal and needs no mask
                //    (normalised to INT_MIN once per warp iteration);
                //  * "whole word matched and symbols remain" is folded into one running maximum, resolved per cell only when it fires.
                int zmax = 0;
#pragma unroll
                for (int j = 0; j < CPT; ++j) {
                    const int m = T::get(vM, j);
                    const int v = m - kc - j;
                    const int maxlen = min(s_plen - v, s_tlen - m);
                    const int w = m | v | maxlen;          // sign bit clear iff 0 <= h <= tlen and 0 <= v <= plen
                    const bool valid = w >= 0;
                    oobm |= ~m & w;                        // sign bit: a non-null offset outside the sequences
                    akAll_b = max(akAll_b, m + v);         // 2*off - k; m (pre-null) dominates every component at k
                    const uint32_t x = ld16s(2 * v + cq_p) ^ ld16s(2 * m + cq_t);
                    const int cnt = __clz(__brev(x)) >> 1;  // matching symbols = trailing zero pairs; 16 when the whole word matches
                    const int ml = valid ? maxlen : 0;
                    zmax = max(zmax, min(ml - 1, cnt));    // 16 iff the whole word matched and symbols remain
                    mm[j] = valid ? m + min(cnt, ml) : T::NULLV;
                }
                oobm >>= 31;
                if (zmax >= 16) {
#pragma unroll
                    for (int j = 0; j < CPT; ++j) more |= (unsigned)((mm[j] >= 0) && (mm[j] - T::get(vM, j) == 16)) << j;
                }
            } else {
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
                const int k = kc + j;
                const int m = T::get(vM, j);
                const int v = m - k;
                const int maxlen = min(s_plen - v, s_tlen - m);
                const int vmask = ~((m | v | maxlen) >> 31);  // all ones iff 0 <= h <= tlen and 0 <= v <= plen
                const int nonneg = ~(m >> 31);
                akAll_b = max(akAll_b, ((m + v) & nonneg) | (INT_MIN & ~nonneg));  // 2*off - k; m (pre-null) dominates every component at k
                oobm |= nonneg & ~vmask;                                           // a non-null offset outside the sequences
                // first round of the extension (16 symbols); invalid cells compare position 0
                const uint32_t x = load16(s_p2, s_p0 + (v & vmask)) ^ load16(s_t2, s_t0 + (m & vmask));
                const int cnt = __popc((x - 1u) & ~x) >> 1;  // matching symbols = trailing zero pairs; 16 when the whole word matches
                const int ext = min(cnt, maxlen);
                mm[j] = ((m + ext) & vmask) | (T::NULLV & ~vmask);
                more |= (unsigned)((cnt >> 4) & ((16 - maxlen) >> 31) & vmask & 1) << j;  // whole word matched and symbols remain
            }
            }
            oob = oob || (oobm != 0);
            while (more) {  // long match runs: continue word by word, one cell at a time (kept small: instruction-cache footprint)
                const int j = __ffs(more) - 1;
                more &= more - 1;
                int h = mm[0];
#pragma unroll
                for (int q = 1; q < CPT; ++q)
                    if (j == q) h = mm[q];
                const int v = h - (kc + j);
                h += lcp2(s_p2, s_t2, s_p0 + v, s_t0 + h, min(s_plen - v, s_tlen - h));
#pragma unroll
                for (int q = 0; q < CPT; ++q)
                    if (j == q) mm[q] = h;
            }
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
                if constexpr (SSEQ) {
                    akM_b = max(akM_b, mm[j] + (mm[j] - kc - j));  // a null cell lands far below every real antidiagonal
                } else {
                    const int nonneg = ~(mm[j] >> 31);
                    akM_b = max(akM_b, ((2 * mm[j] - (kc + j)) & nonneg) | (INT_MIN & ~nonneg));
                }
            }
            if (comp_end == AW_COMP_M && k_end >= kc && k_end < kc + CPT) {
                const int j = k_end - kc;
                int val = mm[0];
#pragma unroll
                for (int q = 1; q < CPT; ++q)
                    if (j == q) val = mm[q];
                red[RED_END] = val;
            }
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                if constexpr (T::CPW == 2) vM[i] = __byte_perm((uint32_t)mm[2 * i], (uint32_t)mm[2 * i + 1], 0x5410);
                else vM[i] = (uint32_t)mm[i];
            }
            st_vec<WS>(at(kc, o_m), vM);
        }
        if (AW_L1_PREFETCH && own) {  // the next step reads the same diagonals of these rows: pull their lines into L1 now
#pragma unroll
            for (int i = 0; i < (TWO ? 7 : 4); ++i) {
                const int o = dsc[24 + i];
                if (o >= 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(ws + kc + o));
            }
        }
        if constexpr (SSEQ) {
            // 2*off - k of a (possibly drifted) null is below -(tlen + 8): NULL16 + drift <= -32000 + plen + tlen + 100 and
            // plan_launch only selects int16 rows when 3 * (plen + tlen) < 63000
            if (akM_b < ak_null) akM_b = INT_MIN;
            if (akAll_b < ak_null) akAll_b = INT_MIN;
        }
        if (blk != nullptr) {
            akM_b = __reduce_max_sync(0xffffffffu, akM_b);
            akAll_b = __reduce_max_sync(0xffffffffu, akAll_b);
            if (lane == 0) *reinterpret_cast<int2*>(blk + 2 * bidx) = make_int2(akM_b, akAll_b);
        }
        akM = max(akM, akM_b);
        akAll = max(akAll, akAll_b);
    }
    // NULL margin either side of the computed chunks (clipped to [wlo,whi]), by the group's last warp
    if (gwarp == gnw - 1) {
        constexpr int MG = VMARGIN / CPT;
        constexpr int NCOMP = TWO ? 5 : 3;
        uint32_t nullv[VW];
#pragma unroll
        for (int i = 0; i < VW; ++i) nullv[i] = T::NULLW;
        for (int i = lane; i < 2 * MG * NCOMP; i += 32) {
            const int ci = i / (2 * MG), j = i - ci * (2 * MG);
            const int comp = TWO ? ci : (ci == 2 ? AW_COMP_D1 : ci);
            const int c = (j < MG) ? (c_lo - MG + j) : (c_hi + 1 + (j - MG));
            const int kc = c << SH;
            if (kc >= wlo && kc + CPT - 1 <= whi) st_vec<WS>(ws + ocoff[comp] + kc, nullv);
        }
    }
    akM = __reduce_max_sync(0xffffffffu, akM);
    akAll = __reduce_max_sync(0xffffffffu, akAll);
    oob = __any_sync(0xffffffffu, oob);
    if (lane == 0) {
        if (akM != INT_MIN) atomicMax(&red[RED_AKM], akM);
        if (akAll != INT_MIN) atomicMax(&red[RED_AKALL], akAll);
        if (oob) red[RED_OOB] = 1;
    }
}

//@region wf_finish
// after the barrier: trimmed ranges (wavefront_compute_trim_ends) from the reductions
template <bool TWO>
__device__ __forceinline__ void wf_finish(const int* red, int lo, int hi, StepOut& so) {
    const bool narrow = (hi - lo) < 2 * EDGE_ZONE;
    so.ambiguous = false;
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        if (!TWO && (c == AW_COMP_I2 || c == AW_COMP_D2)) {
            so.lo[c] = 1;
            so.hi[c] = 0;
            continue;
        }
        const int h = red[RED_HI + c], l = red[RED_LO + c];
        if (h == INT_MIN) {  // nothing in bounds (among the tracked cells)
            so.lo[c] = lo;
            so.hi[c] = lo - 1;
            if (!narrow) so.ambiguous = true;
        } else {
            so.lo[c] = -l;
            so.hi[c] = h;
            // exact only if each end was found inside its tracked zone
            if (!narrow && ((-l) - lo >= EDGE_ZONE || hi - h >= EDGE_ZONE)) so.ambiguous = true;
        }
    }
    so.akM = red[RED_AKM];
    so.akAll = red[RED_AKALL];
    so.endval = red[RED_END];
}

//@region wf_rescan
// exact trim of every component by re-reading the stored wavefront (rare slow path)
// `tt` / `tn`: this thread's index in / the size of the team that owns the row -- the whole CTA, or one warp (wm) when the
// warps of a CTA work on different base cases at the same time
template <int NT, bool TWO, class WS>
__device__ __noinline__ void wf_rescan(const WS* __restrict__ ws, const int (&out)[5], int lo, int hi, int plen_, int tlen_, int* red, StepOut& so, int tt, int tn,
                                       bool wm) {
    const unsigned tlen = (unsigned)tlen_, plen = (unsigned)plen_;
    auto tsync = [&]() {
        if (wm) __syncwarp();
        else cta_sync<NT>();
    };
    auto tmax = [&](int idx, int v) {
        v = __reduce_max_sync(0xffffffffu, v);
        if ((threadIdx.x & 31) == 0 && v != INT_MIN) atomicMax(&red[idx], v);
    };
    tsync();
    if (tt < NRED) red[tt] = INT_MIN;
    tsync();
    int vhi[5], vlo[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) vhi[c] = vlo[c] = INT_MIN;
    for (int k = lo + tt; k <= hi; k += tn) {
#pragma unroll
        for (int c = 0; c < 5; ++c) {
            if (!TWO && (c == AW_COMP_I2 || c == AW_COMP_D2)) continue;
            const int v = ws[out[c] + k];
            if ((unsigned)v <= tlen && (unsigned)(v - k) <= plen) {
                if (vlo[c] == INT_MIN) vlo[c] = -k;
                vhi[c] = k;
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        if (!TWO && (c == AW_COMP_I2 || c == AW_COMP_D2)) continue;
        tmax(RED_HI + c, vhi[c]);
        tmax(RED_LO + c, vlo[c]);
    }
    tsync();
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        if (!TWO && (c == AW_COMP_I2 || c == AW_COMP_D2)) continue;
        const int h = red[RED_HI + c], l = red[RED_LO + c];
        if (h == INT_MIN) {
            so.lo[c] = lo;
            so.hi[c] = lo - 1;
        } else {
            so.lo[c] = -l;
            so.hi[c] = h;
        }
    }
    so.ambiguous = false;
    tsync();
    if (tt < NRED) red[tt] = INT_MIN;
    tsync();
}

//@region misc helpers
__device__ __forceinline__ bool end_reached(const StepOut& so, int comp_end, int k_end, int tlen) {
    const int l = (comp_end == AW_COMP_M) ? so.lo[0] : (comp_end == AW_COMP_I1) ? so.lo[1] : (comp_end == AW_COMP_I2) ? so.lo[2] : (comp_end == AW_COMP_D1) ? so.lo[3] : so.lo[4];
    const int h = (comp_end == AW_COMP_M) ? so.hi[0] : (comp_end == AW_COMP_I1) ? so.hi[1] : (comp_end == AW_COMP_I2) ? so.hi[2] : (comp_end == AW_COMP_D1) ? so.hi[3] : so.hi[4];
    return l <= k_end && k_end <= h && so.endval >= tlen;
}

// number of decimal digits of v
__device__ __forceinline__ int ndigits(unsigned long long v) {
    int n = 1;
    while (v >= 10) {
        v /= 10;
        ++n;
    }
    return n;
}
__device__ __forceinline__ char* put_u64(char* p, unsigned long long v) {
    const int n = ndigits(v);
    for (int i = n - 1; i >= 0; --i) {
        p[i] = (char)('0' + (int)(v % 10));
        v /= 10;
    }
    return p + n;
}

// {:.6} of matches/alignment_length (src/lib.rs:83-87,108): IEEE division, then exact
// round-half-even of x * 10^6 (what Rust's flt2dec and C's printf both produce)
__device__ __forceinline__ unsigned identity_micro(unsigned long long matches, unsigned long long alnlen) {
    if (alnlen == 0 || matches == 0) return 0;
    const double x = (double)matches / (double)alnlen;
    const unsigned long long bits = (unsigned long long)__double_as_longlong(x);
    const int e = (int)((bits >> 52) & 0x7ff);
    const unsigned long long mant = (bits & ((1ull << 52) - 1)) | (1ull << 52);
    const int shift = 1075 - e;  // x = mant * 2^-shift, shift >= 52 because x <= 1
    const unsigned __int128 P = (unsigned __int128)mant * 1000000ull;
    if (shift >= 120) return 0;
    const unsigned __int128 one = (unsigned __int128)1 << shift;
    unsigned long long q = (unsigned long long)(P >> shift);
    const unsigned __int128 rem = P & (one - 1), half = one >> 1;
    if (rem > half || (rem == half && (q & 1))) ++q;
    return (unsigned)q;
}

template <int NT>
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long* sbuf, unsigned long long* total) {
    // sbuf: NT entries of shared memory
    const int tid = threadIdx.x;
    cta_sync<NT>();
    sbuf[tid] = v;
    cta_sync<NT>();
    for (int d = 1; d < NT; d <<= 1) {
        unsigned long long t = (tid >= d) ? sbuf[tid - d] : 0;
        cta_sync<NT>();
        sbuf[tid] += t;
        cta_sync<NT>();
    }
    *total = sbuf[NT - 1];
    return sbuf[tid] - v;
}

// ------------------------------------------------------------------------------------------
// The kernel
// ------------------------------------------------------------------------------------------
//@region kernel prologue + pair setup
// leaving the DFS over sub-problems on failure.  In a cluster kernel a CTA that fails on its own (CTA 0 inside a solo
// sub-problem, a backtrace or the CIGAR assembly) must keep popping sub-problems -- it drops the solo ones and meets the other
// CTAs at the status exchange of the next cluster-wide one -- or the cluster would dead-lock on its next barrier.
#define AW_DFS_FAIL            \
    {                          \
        if (CL > 1 && solo) continue; \
        break;                 \
    }
#define AW_DFS_FAIL_CTA0       \
    {                          \
        if (CL > 1) continue;  \
        break;                 \
    }
// CL > 1 (Mb-scale pairs, int32 chunked path only): one pair per thread-block CLUSTER of CL CTAs.  Every CTA runs the same
// driver on replicated shared state (ring metadata, recursion stack, candidate lists); the cells of a wavefront step are split
// over the warps of the whole cluster, one barrier.cluster per step replaces the CTA barrier, and each CTA then folds the
// other CTAs' per-step reductions (trim ends, antidiagonal maxima, end cell, flags) into its own copy through distributed
// shared memory -- so all CTAs keep taking identical decisions.  Sub-problems shorter than P.solo_len (the deep, narrow levels
// of the biWFA recursion, where a cluster barrier per step would dominate) are left to CTA 0 alone, which also does every
// backtrace and the CIGAR / PAF emission.  The wavefront rings stay in global memory (L2 / HBM): at Mb scale one ring row is
// megabytes.
// SCORE (aw_score_kernel): the optimal penalty of each pair only.  The top-level breakpoint's score is the pair's score, so
// nothing below it runs; a top level that is a base case runs its wavefronts to the end cell and skips the backtrace.  No
// CIGAR, no text and no bytes are produced.
template <int NT, int BITS, bool TWO, class WS, int CL, bool SCORE>
__device__ __forceinline__ void align_driver(const KParams& P) {
    static_assert(CL == 1 || (NT >= 64 && BITS == 2 && sizeof(WS) == 4), "cluster kernels exist for the int32 chunked path only");
    constexpr int NCOMP = TWO ? 5 : 3;
    const unsigned crank = (CL > 1) ? cluster_ctarank() : 0u;  // this CTA's rank in its cluster
    const unsigned cid = (CL > 1) ? blockIdx.x / CL : blockIdx.x;  // workspace / work-queue slot: one per cluster
    constexpr bool VEC = (NT >= 64) && (BITS == 2);        // chunked (16 bytes of cells per thread) wavefront loop
    constexpr bool SEQ_SMEM = VEC && sizeof(WS) == 2;      // int16-sized pairs: sequences staged in shared memory
    constexpr int CPT = 16 / sizeof(WS);                   // diagonals per thread in that loop: 8 int16 or 4 int32
    constexpr int RALIGN = VEC ? CPT : 1;                  // row alignment (elements)
    extern __shared__ unsigned long long smem_raw[];
    const int scope = P.pen.scope;
    const int ring_n = scope + 1;  // one spare slot: the reverse step is computed speculatively
    SlotMeta* ring_meta = reinterpret_cast<SlotMeta*>(smem_raw);                                     // [2][ring_n]
    int* cand = reinterpret_cast<int*>(ring_meta + ((AW_LEAFPAR && VEC && CL == 1) ? 2 + NT / 32 : 2) * ring_n);  // [scope*5] candidate tests (after the SlotMeta rings)
    int* hitk = cand + scope * 5;                                                                    // [scope*5] first hit per candidate
    unsigned long long* scanbuf = reinterpret_cast<unsigned long long*>(hitk + scope * 5);  // [NT]; 8-byte aligned: sizeof(SlotMeta)*2*ring_n + 40*scope
    int* cklo = reinterpret_cast<int*>(scanbuf + NT);                                      // [scope*5] first diagonal of a candidate's scan range
    int* ckhi = cklo + scope * 5;                                                          // [scope*5] last diagonal
    // warp-parallel leaves (LEAFPAR): the base cases (score_remaining <= 250) of a pair are independent of each other, narrow
    // (<= 501 diagonals) and cost one CTA barrier per score when the whole CTA works on one of them -- with three of four
    // warps idle.  They are collected in DFS order and run NW at a time, ONE WARP EACH (chunked engine with a team of one
    // warp, __syncwarp instead of the CTA barrier, own slice of the history arena), then appended to the CIGAR in order.
    constexpr bool LEAFPAR = AW_LEAFPAR && VEC && CL == 1;
    constexpr int NW = NT / 32;
    constexpr int RM_N = LEAFPAR ? 2 + NW : 2;  // SlotMeta rings: forward, reverse (row 0 doubles as the cooperative base case) + one per warp
    __shared__ int red[RM_N][3][NRED];
    __shared__ int s_rescan_w[LEAFPAR ? NW : 1][NRED];
    __shared__ SubProblem s_leaf[LEAFPAR ? NW : 1];
    __shared__ unsigned s_leaf_n[LEAFPAR ? NW : 1];                 // per leaf: runs, status, score, work counters
    __shared__ int s_leaf_st[LEAFPAR ? NW : 1], s_leaf_score[LEAFPAR ? NW : 1];
    __shared__ unsigned long long s_leaf_cells[LEAFPAR ? NW : 1];
    __shared__ unsigned s_leaf_steps[LEAFPAR ? NW : 1];
    __shared__ SubProblem stack[MAX_STACK];
    __shared__ unsigned s_next;
    __shared__ unsigned s_nruns;
    __shared__ int s_rescan[NRED];   // wf_rescan's own reduction buffer (the step's buffer may still be read by other CTAs of a cluster)
    __shared__ int s_cl_status;      // cluster kernels: this CTA's status, exchanged at the start of every cluster-wide sub-problem
    __shared__ int s_ncand, s_nact, s_ov[4];  // s_ov: thresholds for M / other components, first and last diagonal of any candidate
    constexpr int ACT_MAX = 256;
    __shared__ int s_act[ACT_MAX];            // blocks of aligner 0's wavefront that can hold a meeting point
    __shared__ unsigned long long s_acc[8];
    __shared__ unsigned long long s_text_off, s_bytes_off;
    __shared__ uint32_t s_seq[VEC ? 1 : SEQ_SMEM_WORDS];
    __shared__ uint2 s_seq2[SEQ_SMEM ? SEQ2_ENTRIES : 1];  // int16 path: pattern, text, reversed pattern, reversed text as overlapping word pairs
    __shared__ __align__(16) int s_desc[VEC ? NT / 32 : 1][32];  // ... and [24..30] the rows the next step will read (L1 prefetch)  // int16 path, per warp: trimmed lo[8] / hi[8] of the step's inputs, offsets[5] of its outputs

    const int tid = threadIdx.x;
    const AwPen pen = P.pen;
    int* const ws_i = P.ws + (size_t)cid * P.ws_ints_per_cta;
    WS* const ws = reinterpret_cast<WS*>(ws_i);  // all wavefront offsets below are in WS elements
    const int W = P.W;
    // int16 path: after the rings come one all-NULL row and the compact I/D rings (per direction e1+1 rows for each of
    // I1/D1 and e2+1 rows for each of I2/D2): while the two wavefronts are far apart nobody reads an I/D row older than
    // its extension distance, so those rows are overwritten while still in L2 instead of streaming through HBM
    const int null_base = 2 * ring_n * NCOMP * W;
    const int cmp_n1 = P.pen.e1 + 1, cmp_n2 = TWO ? P.pen.e2 + 1 : 0;
    const int cmp_rows = 2 * cmp_n1 + 2 * cmp_n2;               // per direction
    const int cmp_base = null_base + W;
    const int hist_base = VEC ? cmp_base + 2 * cmp_rows * W : null_base;  // history arena starts after the rings
    constexpr int VBW = VBLOCK_CHUNKS * CPT;  // diagonals per block of the per-block maxima
    int* const blk_cta = VEC ? P.ws_blk + (size_t)cid * 2 * ring_n * P.blk_cap * 2 : nullptr;
    auto blk_of = [&](int d, int slot) -> int* { return blk_cta + (size_t)(d * ring_n + slot) * P.blk_cap * 2; };
    int* const hist_meta = P.ws_hist_meta + (size_t)cid * (size_t)P.hist_max_scores * HIST_META_INTS;
    uint32_t* const pair_runs = P.ws_runs + (size_t)cid * 2 * P.runs_cap;
    uint32_t* const leaf_runs = pair_runs + P.runs_cap;

    if constexpr (SEQ_SMEM) {
        // ld16s() confines its addresses to the first SEQ2_WINDOW bytes of the shared window: the staged sequences must lie
        // inside (launch_align pads the dynamic part so that the CTA owns at least that much)
        if (tid == 0 && __cvta_generic_to_shared(s_seq2) + sizeof(s_seq2) > SEQ2_WINDOW) __trap();
    }
    for (int i = tid; i < RM_N * 3 * NRED; i += NT) (&red[0][0][0])[i] = INT_MIN;
    if (tid < NRED) s_rescan[tid] = INT_MIN;
    if (LEAFPAR && (tid & 31) < NRED) s_rescan_w[tid >> 5][tid & 31] = INT_MIN;
    if constexpr (VEC) {
        const uint4 nv = make_uint4(VecT<WS>::NULLW, VecT<WS>::NULLW, VecT<WS>::NULLW, VecT<WS>::NULLW);
        for (int i = tid * CPT; i < W; i += NT * CPT) *reinterpret_cast<uint4*>(ws + null_base + i) = nv;
    }
    int red_i = 0;  // rotating reduction buffer index (uniform)
    cta_sync<NT>();

    auto comp_idx = [](int c) -> int { return TWO ? c : (c == AW_COMP_D1 ? 2 : c); };
    // team context of the step lambdas below: the whole CTA, or -- while a batch of leaves is being aligned -- one warp
    bool wm = false;                 // warp mode
    int t_tid = tid;                 // thread index inside the team
    int t_d = 0;                     // warp mode: this warp's row of red[] (its SlotMeta ring is ring_meta[t_d * ring_n ...])
    int hb_cur = hist_base;          // history arena of the team: first element, capacity, metadata rows, leaf run buffer
    long long hcap_cur = P.hist_ints;
    int* hmeta_cur = hist_meta;
    int hscores_cur = P.hist_max_scores;
    uint32_t* lruns_cur = leaf_runs;
    unsigned long long lcap_cur = P.runs_cap;
    auto team_sync = [&]() {
        if (wm) __syncwarp();
        else cta_sync<NT>();
    };
    auto rotate_red = [&]() {
        // recycle the buffers used two steps ago (everybody finished reading them before the last barrier)
        const int nxt = (red_i + 2) % 3;
        if (wm) {
            if (t_tid < NRED) red[t_d][nxt][t_tid] = INT_MIN;
        } else if (tid < NRED) {
            red[0][nxt][tid] = INT_MIN;
            red[1][nxt][tid] = INT_MIN;
        }
        red_i = (red_i + 1) % 3;
    };

    // one wavefront-step barrier: CTA-wide, or cluster-wide followed by the fold of every CTA's reductions into this CTA's copy
    // (max is idempotent, so a peer that reads a slot this CTA has already folded still ends with the same value; wf_rescan
    // and rotate_red never touch the buffer of the current step, which peers may still be reading)
    auto step_sync = [&](bool solo) {
        if constexpr (CL > 1) {
            if (!solo) {
                cluster_sync_all();
                if (tid < 2 * NRED) {
                    int* slot = &red[tid / NRED][red_i][tid % NRED];
                    int v = *slot;
#pragma unroll
                    for (unsigned r = 0; r < (unsigned)CL; ++r)
                        if (r != crank) v = max(v, ld_dsmem_int(slot, r));
                    *slot = v;
                }
            }
        }
        cta_sync<NT>();
    };
    for (;;) {
        if (tid == 0 && crank == 0) s_next = atomicAdd(P.next_pair, 1u);
        unsigned work_i;
        if constexpr (CL > 1) {
            cluster_sync_all();
            work_i = (unsigned)ld_dsmem_int(reinterpret_cast<const int*>(&s_next), 0);
            cluster_sync_all();  // CTA 0 may overwrite s_next only after everybody has read it
        } else {
            cta_sync<NT>();
            work_i = s_next;
            cta_sync<NT>();
        }
        if (work_i >= P.npairs) break;
        const unsigned pair_i = P.order ? P.order[work_i] : work_i;
        const aw_pair pr = P.pairs[pair_i];
        const unsigned is_rev = P.is_reverse ? P.is_reverse[pair_i] : 0u;
        if (is_rev > 1u) {
            // --wfa-orientation: one of the two orientation alignments ran out of workspace, the strand is undecided.
            // Nothing is aligned here; the host decides the strand with a larger workspace and re-runs the pair.
            if (tid == 0 && crank == 0) {
                AwPairOut o;
                memset(&o, 0, sizeof(o));
                o.status = AW_EWORKSPACE;
                o.score = INT_MAX;
                o.is_reverse = is_rev;
                P.out[pair_i] = o;
            }
            continue;
        }
        const AwSlot qs = P.slots[2 * pr.query_idx + is_rev];
        const AwSlot ts = P.slots[2 * pr.target_idx];
        const uint32_t* pw = (BITS == 2) ? P.packed + qs.packed_off : reinterpret_cast<const uint32_t*>(P.ascii + qs.ascii_off);
        const uint32_t* tw = (BITS == 2) ? P.packed + ts.packed_off : reinterpret_cast<const uint32_t*>(P.ascii + ts.ascii_off);
        const int PLEN = (int)qs.len, TLEN = (int)ts.len;
        const uint2 *pf2 = s_seq2, *tf2 = s_seq2, *pr2 = s_seq2, *tr2 = s_seq2;
        bool seq_fits = true;
        if constexpr (VEC) {
            // entry i of a staged sequence = packed words (i, i+1); the reversed copy R[i] = S[len-1-i] is built from
            // the same global words (bit-reverse a 16-symbol window, then swap the two bits of every symbol back)
            const int np = PLEN / 16 + 2, ntt = TLEN / 16 + 2;
            seq_fits = SEQ_SMEM ? (2 * (np + ntt) <= SEQ2_ENTRIES) : ((unsigned long long)2 * (np + ntt) <= P.seq2_cap);
            // longer pairs keep the four arrays in a per-CTA global scratch (L1/L2-cached 8-byte loads)
            uint2* s_pf = SEQ_SMEM ? s_seq2 : P.ws_seq2 + (size_t)cid * P.seq2_cap;
            uint2* s_tf = s_pf + np;
            uint2* s_pr = s_tf + ntt;
            uint2* s_tr = s_pr + np;
            auto rev16 = [](const uint32_t* w, int len, int j) -> uint32_t {  // symbols 16j .. 16j+15 of the reversed sequence
                const int a = len - 16 - 16 * j;                                 // first original symbol of the window (may be < 0: guard words)
                const int idx = a >> 4;                                          // floor
                const uint32_t x = __funnelshift_r(w[idx], w[idx + 1], (a & 15) * 2);
                const uint32_t b = __brev(x);
                return ((b >> 1) & 0x55555555u) | ((b & 0x55555555u) << 1);
            };
            if (seq_fits) {
                for (int i = tid; i < np; i += NT) {
                    s_pf[i] = make_uint2(pw[i], pw[i + 1]);
                    s_pr[i] = make_uint2(rev16(pw, PLEN, i), rev16(pw, PLEN, i + 1));
                }
                for (int i = tid; i < ntt; i += NT) {
                    s_tf[i] = make_uint2(tw[i], tw[i + 1]);
                    s_tr[i] = make_uint2(rev16(tw, TLEN, i), rev16(tw, TLEN, i + 1));
                }
            }
            pf2 = s_pf;
            tf2 = s_tf;
            pr2 = s_pr;
            tr2 = s_tr;
        } else {
            // stage both sequences (with 2 guard words either side) in shared memory when they fit
            constexpr int SPW = 32 / BITS;
            const int pwords = PLEN / SPW + 1, twords = TLEN / SPW + 1;
            if (pwords + twords + 8 <= SEQ_SMEM_WORDS) {
                for (int i = tid; i < pwords + 4; i += NT) s_seq[i] = pw[i - 2];
                for (int i = tid; i < twords + 4; i += NT) s_seq[pwords + 4 + i] = tw[i - 2];
                pw = s_seq + 2;
                tw = s_seq + pwords + 4 + 2;
            }
        }
        // diagonal k lives at index k + koff.  In-bounds diagonals span [-PLEN, TLEN]: the positive side never needs more than
        // TLEN + 1, so a row wide enough for both sides gives the rest to the negative side (a query much longer than its target
        // drifts far below diagonal -W/2); a narrower row is split evenly.
        const int koff = (min(PLEN + 1, max(W / 2, W - TLEN - 1 - RALIGN)) + RALIGN - 1) & ~(RALIGN - 1);
        const int kmin_alloc = -koff, kmax_alloc = W - 1 - koff;

        int status = seq_fits ? ST_OK : ST_FAIL_WORKSPACE;
        unsigned long long cyc[6] = {0, 0, 0, 0, 0, 0};
        long long tmark = AW_CYCLE_COUNTERS ? clock64() : 0;
        auto lap = [&](int i) {
            if (AW_CYCLE_COUNTERS) {
                const long long t = clock64();
                cyc[i] += (unsigned long long)(t - tmark);
                tmark = t;
            }
        };
        unsigned long long w_cells = 0;
        unsigned w_steps = 0, w_bps = 0, w_base = 0, w_maxbase = 0;
        if (tid == 0) s_nruns = 0;
        int sp_n = 0;
        int sc_pen = 0;  // SCORE: the pair's wavefront penalty (under pen.x, pen.o1, ... -- shifted when match_score < 0)
        {
            // wavefront_bialign: short sequences go straight to the base case
            SubProblem top = {0, PLEN, 0, TLEN, AW_COMP_M, AW_COMP_M, (max(PLEN, TLEN) <= AW_BIALIGN_FALLBACK_MIN_LENGTH) ? 0 : INT_MAX};
            stack[sp_n++] = top;
        }
        cta_sync<NT>();

        // appends a run to the pair's CIGAR (thread 0 only), merging with the previous run
        auto emit_run = [&](unsigned op, unsigned len) {
            if (len == 0) return;
            unsigned n = s_nruns;
            if (n > 0 && (pair_runs[n - 1] & 3u) == op) {
                pair_runs[n - 1] += len << 2;
            } else if (n < P.runs_cap) {
                pair_runs[n] = (len << 2) | op;
                s_nruns = n + 1;
            }
        };
        auto set_empty = [&](SlotMeta& m) {
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                m.lo[c] = 1;
                m.hi[c] = 0;
            }
            m.akM = m.akAll = INT_MIN;
            m.off = 0;
            m.cstride = 0;
            m.wlo = 1;
            m.whi = 0;
        };
        auto store_meta = [&](SlotMeta& m, const StepOut& so) {
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                m.lo[c] = so.lo[c];
                m.hi[c] = so.hi[c];
            }
            m.akM = so.akM;
            m.akAll = so.akAll;
        };
        // wavefront_compute_limits_input over the non-empty inputs
        auto limits = [&](const In (&in)[7], int& lo, int& hi) {
            lo = INT_MAX;
            hi = INT_MIN;
            auto lim = [&](const In& w, int dl, int dh) {
                if (w.lo <= w.hi) {
                    lo = min(lo, w.lo + dl);
                    hi = max(hi, w.hi + dh);
                }
            };
            lim(in[IN_MX], 0, 0);
            lim(in[IN_MO1], -1, 1);
            lim(in[IN_I1E], 1, 1);
            lim(in[IN_D1E], -1, -1);
            if (TWO) {
                lim(in[IN_MO2], -1, 1);
                lim(in[IN_I2E], 1, 1);
                lim(in[IN_D2E], -1, -1);
            }
        };

//@region v_launch (plan + cells)
        // ================= int16 path: one wavefront step =================
        // v_launch: the warps of a group plan wavefront `s` of direction d (inputs, ranges, placement) and
        // compute it; nothing here needs a barrier.  v_finish (every thread, after the barrier) publishes
        // the step's results.  mbase selects the SlotMeta ring (d * ring_n; 0 in the base case).
        struct VRange {
            int lo, hi;   // computed range (null step iff lo > hi); valid in the planning warps only
            int width;    // history mode: allocated elements per component
        };
        long long hist_used = 0;  // history arena bump pointer (base case)
        // gwarp / gnw: this warp's index among / the number of warps that share the step (CTA-local, or cluster-wide when the
        // sub-problem runs on the whole cluster); lwarp: its index among this CTA's warps of the step -- the first of them keeps
        // the CTA's own copy of the ring metadata and of the step's range up to date
        auto v_launch = [&](int d, int mbase, int s, int slot, int gwarp, int gnw, int lwarp, bool hist, bool full, const SeqView& sv, int k_end, int comp_end) -> VRange {
            constexpr int SH = (CPT == 8) ? 3 : 2;
            constexpr int MG = VMARGIN / CPT;
            const int lane = tid & 31;
            int* r = red[d][red_i];
            int* dsc = s_desc[VEC ? (tid >> 5) : 0];
            SlotMeta& mt = ring_meta[mbase + slot];
            // lane i < 7 describes input i
            int comp = AW_COMP_M, back = pen.x;
            if (lane == IN_MO1) back = pen.o1 + pen.e1;
            else if (lane == IN_I1E) { comp = AW_COMP_I1; back = pen.e1; }
            else if (lane == IN_D1E) { comp = AW_COMP_D1; back = pen.e1; }
            else if (lane == IN_MO2) back = pen.o2 + pen.e2;
            else if (lane == IN_I2E) { comp = AW_COMP_I2; back = pen.e2; }
            else if (lane == IN_D2E) { comp = AW_COMP_D2; back = pen.e2; }
            int ilo = VBIG, ihi = -VBIG, ioff = null_base + koff, iwlo = -VBIG, iwhi = VBIG, pf_off = -1;
            if (AW_PREFETCH_STEPS > 0 && (lane == IN_MO1 || (TWO && lane == IN_MO2)) && back > AW_PREFETCH_STEPS && s + AW_PREFETCH_STEPS - back >= 0) {
                int sl = slot + AW_PREFETCH_STEPS - back;
                if (sl < 0) sl += ring_n;
                const SlotMeta& m = ring_meta[mbase + sl];
                if (m.lo[AW_COMP_M] <= m.hi[AW_COMP_M]) pf_off = m.coff[AW_COMP_M];
            }
            if (lane < (TWO ? 7 : 4) && s - back >= 0) {
                int sl = slot - back;
                if (sl < 0) sl += ring_n;
                const SlotMeta& m = ring_meta[mbase + sl];
                const int l = m.lo[comp], h = m.hi[comp];
                if (l <= h) {
                    ilo = l;
                    ihi = h;
                    ioff = m.coff[comp];
                    iwlo = m.wlo;
                    iwhi = m.whi;
                }
            }
            __syncwarp();
            if (lane < 8) {
                dsc[lane] = ilo;
                dsc[8 + lane] = ihi;
            }
            const int fast_lo = max(__reduce_max_sync(0xffffffffu, iwlo), kmin_alloc);
            const int fast_hi = min(__reduce_min_sync(0xffffffffu, iwhi), kmax_alloc);
            __syncwarp();
            const int4 l0 = *reinterpret_cast<const int4*>(dsc), l1 = *reinterpret_cast<const int4*>(dsc + 4);
            const int4 h0 = *reinterpret_cast<const int4*>(dsc + 8), h1 = *reinterpret_cast<const int4*>(dsc + 12);
            // trimmed ranges of the outputs when the row holds no out-of-bounds cell (see wf_cells_v)
            const int i1lo = min(l0.y, l0.z) + 1, i1hi = max(h0.y, h0.z) + 1;
            const int d1lo = min(l0.y, l0.w) - 1, d1hi = max(h0.y, h0.w) - 1;
            const int i2lo = min(l1.x, l1.y) + 1, i2hi = max(h1.x, h1.y) + 1;
            const int d2lo = min(l1.x, l1.z) - 1, d2hi = max(h1.x, h1.z) - 1;
            const int mlo = min(min(l0.x, min(i1lo, i2lo)), min(d1lo, d2lo)), mhi = max(max(h0.x, max(i1hi, i2hi)), max(d1hi, d2hi));
            VRange rg;
            rg.lo = mlo;  // = wavefront_compute_limits_input over the non-empty inputs
            rg.hi = mhi;
            rg.width = 0;
            const bool lead = (lwarp == 0);
            if (status != ST_OK) return rg;
            if (rg.lo > rg.hi) {  // null step
                if (lead) {
                    if (lane < 5) {
                        mt.lo[lane] = 1;
                        mt.hi[lane] = 0;
                    }
                    if (lane == 5) {
                        mt.akM = mt.akAll = INT_MIN;
                        mt.off = mt.cstride = 0;
                        mt.wlo = 1;
                        mt.whi = 0;
                        r[RED_CLO] = 1;
                        r[RED_CHI] = 0;
                    }
                }
                return rg;
            }
            const int c_lo = rg.lo >> SH, c_hi = rg.hi >> SH;
            int out_off, cstride, wlo, whi;
            int my_coff = 0;  // lane c < 5: offset of output component c
            bool fail = false;
            if (!hist) {
                fail = (rg.lo < kmin_alloc || rg.hi > kmax_alloc);
                out_off = ((d * ring_n + slot) * NCOMP) * W + koff;
                cstride = W;
                wlo = max((c_lo - MG) << SH, kmin_alloc);
                whi = min(((c_hi + MG + 1) << SH) - 1, kmax_alloc);
                fail = fail || ((c_hi - c_lo) / VBLOCK_CHUNKS + 1 > P.blk_cap);
                my_coff = out_off + comp_idx(lane) * W;
                if (!full && lane >= 1 && lane < 5) {
                    const bool one = (lane == AW_COMP_I1 || lane == AW_COMP_D1);
                    const int n = one ? cmp_n1 : cmp_n2;
                    const int base = (lane == AW_COMP_I1) ? 0 : (lane == AW_COMP_D1) ? cmp_n1 : (lane == AW_COMP_I2) ? 2 * cmp_n1 : 2 * cmp_n1 + cmp_n2;
                    my_coff = cmp_base + (d * cmp_rows + base + (n > 0 ? s % n : 0)) * W + koff;
                }
            } else {
                const int clo = (c_lo - MG) << SH;
                rg.width = (c_hi - c_lo + 1 + 2 * MG) << SH;
                fail = (hist_used + (long long)NCOMP * rg.width > hcap_cur);
                out_off = hb_cur + (int)hist_used - clo;
                cstride = rg.width;
                wlo = clo;
                whi = clo + rg.width - 1;
                my_coff = out_off + comp_idx(lane) * cstride;
            }
            if (fail) {
                if (lead && lane == 0) r[RED_FAIL] = 1;
                return rg;
            }
            if (lead) {
                if (lane < 5) {
                    int pl = (lane == AW_COMP_M) ? mlo : (lane == AW_COMP_I1) ? i1lo : (lane == AW_COMP_I2) ? i2lo : (lane == AW_COMP_D1) ? d1lo : d2lo;
                    int ph = (lane == AW_COMP_M) ? mhi : (lane == AW_COMP_I1) ? i1hi : (lane == AW_COMP_I2) ? i2hi : (lane == AW_COMP_D1) ? d1hi : d2hi;
                    if (pl > ph) {
                        pl = 1;
                        ph = 0;
                    }
                    mt.lo[lane] = pl;
                    mt.hi[lane] = ph;
                    mt.coff[lane] = my_coff;
                }
                if (lane == 5) {
                    mt.off = out_off;
                    mt.cstride = cstride;
                    mt.wlo = wlo;
                    mt.whi = whi;
                    mt.full = full ? 1 : 0;
                    mt.bk0 = c_lo << SH;
                    mt.nblk = (c_hi - c_lo) / VBLOCK_CHUNKS + 1;
                    r[RED_CLO] = rg.lo;
                    r[RED_CHI] = rg.hi;
                }
            }
            if (lane < 5) dsc[16 + lane] = my_coff;
            if (AW_L1_PREFETCH) {
                // inputs of wavefront s+1: the row being written now (extension distance 1) or an older row
                int pfo = __shfl_sync(0xffffffffu, my_coff, comp);
                if (back != 1) {
                    pfo = -1;
                    if (lane < (TWO ? 7 : 4) && s + 1 - back >= 0) {
                        int sl = slot + 1 - back;
                        if (sl < 0) sl += ring_n;
                        const SlotMeta& m = ring_meta[mbase + sl];
                        if (m.lo[comp] <= m.hi[comp]) pfo = m.coff[comp];
                    }
                }
                if (lane >= (TWO ? 7 : 4)) pfo = -1;
                if (lane < 8) dsc[24 + lane] = pfo;
            }
            __syncwarp();
            if constexpr (VEC)
                wf_cells_v<BITS, TWO, WS>(ws, ioff, dsc, dsc + 16, rg.lo, rg.hi, fast_lo, fast_hi, wlo, whi, reinterpret_cast<const uint2*>(sv.pw),
                                           reinterpret_cast<const uint2*>(sv.tw), sv.p0, sv.t0, sv.plen, sv.tlen, k_end, comp_end, r, gwarp, gnw, pf_off,
                                           hist ? nullptr : blk_of(d, slot));
            return rg;
        };
//@region v_finish
        // after the barrier: END_REACHED of the new wavefront; akM_out = its max M antidiagonal
        auto v_finish = [&](int d, int mbase, int slot, int plen, int tlen, int k_end, int comp_end, int& akM_out) -> bool {
            int* r = red[d][red_i];
            const int clo = r[RED_CLO], chi = r[RED_CHI], akM = r[RED_AKM], akAll = r[RED_AKALL], endval = r[RED_END];
            const bool fail = r[RED_FAIL] != INT_MIN, oob = r[RED_OOB] != INT_MIN;
            akM_out = INT_MIN;
            ++w_steps;
            if (status != ST_OK) return false;
            if (fail) {
                status = ST_FAIL_WORKSPACE;
                return false;
            }
            if (clo > chi) return false;
            w_cells += (unsigned long long)(chi - clo + 1) * NCOMP;
            SlotMeta& mt = ring_meta[mbase + slot];
            if (oob) {  // exact wavefront_compute_trim_ends from the stored row (rare)
                int out[5];
#pragma unroll
                for (int c = 0; c < 5; ++c) out[c] = mt.coff[(TWO || c == AW_COMP_M || c == AW_COMP_I1 || c == AW_COMP_D1) ? c : AW_COMP_M];
                StepOut so;
                wf_rescan<NT, TWO, WS>(ws, out, clo, chi, plen, tlen, (LEAFPAR && wm) ? s_rescan_w[tid >> 5] : s_rescan, so, t_tid, wm ? 32 : NT, wm);
                if (t_tid < 32) {
                    int wl = -VBIG, wh = VBIG;  // cells outside a component's trimmed range hold garbage: only the common part reads unmasked
#pragma unroll
                    for (int c = 0; c < 5; ++c) {
                        mt.lo[c] = so.lo[c];
                        mt.hi[c] = so.hi[c];
                        if (so.lo[c] <= so.hi[c]) {
                            wl = max(wl, so.lo[c]);
                            wh = min(wh, so.hi[c]);
                        }
                    }
                    mt.wlo = wl;
                    mt.whi = wh;
                }
                team_sync();
            }
            if (t_tid < 32) {
                mt.akM = akM;
                mt.akAll = akAll;
            }
            akM_out = akM;
            return mt.lo[comp_end] <= k_end && k_end <= mt.hi[comp_end] && endval >= tlen;
        };
        // score-0 wavefront (wavefront_unialign_init_end2end): cell 0 of component `cb` inside a NULL-filled neighbourhood
        auto v_init_row = [&](int d, int mbase, bool hist, const SeqView& sv, int cb, int ce, int k_end, int& akM_out) -> bool {
            constexpr int SH = (CPT == 8) ? 3 : 2;
            constexpr int MG = VMARGIN / CPT;
            int* r = red[d][red_i];
            SlotMeta& mt = ring_meta[mbase];
            int out_off, cstride;
            const int clo = max((-MG) << SH, kmin_alloc), chi = min(((MG + 1) << SH) - 1, kmax_alloc);
            if (!hist) {
                out_off = ((d * ring_n) * NCOMP) * W + koff;
                cstride = W;
            } else {
                cstride = chi - clo + 1;
                out_off = hb_cur - clo;
                hist_used = (long long)NCOMP * cstride;
            }
            if constexpr (VEC) {
                WS* row = ws + out_off + comp_idx(cb) * cstride;
                if (t_tid <= 2 * MG) {
                    const int kc = (t_tid - MG) << SH;
                    uint32_t v[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) v[i] = VecT<WS>::NULLW;
                    if (kc == 0) {
                        int m = 0;
                        if (cb == AW_COMP_M)
                            m = lcp2(reinterpret_cast<const uint2*>(sv.pw), reinterpret_cast<const uint2*>(sv.tw), sv.p0, sv.t0, min(sv.plen, sv.tlen));
                        v[0] = (sizeof(WS) == 2) ? ((v[0] & 0xffff0000u) | ((uint32_t)m & 0xffffu)) : (uint32_t)m;
                        r[RED_AKM] = (cb == AW_COMP_M) ? 2 * m : INT_MIN;
                        r[RED_AKALL] = 2 * m;
                        if (cb == ce && k_end == 0) r[RED_END] = m;
                        if (!hist) *reinterpret_cast<int2*>(blk_of(d, 0)) = make_int2((cb == AW_COMP_M) ? 2 * m : INT_MIN, 2 * m);
                    }
                    if (kc >= clo && kc + CPT - 1 <= chi) st_vec<WS>(row + kc, v);
                }
            }
            if (t_tid < 32) {
                if (t_tid < 5) {
                    mt.lo[t_tid] = (t_tid == cb) ? 0 : 1;
                    mt.hi[t_tid] = 0;
                }
                if (t_tid < 5) mt.coff[t_tid] = out_off + comp_idx(t_tid) * cstride;
                if (t_tid == 5) {
                    mt.off = out_off;
                    mt.cstride = cstride;
                    mt.wlo = clo;
                    mt.whi = chi;
                    mt.full = 1;
                    mt.bk0 = 0;
                    mt.nblk = 1;
                }
            }
            team_sync();
            const int akM = r[RED_AKM], endval = r[RED_END];
            if (t_tid < 32) {
                mt.akM = akM;
                mt.akAll = r[RED_AKALL];
            }
            akM_out = akM;
            return k_end == 0 && endval >= sv.tlen;  // only component cb is non-empty, at k = 0
        };

        // ---- base-case helpers, team-aware (the whole CTA or one warp, see LEAFPAR) ----
        auto write_hist_meta = [&](int s, const SlotMeta& m) {
            if (t_tid == 0) {
                int* g = hmeta_cur + (size_t)s * HIST_META_INTS;
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                    g[c] = m.lo[c];
                    g[5 + c] = m.hi[c];
                }
                g[10] = m.off;
                g[11] = m.cstride;
            }
        };
        // wavefront_backtrace_affine by ONE warp (all 32 lanes call it): lanes evaluate the nine candidates; returns the number of
        // runs pushed, back to front, into the team's leaf run buffer
        auto bt_run = [&](int ce_, int score_, int plen_, int tlen_, int k_end_) -> unsigned {
            const int lane = tid & 31;
            unsigned n_leaf = 0;
            unsigned last_run = 0;  // pending run (merged before being stored)
            auto push = [&](unsigned op, unsigned len) {
                if (len == 0) return;
                if (last_run != 0 && (last_run & 3u) == op) {
                    last_run += len << 2;
                } else {
                    if (last_run != 0) {
                        if (lane == 0 && n_leaf < lcap_cur) lruns_cur[n_leaf] = last_run;
                        ++n_leaf;
                    }
                    last_run = (len << 2) | op;
                }
            };
            int type = ce_, sc = score_, k = k_end_, offset = tlen_;
            int v = plen_, h = tlen_;
            // lane l evaluates backtrace candidate type l+1 (AW_BT_*)
            while (v > 0 && h > 0 && sc > 0) {
                const int bt = lane + 1;
                int cand_v = INT_MIN;
                if (lane < 9) {
                    int comp_src, cost, dk, add;
                    bool active;
                    switch (bt) {
                        case AW_BT_M: comp_src = AW_COMP_M; cost = pen.x; dk = 0; add = 1; active = (type == AW_COMP_M); break;
                        case AW_BT_I1_OPEN: comp_src = AW_COMP_M; cost = pen.o1 + pen.e1; dk = -1; add = 1; active = (type == AW_COMP_M || type == AW_COMP_I1); break;
                        case AW_BT_I1_EXT: comp_src = AW_COMP_I1; cost = pen.e1; dk = -1; add = 1; active = (type == AW_COMP_M || type == AW_COMP_I1); break;
                        case AW_BT_I2_OPEN: comp_src = AW_COMP_M; cost = pen.o2 + pen.e2; dk = -1; add = 1; active = TWO && (type == AW_COMP_M || type == AW_COMP_I2); break;
                        case AW_BT_I2_EXT: comp_src = AW_COMP_I2; cost = pen.e2; dk = -1; add = 1; active = TWO && (type == AW_COMP_M || type == AW_COMP_I2); break;
                        case AW_BT_D1_OPEN: comp_src = AW_COMP_M; cost = pen.o1 + pen.e1; dk = 1; add = 0; active = (type == AW_COMP_M || type == AW_COMP_D1); break;
                        case AW_BT_D1_EXT: comp_src = AW_COMP_D1; cost = pen.e1; dk = 1; add = 0; active = (type == AW_COMP_M || type == AW_COMP_D1); break;
                        case AW_BT_D2_OPEN: comp_src = AW_COMP_M; cost = pen.o2 + pen.e2; dk = 1; add = 0; active = TWO && (type == AW_COMP_M || type == AW_COMP_D2); break;
                        default: comp_src = AW_COMP_D2; cost = pen.e2; dk = 1; add = 0; active = TWO && (type == AW_COMP_M || type == AW_COMP_D2); break;
                    }
                    const int ss = sc - cost;
                    if (active && ss >= 0) {
                        const int* g = hmeta_cur + (size_t)ss * HIST_META_INTS;
                        const int kk = k + dk;
                        if (g[comp_src] <= kk && kk <= g[5 + comp_src]) {
                            const int val = ws[g[10] + comp_idx(comp_src) * g[11] + kk];
                            if (val >= 0) cand_v = ((val + add) << AW_BT_TYPE_BITS) | bt;
                        }
                    }
                }
                const int max_all = __reduce_max_sync(0xffffffffu, cand_v);
                if (max_all == INT_MIN) {  // cannot happen on a valid path
                    status = ST_FAIL_WORKSPACE;
                    break;
                }
                if (type == AW_COMP_M) {
                    const int max_offset = max_all >> AW_BT_TYPE_BITS;
                    push(AW_OP_M, (unsigned)max(0, offset - max_offset));
                    offset = max_offset;
                    v = offset - k;
                    h = offset;
                    if (v <= 0 || h <= 0) break;
                }
                const int b = max_all & 0xF;
                switch (b) {
                    case AW_BT_M: sc -= pen.x; type = AW_COMP_M; break;
                    case AW_BT_I1_OPEN: sc -= pen.o1 + pen.e1; type = AW_COMP_M; break;
                    case AW_BT_I1_EXT: sc -= pen.e1; type = AW_COMP_I1; break;
                    case AW_BT_I2_OPEN: sc -= pen.o2 + pen.e2; type = AW_COMP_M; break;
                    case AW_BT_I2_EXT: sc -= pen.e2; type = AW_COMP_I2; break;
                    case AW_BT_D1_OPEN: sc -= pen.o1 + pen.e1; type = AW_COMP_M; break;
                    case AW_BT_D1_EXT: sc -= pen.e1; type = AW_COMP_D1; break;
                    case AW_BT_D2_OPEN: sc -= pen.o2 + pen.e2; type = AW_COMP_M; break;
                    default: sc -= pen.e2; type = AW_COMP_D2; break;
                }
                if (b == AW_BT_M) {
                    push(AW_OP_X, 1);
                    --offset;
                } else if (b <= AW_BT_I2_EXT) {
                    push(AW_OP_I, 1);
                    --k;
                    --offset;
                } else {
                    push(AW_OP_D, 1);
                    ++k;
                }
                v = offset - k;
                h = offset;
            }
            if (v > 0 && h > 0) {
                const int nm = min(v, h);
                push(AW_OP_M, (unsigned)nm);
                v -= nm;
                h -= nm;
            }
            if (v > 0) push(AW_OP_D, (unsigned)v);
            if (h > 0) push(AW_OP_I, (unsigned)h);
            if (last_run != 0) {
                if (lane == 0 && n_leaf < lcap_cur) lruns_cur[n_leaf] = last_run;
                ++n_leaf;
            }
            return n_leaf;
        };

        // ---- LEAFPAR: align the pending leaves, one warp each, then append their runs in DFS order ----
        int n_pending = 0;
        auto flush_leaves = [&]() {
            if constexpr (LEAFPAR) {
                cta_sync<NT>();  // s_leaf is complete; no cooperative step is in flight
                const int w = tid >> 5, lane = tid & 31;
                if (w < n_pending) {
                    const SubProblem lf = s_leaf[w];
                    const int lp = lf.pe - lf.pb, lt = lf.te - lf.tb;
                    unsigned n_leaf = 0;
                    int lscore = -1;
                    const unsigned long long cells0 = w_cells;
                    const unsigned steps0 = w_steps;
                    // the team is this warp: its own SlotMeta ring and reduction row, a slice of the history arena, of the
                    // history metadata and of the leaf run buffer
                    wm = true;
                    t_tid = lane;
                    t_d = 2 + w;
                    red_i = 0;
                    hcap_cur = (long long)((P.hist_ints / NW) & ~15);
                    hb_cur = hist_base + w * (int)hcap_cur;
                    hscores_cur = P.hist_max_scores / NW;
                    hmeta_cur = hist_meta + (size_t)w * hscores_cur * HIST_META_INTS;
                    lcap_cur = P.runs_cap / NW;
                    lruns_cur = leaf_runs + (size_t)w * lcap_cur;
                    hist_used = 0;
                    if (lt == 0 || lp == 0) {  // wavefront_bialign_alignment's trivial cases: one pure gap
                        const unsigned len = (unsigned)(lt == 0 ? lp : lt);
                        if (len) {
                            if (lane == 0) lruns_cur[0] = (len << 2) | (lt == 0 ? AW_OP_D : AW_OP_I);
                            n_leaf = 1;
                        }
                    } else {
                        const int k_end = lt - lp;
                        const SeqView sv = SeqView{reinterpret_cast<const uint32_t*>(pf2), reinterpret_cast<const uint32_t*>(tf2), lf.pb, lf.tb, lp, lt, false};
                        for (int i = lane; i < 3 * NRED; i += 32) (&red[t_d][0][0])[i] = INT_MIN;
                        __syncwarp();
                        const int mbase = t_d * ring_n;
                        int ak, score = 0, slot = 0;
                        bool done = v_init_row(t_d, mbase, true, sv, lf.cb, lf.ce, k_end, ak);
                        write_hist_meta(0, ring_meta[mbase]);
                        rotate_red();
                        while (!done) {
                            ++score;
                            slot = (slot + 1 == ring_n) ? 0 : slot + 1;
                            if (score >= hscores_cur) {
                                status = ST_FAIL_WORKSPACE;
                                break;
                            }
                            const VRange rg = v_launch(t_d, mbase, score, slot, 0, 1, 0, true, true, sv, k_end, lf.ce);
                            hist_used += (long long)NCOMP * rg.width;
                            __syncwarp();
                            done = v_finish(t_d, mbase, slot, lp, lt, k_end, lf.ce, ak);
                            if (status != ST_OK) break;
                            write_hist_meta(score, ring_meta[mbase + slot]);
                            rotate_red();
                        }
                        __syncwarp();  // the warp's history rows and metadata are visible to all of its lanes
                        if constexpr (!SCORE) {
                            if (status == ST_OK) n_leaf = bt_run(lf.ce, score, lp, lt, k_end);
                        }
                        lscore = score;
                    }
                    if (lane == 0) {
                        s_leaf_n[w] = n_leaf;
                        s_leaf_st[w] = status;
                        s_leaf_score[w] = lscore;
                        s_leaf_cells[w] = w_cells - cells0;
                        s_leaf_steps[w] = w_steps - steps0;
                    }
                    w_cells = cells0;  // every thread adds every leaf's work below, so that the counters stay CTA-uniform
                    w_steps = steps0;
                    wm = false;
                    t_tid = tid;
                    t_d = 0;
                    hb_cur = hist_base;
                    hcap_cur = P.hist_ints;
                    hscores_cur = P.hist_max_scores;
                    hmeta_cur = hist_meta;
                    lcap_cur = P.runs_cap;
                    lruns_cur = leaf_runs;
                }
                cta_sync<NT>();
                for (int q = 0; q < n_pending; ++q) {
                    status = max(status, s_leaf_st[q]);
                    w_cells += s_leaf_cells[q];
                    w_steps += s_leaf_steps[q];
                    if (s_leaf_score[q] >= 0) {
                        ++w_base;
                        w_maxbase = max(w_maxbase, (unsigned)s_leaf_score[q]);
                    }
                }
                for (int i = tid; i < RM_N * 3 * NRED; i += NT) (&red[0][0][0])[i] = INT_MIN;  // the warps rotated their rows on their own
                red_i = 0;
                if constexpr (SCORE) {  // the one leaf is the top level (a pure gap leaves -1 here, see K8); it has no runs to append
                    sc_pen = s_leaf_score[0];
                    n_pending = 0;
                    cta_sync<NT>();
                    return;
                }
                const unsigned long long lpart = P.runs_cap / NW;
                for (int q = 0; q < n_pending && status == ST_OK; ++q) {
                    // append leaf q's runs (stored back to front) to the pair's CIGAR, merging with the last run when the op continues
                    const uint32_t* lr = leaf_runs + (size_t)q * lpart;
                    const unsigned n_leaf = s_leaf_n[q];
                    const unsigned base_n = s_nruns;
                    unsigned skip = 0;
                    if (n_leaf > 0 && base_n > 0 && (pair_runs[base_n - 1] & 3u) == (lr[n_leaf - 1] & 3u)) skip = 1;
                    cta_sync<NT>();
                    if (n_leaf > lpart || base_n + n_leaf > P.runs_cap) {
                        status = ST_FAIL_WORKSPACE;
                        break;
                    }
                    if (tid == 0 && skip) pair_runs[base_n - 1] += lr[n_leaf - 1] & ~3u;
                    for (unsigned i = skip + tid; i < n_leaf; i += NT) pair_runs[base_n + i - skip] = lr[n_leaf - 1 - i];
                    if (tid == 0) s_nruns = base_n + n_leaf - skip;
                    cta_sync<NT>();
                }
                n_pending = 0;
                cta_sync<NT>();
            }
        };

//@region subproblem setup
        bool flush_req = false;  // LEAFPAR: the pending leaves must be appended before the sub-problem on top of the stack runs
        for (;;) {
            // the single call site of flush_leaves (instruction-cache footprint): a full batch, a request, or the end of the DFS
            if (LEAFPAR && n_pending > 0 && status == ST_OK && (n_pending == NW || flush_req || sp_n == 0)) flush_leaves();
            flush_req = false;
            if (!(sp_n > 0 && (status == ST_OK || CL > 1))) break;
            const SubProblem sp = stack[--sp_n];
            const int plen = sp.pe - sp.pb, tlen = sp.te - sp.tb;
            // cluster kernels: short sub-problems (and the trivial ones) belong to CTA 0 alone -- the other CTAs drop them
            // and run ahead to the next cluster-wide sub-problem, where they wait for CTA 0
            const bool solo = (CL > 1) && (tlen == 0 || plen == 0 || plen + tlen < P.solo_len);
            const int cl_off = (CL > 1 && !solo) ? (int)crank : 0, cl_n = (CL > 1 && !solo) ? CL : 1;
            if constexpr (CL > 1) {
                if (solo) {
                    if (crank != 0 || status != ST_OK) continue;
                } else {
                    // every CTA must enter a cluster-wide sub-problem with the same status (CTA 0 may have failed on its own);
                    // the barriers also keep CTA 0's solo writes apart from the other CTAs' last reads of the rings
                    // ... and with the same reduction-buffer rotation: CTA 0 has rotated its buffers through every solo step
                    // since the last cluster-wide sub-problem, the others have not
                    for (int i = tid; i < 2 * 3 * NRED; i += NT) (&red[0][0][0])[i] = INT_MIN;
                    red_i = 0;
                    if (tid == 0) s_cl_status = status;
                    cluster_sync_all();
                    int st = status;
#pragma unroll
                    for (unsigned r = 0; r < (unsigned)CL; ++r) st = max(st, ld_dsmem_int(&s_cl_status, r));
                    cluster_sync_all();
                    status = st;
                    if (status != ST_OK) break;
                }
            }
            if constexpr (LEAFPAR) {
                // trivial sub-problems and base cases are leaves of the recursion: they wait until NW of them can run side by side
                // (rem == -1 marks an END_REACHED fallback that was put back: it runs cooperatively, see below)
                if (tlen == 0 || plen == 0 || (sp.rem <= AW_BIALIGN_FALLBACK_MIN_SCORE && sp.rem != -1)) {
                    if (tid == 0) s_leaf[n_pending] = sp;
                    ++n_pending;
                    continue;
                }
            }
            // ---- wavefront_bialign_alignment: trivial cases ----
            if (tlen == 0 || plen == 0) {
                if (tid == 0) {
                    if (tlen == 0) emit_run(AW_OP_D, (unsigned)plen);
                    else emit_run(AW_OP_I, (unsigned)tlen);
                }
                cta_sync<NT>();
                continue;
            }
            const int k_end = tlen - plen;
            bool do_base = sp.rem <= AW_BIALIGN_FALLBACK_MIN_SCORE;
            Breakpoint bp;
            bp.score = INT_MAX;
            bp.score_f = bp.score_r = bp.k_f = bp.off_f = 0;
            bp.comp = AW_COMP_M;

            bool force_full = false;  // int16 path: keep every I/D row in the full ring (second attempt, see below)
            if (!do_base) {
            retry_breakpoint:
                // =========== K6: wavefront_bialign_find_breakpoint ===========
                SeqView svd[2];
                if constexpr (VEC) {
                    svd[0] = SeqView{reinterpret_cast<const uint32_t*>(pf2), reinterpret_cast<const uint32_t*>(tf2), sp.pb, sp.tb, plen, tlen, false};
                    svd[1] = SeqView{reinterpret_cast<const uint32_t*>(pr2), reinterpret_cast<const uint32_t*>(tr2), PLEN - sp.pe, TLEN - sp.te, plen, tlen, false};
                } else {
                    svd[0] = SeqView{pw, tw, sp.pb, sp.tb, plen, tlen, false};
                    svd[1] = SeqView{pw, tw, sp.pe - 1, sp.te - 1, plen, tlen, true};
                }
                const int cbeg[2] = {sp.cb, sp.ce}, cend[2] = {sp.ce, sp.cb};
                int cur_slot[2] = {0, 0};  // ring slot of the newest committed/computed score per direction
                auto ring_off = [&](int d, int slot, int c) -> int { return ((d * ring_n + slot) * NCOMP + comp_idx(c)) * W + koff; };
                auto slot_back = [&](int slot, int back) -> int {  // slot of (score - back), back <= scope
                    const int s = slot - back;
                    return s < 0 ? s + ring_n : s;
                };
                // score-0 wavefront of direction d (wavefront_unialign_init_end2end) + extend
                auto init_dir = [&](int d, StepOut& so) {
                    int* r = red[d][red_i];
                    if (tid == 0) {
                        int m = 0;
                        if (cbeg[d] == AW_COMP_M) m = extend_cell<BITS>(svd[d], 0, 0);
                        ws[ring_off(d, 0, cbeg[d])] = to_ws<WS>(m);
                        r[RED_AKM] = (cbeg[d] == AW_COMP_M) ? 2 * m : INT_MIN;
                        r[RED_AKALL] = 2 * m;
                        if (cbeg[d] == AW_COMP_M && cend[d] == AW_COMP_M && k_end == 0) r[RED_END] = m;
                    }
                    cta_sync<NT>();
#pragma unroll
                    for (int c = 0; c < 5; ++c) {
                        so.lo[c] = (c == cbeg[d]) ? 0 : 1;
                        so.hi[c] = 0;
                    }
                    so.akM = r[RED_AKM];
                    so.akAll = r[RED_AKALL];
                    so.endval = r[RED_END];
                    so.ambiguous = false;
                    cur_slot[d] = 0;
                    store_meta(ring_meta[d * ring_n + 0], so);
                    rotate_red();
                };
                // what survives of a step until its barrier: the computed range (null step iff lo > hi)
                struct Range {
                    int lo, hi;
                };
                auto out_offsets = [&](int d, int slot, int (&out)[5]) {
#pragma unroll
                    for (int c = 0; c < 5; ++c) out[c] = ring_off(d, slot, (TWO || c == AW_COMP_M || c == AW_COMP_I1 || c == AW_COMP_D1) ? c : AW_COMP_M);
                };
                // descriptors + limits + cell loop of wavefront `s` (ring slot `slot`) of direction d; no barrier
//@region launch_dir
                auto launch_dir = [&](int d, int s, int slot) -> Range {
                    In in[7];
                    auto fetch = [&](int c, int back) -> In {
                        In w;
                        if (s - back < 0) {
                            w.off = 0;
                            w.lo = 1;
                            w.hi = 0;
                            return w;
                        }
                        const int sl = slot_back(slot, back);
                        const SlotMeta& m = ring_meta[d * ring_n + sl];
                        w.off = ring_off(d, sl, c);
                        w.lo = m.lo[c];
                        w.hi = m.hi[c];
                        return w;
                    };
                    in[IN_MX] = fetch(AW_COMP_M, pen.x);
                    in[IN_MO1] = fetch(AW_COMP_M, pen.o1 + pen.e1);
                    in[IN_I1E] = fetch(AW_COMP_I1, pen.e1);
                    in[IN_D1E] = fetch(AW_COMP_D1, pen.e1);
                    if (TWO) {
                        in[IN_MO2] = fetch(AW_COMP_M, pen.o2 + pen.e2);
                        in[IN_I2E] = fetch(AW_COMP_I2, pen.e2);
                        in[IN_D2E] = fetch(AW_COMP_D2, pen.e2);
                    } else {
                        in[IN_MO2].off = in[IN_I2E].off = in[IN_D2E].off = 0;
                        in[IN_MO2].lo = in[IN_I2E].lo = in[IN_D2E].lo = 1;
                        in[IN_MO2].hi = in[IN_I2E].hi = in[IN_D2E].hi = 0;
                    }
                    Range r;
                    limits(in, r.lo, r.hi);
                    ++w_steps;
                    if (r.lo > r.hi) return r;
                    if (r.lo < kmin_alloc || r.hi > kmax_alloc) {
                        status = ST_FAIL_WORKSPACE;
                        return r;
                    }
                    if (status != ST_OK) return r;
                    int out[5];
                    out_offsets(d, slot, out);
                    wf_cells<NT, BITS, TWO, WS>(ws, in, out, r.lo, r.hi, d == 0 ? svd[0] : svd[1], k_end, d == 0 ? cend[0] : cend[1], red[d][red_i]);
                    w_cells += (unsigned long long)(r.hi - r.lo + 1) * NCOMP;
                    return r;
                };
                // after the barrier: trimmed ranges -> ring meta; returns END_REACHED of this wavefront
//@region finish_dir
                auto finish_dir = [&](int d, int slot, const Range& r) -> bool {
                    SlotMeta& mt = ring_meta[d * ring_n + slot];
                    if (r.lo > r.hi || status != ST_OK) {
                        set_empty(mt);
                        return false;
                    }
                    StepOut so;
                    wf_finish<TWO>(red[d][red_i], r.lo, r.hi, so);
                    if (so.ambiguous) {
                        int out[5];
                        out_offsets(d, slot, out);
                        wf_rescan<NT, TWO, WS>(ws, out, r.lo, r.hi, plen, tlen, red[d][red_i], so, tid, NT, false);
                    }
                    store_meta(mt, so);
                    return end_reached(so, d == 0 ? cend[0] : cend[1], k_end, tlen);
                };
                auto next_slot = [&](int slot) -> int { return slot + 1 == ring_n ? 0 : slot + 1; };

//@region overlap
                // wavefront_bialign_overlap: A0 = direction d0 at score s0, A1 = direction d1 at scores s1..s1-scope+1
                auto overlap = [&](int d0, int d1, int s0, int s1) {
                    const int slot0 = cur_slot[d0];
                    const SlotMeta& m0 = ring_meta[d0 * ring_n + slot0];
                    const int kinv = tlen - plen;
                    const int bp_entry = bp.score;
                    // test t = i*5 + oi: reverse score s1-i, component order D2,I2,D1,I1,M
                    auto test_comp = [](int oi) -> int { return oi == 0 ? AW_COMP_D2 : oi == 1 ? AW_COMP_I2 : oi == 2 ? AW_COMP_D1 : oi == 3 ? AW_COMP_I1 : AW_COMP_M; };
                    auto credit_of = [&](int c) -> int { return (c == AW_COMP_M) ? 0 : ((c == AW_COMP_D1 || c == AW_COMP_I1) ? pen.o1 : pen.o2); };
                    // candidate tests (gate + range intersection + antidiagonal bound), kept in order, by warp 0
                    // the scan ranges are cut along the block grid of A0's wavefront (int16 path; else a fixed grid)
                    constexpr int OV_U = 8, OV_CH = VEC ? VBW : 32 * OV_U;  // diagonals per lane / per warp chunk of the scan
                    static_assert(OV_CH <= 32 * OV_U, "a warp chunk must fit OV_U diagonals per lane");
                    const int grid0 = VEC ? m0.bk0 : kmin_alloc;
                    if (tid < 32) {
                        int ncand = 0;
                        int a1m = INT_MIN, a1a = INT_MIN, gmin = INT_MAX, gmax = INT_MIN;  // best antidiagonal bound of A1 per class, candidates' span
                        const int ntests = min(scope, s1 + 1) * 5;
                        for (int base = 0; base < ntests; base += 32) {
                            const int t = base + tid;
                            bool ok = false;
                            int klo = 0, khi = -1;
                            if (t < ntests) {
                                const int i = t / 5, oi = t - 5 * i, c = test_comp(oi);
                                const int si = s1 - i;
                                if (TWO || (c != AW_COMP_D2 && c != AW_COMP_I2)) {
                                    const SlotMeta& m1 = ring_meta[d1 * ring_n + slot_back(cur_slot[d1], i)];
                                    const int lo0 = m0.lo[c], hi0 = m0.hi[c], lo1 = kinv - m1.hi[c], hi1 = kinv - m1.lo[c];
                                    ok = (s0 + si - credit_of(c) < bp_entry) && lo0 <= hi0 && m1.lo[c] <= m1.hi[c] && !(hi1 < lo0 || hi0 < lo1);
                                    klo = max(lo0, lo1);
                                    khi = min(hi0, hi1);
                                    if (ok) {
                                        const long long a0 = (c == AW_COMP_M) ? m0.akM : m0.akAll, a1 = (c == AW_COMP_M) ? m1.akM : m1.akAll;
                                        ok = a0 + a1 >= (long long)plen + tlen;  // necessary for off0 + off1 >= tlen
                                        if (ok) {
                                            if (c == AW_COMP_M) a1m = max(a1m, (int)a1);
                                            else a1a = max(a1a, (int)a1);
                                            gmin = min(gmin, klo);
                                            gmax = max(gmax, khi);
                                        }
                                    }
                                }
                            }
                            const unsigned mask = __ballot_sync(0xffffffffu, ok);
                            if (ok) {
                                const int pos = ncand + __popc(mask & ((1u << tid) - 1u));
                                cand[pos] = t;
                                hitk[pos] = INT_MAX;
                                cklo[pos] = klo;
                                ckhi[pos] = khi;
                            }
                            ncand += __popc(mask);
                        }
                        a1m = __reduce_max_sync(0xffffffffu, a1m);
                        a1a = __reduce_max_sync(0xffffffffu, a1a);
                        gmin = __reduce_min_sync(0xffffffffu, gmin);
                        gmax = __reduce_max_sync(0xffffffffu, gmax);
                        if (tid == 0) {
                            s_ncand = ncand;
                            s_nact = 0;
                            s_ov[0] = (a1m == INT_MIN) ? INT_MAX : plen + tlen - a1m;  // a block of A0 needs at least this much to meet an M cell
                            s_ov[1] = (a1a == INT_MIN) ? INT_MAX : plen + tlen - a1a;
                            s_ov[2] = gmin;
                            s_ov[3] = gmax;
                        }
                    }
                    cta_sync<NT>();
                    const int ncand = s_ncand;
                    // blocks of A0's wavefront whose own maxima can reach any candidate at all: almost none, the wavefronts
                    // only touch near the optimal path.  The scan then visits (candidate, active block) pairs only.
                    const int b_lo = ncand ? (s_ov[2] - grid0) / OV_CH : 0, b_hi = ncand ? (s_ov[3] - grid0) / OV_CH : -1;
                    bool implicit = !VEC;  // implicit list = every block between b_lo and b_hi
                    if constexpr (VEC) {
                        const int thr_m = s_ov[0], thr_a = s_ov[1];
                        const int2* bl0 = reinterpret_cast<const int2*>(blk_of(d0, slot0));
                        for (int b = b_lo + tid; b <= b_hi; b += NT) {
                            const int2 v = bl0[b];
                            if (v.x >= thr_m || v.y >= thr_a) {
                                const int pos = atomicAdd(&s_nact, 1);
                                if (pos < ACT_MAX) s_act[pos] = b;
                            }
                        }
                        cta_sync<NT>();
                        implicit = s_nact > ACT_MAX;
                    }
                    const int nact = implicit ? (b_hi - b_lo + 1) : s_nact;
                    {
                        const int lane = tid & 31;
                        const long long nitems = (long long)ncand * nact;
                        for (long long item = tid >> 5; item < nitems; item += NT / 32) {
                            const int j = (int)(item / nact), a = (int)(item - (long long)j * nact);
                            const int b0 = implicit ? b_lo + a : s_act[a];
                            const int kb = grid0 + b0 * OV_CH;
                            const int max_lo = max(cklo[j], kb), min_hi = min(ckhi[j], kb + OV_CH - 1);
                            if (max_lo > min_hi) continue;
                            const int kbase = max_lo;
                            if (hitk[j] < kbase) continue;  // an earlier block already holds a hit
                            const int t = cand[j], i = t / 5, c = test_comp(t - 5 * i);
                            const int sl1 = slot_back(cur_slot[d1], i);
                            const SlotMeta& m1 = ring_meta[d1 * ring_n + sl1];
                            if constexpr (VEC) {
                                // off0 + off1 >= tlen  <=>  (2 off0 - k0) + (2 off1 - k1) >= plen + tlen: bound both sides by their blocks' maxima
                                const int sel = (c == AW_COMP_M) ? 0 : 1;
                                const int* bl1 = blk_of(d1, sl1);
                                const int a0 = blk_of(d0, slot0)[2 * b0 + sel];
                                const int nb1 = m1.nblk - 1;
                                const int b1a = min(max((kinv - min_hi - m1.bk0) / VBW, 0), nb1), b1b = min(max((kinv - max_lo - m1.bk0) / VBW, 0), nb1);
                                const int a1 = max(bl1[2 * b1a + sel], bl1[2 * b1b + sel]);
                                if ((long long)a0 + a1 < (long long)plen + tlen) continue;
                            }
                            const WS* p0 = ws + (VEC ? m0.coff[c] : ring_off(d0, slot0, c));
                            const WS* p1 = ws + (VEC ? m1.coff[c] : ring_off(d1, sl1, c)) + kinv;
                            int h0[OV_U], h1[OV_U];
#pragma unroll
                            for (int u = 0; u < OV_U; ++u) {
                                const int k0 = min(kbase + u * 32 + lane, min_hi);  // clamped duplicates are re-tested harmlessly
                                h0[u] = p0[k0];
                                h1[u] = p1[-k0];
                            }
                            int best = INT_MAX;
#pragma unroll
                            for (int u = OV_U - 1; u >= 0; --u) {
                                const int k0 = kbase + u * 32 + lane;
                                bool hit = (k0 <= min_hi) && (h0[u] + h1[u] >= tlen);
                                if (hit && c != AW_COMP_M) {  // indel2indel: the forward cell must be in bounds
                                    const int kk = (d0 == 0) ? k0 : kinv - k0, hh = (d0 == 0) ? h0[u] : h1[u];
                                    hit = !(hh - kk > plen || hh > tlen);
                                }
                                if (hit) best = k0;
                            }
                            best = __reduce_min_sync(0xffffffffu, best);
                            if (lane == 0 && best != INT_MAX) atomicMin(&hitk[j], best);
                        }
                    }
                    cta_sync<NT>();
                    // replay the candidate tests in WFA2's order with the live breakpoint score
                    for (int j = 0; j < ncand; ++j) {
                        const int k0 = hitk[j];
                        if (k0 == INT_MAX) continue;
                        const int t = cand[j], i = t / 5, c = test_comp(t - 5 * i);
                        const int si = s1 - i, credit = credit_of(c);
                        if (s0 + si - credit >= bp.score) continue;
                        const int sl1 = slot_back(cur_slot[d1], i);
                        const int k1 = kinv - k0;
                        const int h0 = ws[(VEC ? m0.coff[c] : ring_off(d0, slot0, c)) + k0];
                        const int h1 = ws[(VEC ? ring_meta[d1 * ring_n + sl1].coff[c] : ring_off(d1, sl1, c)) + k1];
                        if (d0 == 0) {
                            bp.score_f = s0;
                            bp.score_r = si;
                            bp.k_f = k0;
                            bp.off_f = h0;
                        } else {
                            bp.score_f = si;
                            bp.score_r = s0;
                            bp.k_f = k1;
                            bp.off_f = h1;
                        }
                        bp.score = s0 + si - credit;
                        bp.comp = c;
                    }
                    cta_sync<NT>();  // cand/hitk are rewritten by the next call
                };

//@region phase driver
                StepOut so;
                int score_f = 0, score_r = 0, f_ak = 0, r_ak = 0;
                bool fb_end = false;  // END_REACHED -> fall back to the base case
                if constexpr (VEC) {
                    int ak;
                    if (v_init_row(0, 0, false, svd[0], cbeg[0], cend[0], k_end, ak)) fb_end = true;
                    rotate_red();
                    f_ak = max(0, ak);
                    if (!fb_end) {
                        if (v_init_row(1, ring_n, false, svd[1], cbeg[1], cend[1], k_end, ak)) fb_end = true;
                        rotate_red();
                        r_ak = max(0, ak);
                    }
                } else {
                    init_dir(0, so);
                    if (end_reached(so, cend[0], k_end, tlen)) fb_end = true;
                    f_ak = max(0, so.akM);
                    if (!fb_end) {
                        init_dir(1, so);
                        if (end_reached(so, cend[1], k_end, tlen)) fb_end = true;
                        r_ak = max(0, so.akM);
                    }
                }
                bool last_forward = false;
                bool rev_pending = false;  // reverse wavefront score_r+1 already sits in slot next_slot(cur_slot[1])
                const int max_antidiagonal = plen + tlen - 1;
                bool rev_pending_done = false;  // END_REACHED flag of that speculative wavefront
                // int16 path: I/D rows go to the compact rings until the wavefronts come close; the overlap phase needs the
                // last `scope` rows of both directions in the full ring.  first_full = first score of the current run of full rows.
                int first_full = 1;
                lap(4);
                // ---- phase 1: forward step s_f+1 and (speculative) reverse step s_r+1 share one barrier ----
                while (!fb_end && status == ST_OK) {
                    if (f_ak + r_ak >= max_antidiagonal) break;
                    const int slot_f = next_slot(cur_slot[0]), slot_r = next_slot(cur_slot[1]);
                    bool done, done_r;
                    int akM_f, akM_r;
                    if constexpr (VEC) {
                        // half of the warps advance the forward wavefront, the other half the reverse one
                        constexpr int HW = NT / 64;
                        const int warp = tid >> 5;
                        // switch to the full ring 3 x scope expected steps before the wavefronts can touch
                        const int reached = f_ak + r_ak;
                        const int rate = reached / max(1, score_f) + 2;  // antidiagonals gained per step pair so far
                        const bool full = !AW_COMPACT_ID_RINGS || force_full || (max_antidiagonal - reached <= 3 * scope * rate + 128);
                        if (!full) first_full = INT_MAX;
                        else if (first_full == INT_MAX) first_full = score_f + 1;
                        {
                            const int d = (warp < HW) ? 0 : 1;  // one call site for both directions (instruction-cache footprint)
                            const int lw = d ? warp - HW : warp;
                            v_launch(d, d * ring_n, (d ? score_r : score_f) + 1, d ? slot_r : slot_f, cl_off * HW + lw, cl_n * HW, lw, false, full,
                                     d ? svd[1] : svd[0], k_end, d ? cend[1] : cend[0]);
                        }
                        step_sync(solo);
                        bool dn[2];
                        int ak2[2];
#pragma unroll 1
                        for (int d = 0; d < 2; ++d) {
                            int ak;
                            const bool f = v_finish(d, d * ring_n, d ? slot_r : slot_f, plen, tlen, k_end, d ? cend[1] : cend[0], ak);
                            if (d == 0) {
                                dn[0] = f;
                                ak2[0] = ak;
                            } else {
                                dn[1] = f;
                                ak2[1] = ak;
                            }
                        }
                        done = dn[0];
                        done_r = dn[1];
                        akM_f = ak2[0];
                        akM_r = ak2[1];
                    } else {
                        const Range rf = launch_dir(0, score_f + 1, slot_f);
                        const Range rr = launch_dir(1, score_r + 1, slot_r);
                        cta_sync<NT>();
                        done = finish_dir(0, slot_f, rf);
                        akM_f = ring_meta[0 * ring_n + slot_f].akM;
                        done_r = finish_dir(1, slot_r, rr);
                        akM_r = ring_meta[1 * ring_n + slot_r].akM;
                    }
                    rotate_red();
                    if (status != ST_OK) break;
                    // commit forward
                    ++score_f;
                    cur_slot[0] = slot_f;
                    f_ak = max(f_ak, max(0, done ? 0 : akM_f));
                    last_forward = true;
                    if (AW_BIALIGN_PHASE1_END_REACHED_RETURNS && done) {
                        fb_end = true;
                        break;
                    }
                    if (f_ak + r_ak >= max_antidiagonal) {
                        rev_pending = true;
                        rev_pending_done = done_r;
                        break;
                    }
                    // commit reverse
                    ++score_r;
                    cur_slot[1] = slot_r;
                    r_ak = max(r_ak, max(0, done_r ? 0 : akM_r));
                    last_forward = false;
                    if (AW_BIALIGN_PHASE1_END_REACHED_RETURNS && done_r) {
                        fb_end = true;
                        break;
                    }
                }
                lap(0);
                if constexpr (VEC) {
                    if (!fb_end && status == ST_OK && first_full > max(1, score_r - (scope - 1))) {
                        // the wavefronts met earlier than predicted: redo this breakpoint search with full rows only (rare)
                        force_full = true;
                        cta_sync<NT>();
                        goto retry_breakpoint;
                    }
                }
                // one committed step of direction d (phase 2): cells, barrier, finish
                auto step_dir = [&](int d, int s) -> bool {
                    const int slot = next_slot(cur_slot[d]);
                    bool done;
                    if constexpr (VEC) {
                        int ak;
                        v_launch(d, d * ring_n, s, slot, cl_off * (NT / 32) + (tid >> 5), cl_n * (NT / 32), tid >> 5, false, true, d == 0 ? svd[0] : svd[1], k_end,
                                 d == 0 ? cend[0] : cend[1]);
                        step_sync(solo);
                        done = v_finish(d, d * ring_n, slot, plen, tlen, k_end, d == 0 ? cend[0] : cend[1], ak);
                    } else {
                        const Range r = launch_dir(d, s, slot);
                        cta_sync<NT>();
                        done = finish_dir(d, slot, r);
                    }
                    rotate_red();
                    cur_slot[d] = slot;
                    return done;
                };
                // ---- phase 2: advance until no better breakpoint is possible ----
                // Half-steps: the direction that stepped last acts as aligner 0 of wavefront_bialign_overlap, then the other
                // direction steps (one overlap / one step call site: instruction-cache footprint).
                const int gap_opening = AW_BIALIGN_GAP_OPENING(TWO, pen.o1, pen.o2);
                int a0 = last_forward ? 0 : 1;
                while (!fb_end && status == ST_OK) {
                    const int d0 = a0, d1 = 1 - a0;
                    const int s0 = d0 ? score_r : score_f, s1 = d1 ? score_r : score_f;
                    const int min1 = (s1 > scope - 1) ? s1 - (scope - 1) : 0;
                    if (s0 + min1 - gap_opening >= bp.score) break;
                    overlap(d0, d1, s0, s1);
                    bool done;
                    if (d1 == 1) ++score_r;
                    else ++score_f;
                    if (d1 == 1 && rev_pending) {  // computed speculatively in phase 1
                        rev_pending = false;
                        cur_slot[1] = next_slot(cur_slot[1]);
                        done = rev_pending_done;
                    } else {
                        done = step_dir(d1, d1 ? score_r : score_f);
                    }
                    if (AW_BIALIGN_PHASE2_END_REACHED_RETURNS && done) {
                        fb_end = true;
                        break;
                    }
                    a0 = d1;
                }
                lap(1);
                // cluster-wide sub-problem: nobody may write the rings again (CTA 0's next solo sub-problem) before every CTA
                // has finished its last overlap scan
                if (CL > 1 && !solo) cluster_sync_all();
                if (status != ST_OK) AW_DFS_FAIL;
                if (fb_end) {
                    do_base = true;
                } else {
                    ++w_bps;
                    if constexpr (SCORE) {  // the top-level breakpoint's score is the pair's optimal score
                        sc_pen = bp.score;
                        break;
                    }
                    const int bh = bp.off_f, bv = bp.off_f - bp.k_f;
                    if (bv < 0 || bv > plen || bh < 0 || bh > tlen || sp_n + 2 > MAX_STACK) {
                        status = ST_FAIL_WORKSPACE;
                        AW_DFS_FAIL;
                    }
                    // right half is pushed first so that the left half is aligned (and emitted) first
                    SubProblem right = {sp.pb + bv, sp.pe, sp.tb + bh, sp.te, bp.comp, sp.ce, bp.score_r};
                    SubProblem left = {sp.pb, sp.pb + bv, sp.tb, sp.tb + bh, sp.cb, bp.comp, bp.score_f};
                    stack[sp_n++] = right;
                    stack[sp_n++] = left;
                    cta_sync<NT>();
                    continue;
                }
            }

//@region base case
            // =========== K7: wavefront_bialign_base: full-history WFA + backtrace ===========
            {
                if (LEAFPAR && n_pending) {
                    // this base case (an END_REACHED fallback) comes after the pending leaves in CIGAR order: put it back, marked,
                    // and let the top of the loop flush them first
                    SubProblem again = sp;
                    again.rem = -1;
                    stack[sp_n++] = again;
                    flush_req = true;
                    cta_sync<NT>();
                    continue;
                }
                ++w_base;
                lap(5);
                const SeqView sv = VEC ? SeqView{reinterpret_cast<const uint32_t*>(pf2), reinterpret_cast<const uint32_t*>(tf2), sp.pb, sp.tb, plen, tlen, false}
                                       : SeqView{pw, tw, sp.pb, sp.tb, plen, tlen, false};
                hist_used = 0;
                // component block of a history wavefront: element (c,k) at ws[hist_off(off,width,clo,c) + k]
                auto hist_off = [&](int off, int width, int clo, int c) -> int { return hist_base + off + comp_idx(c) * width - clo; };
                auto slot_back = [&](int slot, int back) -> int {
                    const int s = slot - back;
                    return s < 0 ? s + ring_n : s;
                };
                StepOut so;
                int score = 0, slot = 0;
                bool done;
                if constexpr (VEC) {
                    int ak;
                    done = v_init_row(0, 0, true, sv, sp.cb, sp.ce, k_end, ak);
                    write_hist_meta(0, ring_meta[0]);
                    rotate_red();
                    while (!done) {
                        ++score;
                        slot = (slot + 1 == ring_n) ? 0 : slot + 1;
                        if (score >= hscores_cur) {
                            status = ST_FAIL_WORKSPACE;
                            break;
                        }
                        const VRange rg = v_launch(0, 0, score, slot, cl_off * (NT / 32) + (tid >> 5), cl_n * (NT / 32), tid >> 5, true, true, sv, k_end, sp.ce);
                        hist_used += (long long)NCOMP * rg.width;
                        step_sync(solo);
                        done = v_finish(0, 0, slot, plen, tlen, k_end, sp.ce, ak);
                        if (status != ST_OK) break;
                        write_hist_meta(score, ring_meta[slot]);
                        rotate_red();
                    }
                } else {
                {  // score 0
                    int* r = red[0][red_i];
                    SlotMeta& mt = ring_meta[0];
                    if (tid == 0) {
                        int m = 0;
                        if (sp.cb == AW_COMP_M) m = extend_cell<BITS>(sv, 0, 0);
                        ws[hist_off(0, 1, 0, sp.cb)] = to_ws<WS>(m);
                        if (sp.cb == AW_COMP_M && sp.ce == AW_COMP_M && k_end == 0) r[RED_END] = m;
                    }
                    cta_sync<NT>();
#pragma unroll
                    for (int c = 0; c < 5; ++c) {
                        so.lo[c] = (c == sp.cb) ? 0 : 1;
                        so.hi[c] = 0;
                    }
                    so.akM = so.akAll = INT_MIN;
                    so.endval = r[RED_END];
                    so.ambiguous = false;
                    store_meta(mt, so);
                    mt.off = hist_base;
                    mt.cstride = 1;
                    hist_used = NCOMP;
                    write_hist_meta(0, mt);
                    rotate_red();
                    done = end_reached(so, sp.ce, k_end, tlen);
                }
                while (!done) {
                    ++score;
                    slot = (slot + 1 == ring_n) ? 0 : slot + 1;
                    if (score >= P.hist_max_scores) {
                        status = ST_FAIL_WORKSPACE;
                        break;
                    }
                    In in[7];
                    auto fetch = [&](int c, int back) -> In {
                        In w;
                        if (score - back < 0) {
                            w.off = 0;
                            w.lo = 1;
                            w.hi = 0;
                            return w;
                        }
                        const SlotMeta& m = ring_meta[slot_back(slot, back)];
                        w.off = m.off + comp_idx(c) * m.cstride;
                        w.lo = m.lo[c];
                        w.hi = m.hi[c];
                        return w;
                    };
                    in[IN_MX] = fetch(AW_COMP_M, pen.x);
                    in[IN_MO1] = fetch(AW_COMP_M, pen.o1 + pen.e1);
                    in[IN_I1E] = fetch(AW_COMP_I1, pen.e1);
                    in[IN_D1E] = fetch(AW_COMP_D1, pen.e1);
                    if (TWO) {
                        in[IN_MO2] = fetch(AW_COMP_M, pen.o2 + pen.e2);
                        in[IN_I2E] = fetch(AW_COMP_I2, pen.e2);
                        in[IN_D2E] = fetch(AW_COMP_D2, pen.e2);
                    } else {
                        in[IN_MO2].off = in[IN_I2E].off = in[IN_D2E].off = 0;
                        in[IN_MO2].lo = in[IN_I2E].lo = in[IN_D2E].lo = 1;
                        in[IN_MO2].hi = in[IN_I2E].hi = in[IN_D2E].hi = 0;
                    }
                    int lo, hi;
                    limits(in, lo, hi);
                    SlotMeta& mt = ring_meta[slot];
                    ++w_steps;
                    if (lo > hi) {
                        set_empty(mt);
                        write_hist_meta(score, mt);
                        continue;
                    }
                    const int clo = lo;
                    const int width = hi - lo + 1;
                    if (hist_used + (long long)NCOMP * width > (long long)P.hist_ints) {
                        status = ST_FAIL_WORKSPACE;
                        break;
                    }
                    const int off = (int)hist_used;
                    hist_used += (long long)NCOMP * width;
                    int out[5];
#pragma unroll
                    for (int c = 0; c < 5; ++c) out[c] = hist_off(off, width, clo, (TWO || c == AW_COMP_M || c == AW_COMP_I1 || c == AW_COMP_D1) ? c : AW_COMP_M);
                    wf_cells<NT, BITS, TWO, WS>(ws, in, out, lo, hi, sv, k_end, sp.ce, red[0][red_i]);
                    cta_sync<NT>();
                    wf_finish<TWO>(red[0][red_i], lo, hi, so);
                    if (so.ambiguous) wf_rescan<NT, TWO, WS>(ws, out, lo, hi, plen, tlen, red[0][red_i], so, tid, NT, false);
                    w_cells += (unsigned long long)(hi - lo + 1) * NCOMP;
                    store_meta(mt, so);
                    mt.off = hist_off(off, width, clo, AW_COMP_M);
                    mt.cstride = width;
                    write_hist_meta(score, mt);
                    rotate_red();
                    done = end_reached(so, sp.ce, k_end, tlen);
                }
                }
                if (CL > 1 && !solo) cluster_sync_all();  // the whole history is in place (and see the note after phase 2)
                if (status != ST_OK) AW_DFS_FAIL;
                if constexpr (SCORE) {  // the score at which the end cell is reached is the pair's score: no backtrace
                    sc_pen = score;
                    w_maxbase = max(w_maxbase, (unsigned)score);
                    break;
                }
                if (CL > 1 && crank != 0) continue;  // the backtrace and the CIGAR belong to CTA 0
                w_maxbase = max(w_maxbase, (unsigned)score);
                cta_sync<NT>();  // history + meta visible to warp 0
                lap(2);

//@region backtrace
                // ---- wavefront_backtrace_affine by warp 0: lanes evaluate the candidates ----
                unsigned n_leaf = 0;  // runs pushed (reverse order) into leaf_runs; uniform within warp 0
                if (tid < 32) {
                    n_leaf = bt_run(sp.ce, score, plen, tlen, k_end);
                    if (tid == 0) {
                        s_acc[0] = n_leaf;
                        s_acc[1] = (unsigned long long)status;
                    }
                }
                cta_sync<NT>();
                n_leaf = (unsigned)s_acc[0];
                if (s_acc[1] != ST_OK) status = (int)s_acc[1];
                if (status != ST_OK) AW_DFS_FAIL_CTA0;
                // append the leaf's runs (stored back to front) to the pair's CIGAR
                unsigned base_n = s_nruns, skip = 0;
                if (n_leaf > 0 && base_n > 0 && (pair_runs[base_n - 1] & 3u) == (leaf_runs[n_leaf - 1] & 3u)) skip = 1;
                cta_sync<NT>();
                if (base_n + n_leaf > P.runs_cap) {
                    status = ST_FAIL_WORKSPACE;
                    AW_DFS_FAIL_CTA0;
                }
                if (tid == 0 && skip) pair_runs[base_n - 1] += leaf_runs[n_leaf - 1] & ~3u;
                for (unsigned i = skip + tid; i < n_leaf; i += NT) pair_runs[base_n + i - skip] = leaf_runs[n_leaf - 1 - i];
                if (tid == 0) s_nruns = base_n + n_leaf - skip;
                cta_sync<NT>();
                lap(3);
            }
        }  // DFS over sub-problems

//@region emit
        // =========== K8: statistics, score, PAF text ===========
        cta_sync<NT>();
        if (CL > 1 && crank != 0) continue;  // CTA 0 owns the pair's CIGAR; the others go and wait for the next pair
        if constexpr (SCORE) {
            if (tid == 0) {
                long long p = sc_pen;
                if (PLEN == 0 || TLEN == 0) {  // one pure gap, or nothing
                    const long long len = PLEN + TLEN;
                    p = len ? pen.o1 + len * pen.e1 : 0;
                    if (TWO && len) p = min(p, pen.o2 + len * pen.e2);
                }
                // with match_score M < 0 the wavefronts ran on the shifted penalties (aw_wfa2_compat.h): every column gives up
                // M/2 per consumed character, so the user's penalty is exactly (P' + M (plen + tlen)) / 2
                if (pen.smatch < 0) p = (p + (long long)pen.smatch * (PLEN + TLEN)) / 2;
                AwPairOut o;
                memset(&o, 0, sizeof(o));
                o.status = (status == ST_OK) ? AW_OK : AW_EWORKSPACE;
                o.score = (status == ST_OK) ? (int32_t)-p : INT_MAX;
                o.is_reverse = is_rev;
                o.cells = w_cells;
                o.steps = w_steps;
                o.n_breakpoints = w_bps;
                o.n_base = w_base;
                o.max_base_score = w_maxbase;
                for (int i = 0; i < 6; ++i) o.cyc[i] = cyc[i];
                P.out[pair_i] = o;
            }
            cta_sync<NT>();
            continue;
        }
        const unsigned nruns = (status == ST_OK) ? s_nruns : 0;
        if (tid < 8) s_acc[tid] = 0;
        cta_sync<NT>();
        {
            unsigned long long cnt[4] = {0, 0, 0, 0}, textlen = 0, penalty = 0;
            for (unsigned r = tid; r < nruns; r += NT) {
                const unsigned run = pair_runs[r], op = run & 3u;
                const unsigned long long len = run >> 2;
                cnt[op] += len;
                textlen += ndigits(len) + 1;
                // score of the final CIGAR under the user's own penalties (they differ from pen.x ... when match_score < 0)
                if (op == AW_OP_X) penalty += len * pen.sx;
                else if (op != AW_OP_M) {
                    unsigned long long c1 = pen.so1 + len * pen.se1;
                    if (TWO) c1 = min(c1, pen.so2 + len * (unsigned long long)pen.se2);
                    penalty += c1;
                }
            }
            unsigned long long vals[6] = {cnt[0], cnt[1], cnt[2], cnt[3], textlen, penalty};
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                unsigned long long v = vals[i];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                if ((tid & 31) == 0 && v) atomicAdd(&s_acc[i], v);
            }
        }
        cta_sync<NT>();
        const unsigned long long n_m = s_acc[0], n_x = s_acc[1], n_i = s_acc[2], n_d = s_acc[3], cg_len = s_acc[4], penalty = s_acc[5];
        const unsigned long long q_end = n_m + n_x + n_d, t_end = n_m + n_x + n_i;  // parse_cigar_lengths
        const unsigned long long block_len = max(q_end, t_end);
        const unsigned long long aln_len = n_m + n_x;                               // count_cigar_operations
        const uint32_t qid0 = P.id_off[pr.query_idx], qid1 = P.id_off[pr.query_idx + 1];
        const uint32_t tid0 = P.id_off[pr.target_idx], tid1 = P.id_off[pr.target_idx + 1];
        const bool want_paf = !(P.flags & AW_FLAG_NO_PAF);
        const bool count_only = (P.flags & AW_KFLAG_COUNT_ONLY) != 0;
        // header: q qlen qs qe strand t tlen ts te matches block 60 gi:f:x.xxxxxx cg:Z:
        const unsigned hdr_len = (qid1 - qid0) + 1 + ndigits(PLEN) + 1 + 1 + 1 + ndigits(q_end) + 1 + 1 + 1 + (tid1 - tid0) + 1 + ndigits(TLEN) + 1 + 1 + 1 +
                                 ndigits(t_end) + 1 + ndigits(n_m) + 1 + ndigits(block_len) + 1 + 2 + 1 + 5 + 8 + 1 + 5;
        // a failed pair reserves nothing, so the text arena stays gap-free (AW_FLAG_PAF_BLOCKS hands it out as one block)
        const unsigned long long line_len = (count_only || status != ST_OK) ? 0 : (want_paf ? hdr_len + cg_len : cg_len);
        const unsigned long long nl = (line_len && (P.flags & AW_FLAG_PAF_BLOCKS)) ? 1 : 0;  // '\n' after the line, not counted in paf_len
        const unsigned long long nbytes = (status == ST_OK && !count_only && (P.flags & AW_FLAG_CIGAR_BYTES)) ? (n_m + n_x + n_i + n_d) : 0;
        if (tid == 0) {
            s_text_off = atomicAdd(P.text_cursor, line_len + nl);
            s_bytes_off = nbytes ? atomicAdd(P.bytes_cursor, nbytes) : 0ull;
        }
        cta_sync<NT>();
        const unsigned long long text_off = s_text_off, bytes_off = s_bytes_off;
        if (status == ST_OK && (text_off + line_len + nl > P.text_cap || bytes_off + nbytes > P.bytes_cap)) status = ST_FAIL_WORKSPACE;
        if (status == ST_OK && !count_only) {
            char* line = P.text + text_off;
            char* cg = line;
            if (nl && tid == 32 % NT) line[line_len] = '\n';
            if (want_paf) {
                cg = line + hdr_len;
                if (tid == 0) {
                    char* p = line;
                    for (uint32_t i = qid0; i < qid1; ++i) *p++ = P.ids[i];
                    *p++ = '\t';
                    p = put_u64(p, (unsigned long long)PLEN);
                    *p++ = '\t';
                    *p++ = '0';
                    *p++ = '\t';
                    p = put_u64(p, q_end);
                    *p++ = '\t';
                    *p++ = is_rev ? '-' : '+';
                    *p++ = '\t';
                    for (uint32_t i = tid0; i < tid1; ++i) *p++ = P.ids[i];
                    *p++ = '\t';
                    p = put_u64(p, (unsigned long long)TLEN);
                    *p++ = '\t';
                    *p++ = '0';
                    *p++ = '\t';
                    p = put_u64(p, t_end);
                    *p++ = '\t';
                    p = put_u64(p, n_m);
                    *p++ = '\t';
                    p = put_u64(p, block_len);
                    *p++ = '\t';
                    *p++ = '6';
                    *p++ = '0';
                    *p++ = '\t';
                    const char gi[5] = {'g', 'i', ':', 'f', ':'};
                    for (int i = 0; i < 5; ++i) *p++ = gi[i];
                    const unsigned micro = identity_micro(n_m, aln_len);
                    *p++ = (char)('0' + micro / 1000000u);
                    *p++ = '.';
                    unsigned fr = micro % 1000000u;
                    for (int i = 5; i >= 0; --i) {
                        p[i] = (char)('0' + fr % 10u);
                        fr /= 10u;
                    }
                    p += 6;
                    *p++ = '\t';
                    const char cz[5] = {'c', 'g', ':', 'Z', ':'};
                    for (int i = 0; i < 5; ++i) *p++ = cz[i];
                }
            }
            // cigar_bytes_to_string: contiguous chunk of runs per thread, offsets by block scan
            const unsigned chunk = (nruns + NT - 1) / NT;
            const unsigned r0 = min(nruns, tid * chunk), r1 = min(nruns, r0 + chunk);
            unsigned long long my_text = 0, my_cols = 0;
            for (unsigned r = r0; r < r1; ++r) {
                const unsigned run = pair_runs[r];
                my_text += ndigits(run >> 2) + 1;
                my_cols += run >> 2;
            }
            unsigned long long total;
            unsigned long long toff = block_excl_scan<NT>(my_text, scanbuf, &total);
            {
                char* p = cg + toff;
                for (unsigned r = r0; r < r1; ++r) {
                    const unsigned run = pair_runs[r], op = run & 3u;
                    p = put_u64(p, run >> 2);
                    *p++ = (op == AW_OP_M) ? '=' : (op == AW_OP_X) ? 'X' : (op == AW_OP_I) ? 'D' : 'I';
                }
            }
            if (nbytes) {
                unsigned long long boff = block_excl_scan<NT>(my_cols, scanbuf, &total);
                uint8_t* b = P.bytes + bytes_off + boff;
                for (unsigned r = r0; r < r1; ++r) {
                    const unsigned run = pair_runs[r], op = run & 3u, len = run >> 2;
                    const uint8_t ch = (op == AW_OP_M) ? 'M' : (op == AW_OP_X) ? 'X' : (op == AW_OP_I) ? 'I' : 'D';
                    for (unsigned i = 0; i < len; ++i) *b++ = ch;
                }
            }
        }
        lap(4);
        if (tid == 0) {
            AwPairOut o;
            o.status = (status == ST_OK) ? AW_OK : AW_EWORKSPACE;
            o.score = (status == ST_OK) ? (int32_t)(-(long long)penalty - (long long)pen.smatch * (long long)n_m) : INT_MAX;
            o.is_reverse = is_rev;
            o.nruns = nruns;
            o.n_m = n_m;
            o.n_x = n_x;
            o.n_i = n_i;
            o.n_d = n_d;
            o.paf_off = text_off;
            o.paf_len = (uint32_t)line_len;
            o.cg_off = want_paf ? hdr_len : 0;
            o.bytes_off = bytes_off;
            o.runs_off = 0;
            o.cells = w_cells;
            o.steps = w_steps;
            o.n_breakpoints = w_bps;
            o.n_base = w_base;
            o.max_base_score = w_maxbase;
            for (int i = 0; i < 6; ++i) o.cyc[i] = cyc[i];
            P.out[pair_i] = o;
        }
        cta_sync<NT>();
    }
    if constexpr (CL > 1) cluster_sync_all();  // no CTA may exit while another one can still read its shared memory
}

template <int NT, int BITS, bool TWO, class WS, int CL = 1>
__global__ void __launch_bounds__(NT, AW_CTAS_PER_SM(NT)) aw_align_kernel(const KParams P) {
    align_driver<NT, BITS, TWO, WS, CL, false>(P);
}
template <int NT, int BITS, bool TWO, class WS, int CL = 1>
__global__ void __launch_bounds__(NT, AW_CTAS_PER_SM(NT)) aw_score_kernel(const KParams P) {
    align_driver<NT, BITS, TWO, WS, CL, true>(P);
}
#undef AW_DFS_FAIL
#undef AW_DFS_FAIL_CTA0

}  // namespace awk
