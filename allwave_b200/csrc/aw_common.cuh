// aw_common.cuh -- shared device/host definitions of liballwave_cuda (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/allwave_cuda.h"
#include "../../include/aw_wfa2_compat.h"

#define AW_NULLV AW_OFFSET_NULL

// ---- sequence store (HBM layout, see DESIGN.md "Data layout") ------------------------------
// Every sequence i owns two slots: 2*i = as given, 2*i+1 = reverse_complement(seq)
// (src/alignment.rs:178-190).  Each slot has an ASCII copy (16-byte aligned, 16 guard bytes
// either side) and, a 2-bit packed copy (A=0 C=1 G=2 T=3, 16 bases per u32 word, little end
// first, 4 guard words either side).  `clean` is 1 iff every byte is upper-case ACGT, i.e.
// iff 2-bit equality == byte equality (SURVEY fact 8).
struct AwSlot {
    uint64_t ascii_off;   // byte offset of base 0 in the ASCII buffer
    uint64_t packed_off;  // word offset of base 0 in the packed buffer
    uint32_t len;
    uint32_t clean;
};

// WFA2 penalties after create_wfa_aligner's mode mapping (src/alignment.rs:263-289)
struct AwPen {
    int x, o1, e1, o2, e2;  // what the wavefronts run on: the user's penalties, or AW_SHIFT_* of them when match_score < 0
    int two_piece;
    int scope;  // max_score_scope = max(x, o1+e1, o2+e2) + 1
    // the user's own penalties, for the reported score of the final CIGAR (cigar_score_gap_affine*): equal to the above when
    // match_score == 0
    int sx, so1, se1, so2, se2, smatch;
};

// CIGAR run: (len << 2) | op, op: 0=M 1=X 2=I 3=D (WFA2 letters)
#define AW_OP_M 0u
#define AW_OP_X 1u
#define AW_OP_I 2u
#define AW_OP_D 3u

// per-pair fixed-size output record (device -> host)
struct AwPairOut {
    int32_t status;       // AW_OK / AW_EWORKSPACE (retry) / AW_EALIGN
    int32_t score;        // -(penalty)
    uint32_t is_reverse;
    uint32_t nruns;
    uint64_t n_m, n_x, n_i, n_d;  // column counts per WFA2 op
    uint64_t paf_off;     // into the text arena
    uint32_t paf_len;
    uint32_t cg_off;      // offset of the cg:Z: value inside the PAF line
    uint64_t bytes_off;   // into the cigar-bytes arena (when requested)
    uint64_t runs_off;    // into the runs arena (when requested)
    // work counters
    uint64_t cells;       // computed (score,diagonal) cells x components
    uint32_t steps;
    uint32_t n_breakpoints;
    uint32_t n_base;
    uint32_t max_base_score;
    // device-clock breakdown (thread 0): phase 1, phase 2, base compute, backtrace, emission
    unsigned long long cyc[6];
};

// where the cs:Z: value of a pair (AW_FLAG_CS) lies in the tag arena
struct AwCsOut {
    unsigned long long off, len;
};

#define AW_CUDA_CHECK(call)                                                         \
    do {                                                                            \
        cudaError_t _e = (call);                                                    \
        if (_e != cudaSuccess) {                                                    \
            aw_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return AW_ECUDA;                                                        \
        }                                                                           \
    } while (0)

void aw_set_error(const char* fmt, ...);
