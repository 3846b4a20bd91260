//! Raw bindings of `include/allwave_cuda.h` (ABI version 1).  One item per C declaration, same order as the header.
//! What each entry point replaces in allwave is documented in the header (file:line into the reference).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const AW_ABI_VERSION: c_int = 1;

// aw_status
pub const AW_OK: c_int = 0;
pub const AW_EINVAL: c_int = -1;
pub const AW_ENODEVICE: c_int = -2;
pub const AW_ECUDA: c_int = -3;
pub const AW_ENOMEM: c_int = -4;
pub const AW_EUNSUPPORTED: c_int = -5;
pub const AW_EWORKSPACE: c_int = -6;
pub const AW_ECALLBACK: c_int = -7;
pub const AW_EALIGN: c_int = -8;

// aw_orientation_mode
pub const AW_ORIENT_MASH: c_int = 0;
pub const AW_ORIENT_WFA: c_int = 1;
pub const AW_ORIENT_FORWARD: c_int = 2;

// flags
pub const AW_FLAG_CIGAR_BYTES: u32 = 1;
pub const AW_FLAG_ORDERED: u32 = 2;
pub const AW_FLAG_NO_PAF: u32 = 4;
pub const AW_FLAG_PAF_BLOCKS: u32 = 8;
pub const AW_FLAG_SCORE_ONLY: u32 = 16;

// aw_memory_mode / aw_alignment_scope / aw_alignment_span / aw_heuristic / aw_alignment_status (lib_wfa2 names)
pub const AW_MEMORY_HIGH: c_int = 0;
pub const AW_MEMORY_MEDIUM: c_int = 1;
pub const AW_MEMORY_LOW: c_int = 2;
pub const AW_MEMORY_ULTRALOW: c_int = 3;
pub const AW_SCOPE_SCORE: c_int = 0;
pub const AW_SCOPE_ALIGNMENT: c_int = 1;
pub const AW_SPAN_END2END: c_int = 0;
pub const AW_SPAN_ENDSFREE: c_int = 1;
pub const AW_HEURISTIC_NONE: c_int = 0;
pub const AW_ALIGN_COMPLETED: c_int = 0;
pub const AW_ALIGN_PARTIAL: c_int = 1;
pub const AW_ALIGN_MAX_STEPS: c_int = -100;
pub const AW_ALIGN_OOM: c_int = -200;
pub const AW_ALIGN_UNATTAINABLE: c_int = -300;
pub const AW_ALIGN_UNDEFINED: c_int = -1;

/// mirrors `AlignmentParams` (src/types.rs:37-45)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aw_params {
    pub match_score: i32,
    pub mismatch_penalty: i32,
    pub gap_open: i32,
    pub gap_extend: i32,
    pub gap2_open: i32,
    pub gap2_extend: i32,
    pub has_gap2_open: u8,
    pub has_gap2_extend: u8,
}

/// one directed pair (src/iterator.rs:40-46)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct aw_pair {
    pub query_idx: u32,
    pub target_idx: u32,
}

/// mirrors `AlignmentResult` (src/types.rs:14-33) plus the strings the CLI derives from it
#[repr(C)]
pub struct aw_result {
    pub query_idx: u64,
    pub target_idx: u64,
    pub query_start: u64,
    pub query_end: u64,
    pub target_start: u64,
    pub target_end: u64,
    pub is_reverse: u8,
    pub status: i32,
    pub score: i32,
    pub num_matches: u64,
    pub alignment_length: u64,
    pub cigar_bytes: *const u8,
    pub cigar_len: u64,
    pub cg: *const c_char,
    pub cg_len: u64,
    pub paf: *const c_char,
    pub paf_len: u64,
}

#[repr(C)]
pub struct aw_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct aw_batch {
    _private: [u8; 0],
}
#[repr(C)]
pub struct aw_aligner {
    _private: [u8; 0],
}

pub type aw_result_cb = Option<unsafe extern "C" fn(result: *const aw_result, user: *mut c_void) -> c_int>;
pub type aw_chunk_source = Option<unsafe extern "C" fn(user: *mut c_void, pairs: *mut *const aw_pair) -> u64>;
pub type aw_paf_block_cb = Option<unsafe extern "C" fn(text: *const c_char, len: u64, n_lines: u64, user: *mut c_void) -> c_int>;

extern "C" {
    pub fn aw_abi_version() -> c_int;
    pub fn aw_strerror(status: c_int) -> *const c_char;
    pub fn aw_last_error() -> *const c_char;
    pub fn aw_device_count() -> c_int;

    pub fn aw_create(device: c_int, out: *mut *mut aw_ctx) -> c_int;
    pub fn aw_destroy(ctx: *mut aw_ctx);
    pub fn aw_set_option(ctx: *mut aw_ctx, key: *const c_char, value: i64) -> c_int;
    pub fn aw_trim_cache();

    pub fn aw_load_sequences(ctx: *mut aw_ctx, n: u32, seqs: *const *const u8, lens: *const u64, ids: *const *const c_char) -> c_int;
    pub fn aw_num_sequences(ctx: *const aw_ctx) -> u32;
    pub fn aw_set_orientation_params(ctx: *mut aw_ctx, params: *const aw_params) -> c_int;

    pub fn aw_align_pairs(ctx: *mut aw_ctx, params: *const aw_params, orientation_mode: c_int, pairs: *const aw_pair, npairs: u64, flags: u32,
                          cb: aw_result_cb, user: *mut c_void) -> c_int;
    pub fn aw_align_stream(ctx: *mut aw_ctx, params: *const aw_params, orientation_mode: c_int, flags: u32, next: aw_chunk_source,
                           next_user: *mut c_void, cb: aw_result_cb, block_cb: aw_paf_block_cb, user: *mut c_void) -> c_int;

    pub fn aw_batch_create(ctx: *mut aw_ctx, params: *const aw_params, orientation_mode: c_int, pairs: *const aw_pair, npairs: u64, flags: u32,
                           out: *mut *mut aw_batch) -> c_int;
    pub fn aw_batch_launch(ctx: *mut aw_ctx, batch: *mut aw_batch, stream: *mut c_void) -> c_int;
    pub fn aw_batch_fetch(ctx: *mut aw_ctx, batch: *mut aw_batch, cb: aw_result_cb, user: *mut c_void) -> c_int;
    pub fn aw_batch_stats(ctx: *mut aw_ctx, batch: *mut aw_batch, out: *mut u64) -> c_int;
    pub fn aw_batch_kernel_ms(ctx: *mut aw_ctx, batch: *mut aw_batch, out_ms: *mut f32) -> c_int;
    pub fn aw_batch_debug_cycles(ctx: *mut aw_ctx, batch: *mut aw_batch, out: *mut u64) -> c_int;
    pub fn aw_batch_destroy(ctx: *mut aw_ctx, batch: *mut aw_batch);

    pub fn aw_orient_pairs(ctx: *mut aw_ctx, pairs: *const aw_pair, npairs: u64, out_is_reverse: *mut u8) -> c_int;
    pub fn aw_estimate_divergence(ctx: *mut aw_ctx, pairs: *const aw_pair, npairs: u64, out: *mut f32) -> c_int;
    pub fn aw_get_sketch(ctx: *mut aw_ctx, idx: u32, reverse_complement: c_int, canonical: c_int, k: c_int, sketch_size: u32, out: *mut u64,
                         out_n: *mut u32) -> c_int;
    pub fn aw_mash_jaccard_counts(ctx: *mut aw_ctx, k: c_int, sketch_size: u32, inter: *mut u32, uni: *mut u32) -> c_int;

    pub fn aw_aligner_new_affine(ctx: *mut aw_ctx, match_: i32, mismatch: i32, gap_opening: i32, gap_extension: i32, memory_mode: c_int,
                                 out: *mut *mut aw_aligner) -> c_int;
    pub fn aw_aligner_new_affine2p(ctx: *mut aw_ctx, match_: i32, mismatch: i32, gap_opening1: i32, gap_extension1: i32, gap_opening2: i32,
                                   gap_extension2: i32, memory_mode: c_int, out: *mut *mut aw_aligner) -> c_int;
    pub fn aw_aligner_set_alignment_scope(a: *mut aw_aligner, scope: c_int) -> c_int;
    pub fn aw_aligner_set_alignment_span(a: *mut aw_aligner, span: c_int) -> c_int;
    pub fn aw_aligner_set_heuristic(a: *mut aw_aligner, heuristic: c_int) -> c_int;
    pub fn aw_aligner_get_memory_mode(a: *const aw_aligner) -> c_int;
    pub fn aw_aligner_align(a: *mut aw_aligner, pattern: *const u8, pattern_len: i32, text: *const u8, text_len: i32) -> c_int;
    pub fn aw_aligner_score(a: *const aw_aligner) -> i32;
    pub fn aw_aligner_cigar(a: *const aw_aligner, len: *mut u64) -> *const u8;
    pub fn aw_aligner_delete(a: *mut aw_aligner);
}
