"""ctypes binding of liballwave_cuda.so (include/allwave_cuda.h).

Thin by design: every call goes straight through the C ABI a Rust/cgo/JNI binding would use.
The product path fails loudly when the CUDA library is missing or no B200 is visible; there is
no CPU fallback and nothing here imports oracle/.
"""
import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_PKG, "liballwave_cuda.so")

AW_OK = 0
AW_EINVAL, AW_ENODEVICE, AW_ECUDA, AW_ENOMEM, AW_EUNSUPPORTED, AW_EWORKSPACE, AW_ECALLBACK, AW_EALIGN = -1, -2, -3, -4, -5, -6, -7, -8
AW_ORIENT_MASH, AW_ORIENT_WFA, AW_ORIENT_FORWARD = 0, 1, 2
AW_FLAG_CIGAR_BYTES, AW_FLAG_ORDERED, AW_FLAG_NO_PAF, AW_FLAG_PAF_BLOCKS, AW_FLAG_SCORE_ONLY = 1, 2, 4, 8, 16
AW_FLAG_CS, AW_FLAG_CS_LONG = 32, 64
AW_MEMORY_HIGH, AW_MEMORY_MEDIUM, AW_MEMORY_LOW, AW_MEMORY_ULTRALOW = 0, 1, 2, 3
AW_SCOPE_SCORE, AW_SCOPE_ALIGNMENT = 0, 1

EXPORTS = [
    "aw_abi_version", "aw_strerror", "aw_last_error", "aw_device_count", "aw_create", "aw_destroy", "aw_set_option",
    "aw_load_sequences", "aw_num_sequences", "aw_set_orientation_params", "aw_align_pairs", "aw_batch_create", "aw_batch_launch", "aw_batch_fetch",
    "aw_batch_stats", "aw_batch_kernel_ms", "aw_batch_debug_cycles", "aw_batch_destroy", "aw_orient_pairs", "aw_get_sketch", "aw_mash_jaccard_counts",
    "aw_aligner_new_affine", "aw_aligner_new_affine2p", "aw_aligner_set_alignment_scope", "aw_aligner_set_alignment_span",
    "aw_aligner_set_heuristic", "aw_aligner_get_memory_mode", "aw_aligner_align", "aw_aligner_score", "aw_aligner_cigar",
    "aw_aligner_delete", "aw_align_stream", "aw_estimate_divergence", "aw_trim_cache",
]


class AwParams(C.Structure):
    _fields_ = [
        ("match_score", C.c_int32),
        ("mismatch_penalty", C.c_int32),
        ("gap_open", C.c_int32),
        ("gap_extend", C.c_int32),
        ("gap2_open", C.c_int32),
        ("gap2_extend", C.c_int32),
        ("has_gap2_open", C.c_uint8),
        ("has_gap2_extend", C.c_uint8),
    ]


class AwPair(C.Structure):
    _fields_ = [("query_idx", C.c_uint32), ("target_idx", C.c_uint32)]


class AwResult(C.Structure):
    _fields_ = [
        ("query_idx", C.c_uint64),
        ("target_idx", C.c_uint64),
        ("query_start", C.c_uint64),
        ("query_end", C.c_uint64),
        ("target_start", C.c_uint64),
        ("target_end", C.c_uint64),
        ("is_reverse", C.c_uint8),
        ("status", C.c_int32),
        ("score", C.c_int32),
        ("num_matches", C.c_uint64),
        ("alignment_length", C.c_uint64),
        ("cigar_bytes", C.POINTER(C.c_uint8)),
        ("cigar_len", C.c_uint64),
        ("cg", C.POINTER(C.c_char)),
        ("cg_len", C.c_uint64),
        ("paf", C.POINTER(C.c_char)),
        ("paf_len", C.c_uint64),
        ("cs", C.POINTER(C.c_char)),
        ("cs_len", C.c_uint64),
    ]


RESULT_CB = C.CFUNCTYPE(C.c_int, C.POINTER(AwResult), C.c_void_p)
CHUNK_SOURCE = C.CFUNCTYPE(C.c_uint64, C.c_void_p, C.POINTER(C.POINTER(AwPair)))
PAF_BLOCK_CB = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_char), C.c_uint64, C.c_uint64, C.c_void_p)

_lib = None


class AllwaveError(RuntimeError):
    def __init__(self, status, where):
        self.status = status
        L = _lib
        msg = L.aw_strerror(status).decode() if L else "?"
        detail = L.aw_last_error().decode() if L else ""
        super().__init__(f"{where}: {msg} ({status}) {detail}")


def so_path():
    return _SO


def build(verbose=False):
    """compile liballwave_cuda.so for sm_100a in-tree (nvcc cross-compiles without a GPU)"""
    subprocess.check_call(["make", "-s", "-C", os.path.join(_PKG, "csrc")])
    subprocess.check_call(["make", "-s", "-C", os.path.join(_PKG, "host")])


def lib():
    global _lib
    if _lib is not None:
        return _lib
    # dev aid: ALLWAVE_CUDA_LIB selects another build of the same library (kernel tuning variants)
    _so = os.environ.get("ALLWAVE_CUDA_LIB", _SO)
    if not os.path.exists(_so):
        raise ImportError(f"{_so} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    L = C.CDLL(_so)
    vp = C.c_void_p
    L.aw_abi_version.restype = C.c_int
    L.aw_strerror.argtypes = [C.c_int]
    L.aw_strerror.restype = C.c_char_p
    L.aw_last_error.restype = C.c_char_p
    L.aw_device_count.restype = C.c_int
    L.aw_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.aw_destroy.argtypes = [vp]
    L.aw_destroy.restype = None
    L.aw_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.aw_load_sequences.argtypes = [vp, C.c_uint32, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.POINTER(C.c_char_p)]
    L.aw_num_sequences.argtypes = [vp]
    L.aw_num_sequences.restype = C.c_uint32
    L.aw_set_orientation_params.argtypes = [vp, C.POINTER(AwParams)]
    L.aw_align_pairs.argtypes = [vp, C.POINTER(AwParams), C.c_int, C.POINTER(AwPair), C.c_uint64, C.c_uint32, RESULT_CB, vp]
    L.aw_align_stream.argtypes = [vp, C.POINTER(AwParams), C.c_int, C.c_uint32, CHUNK_SOURCE, vp, RESULT_CB, PAF_BLOCK_CB, vp]
    L.aw_estimate_divergence.argtypes = [vp, C.POINTER(AwPair), C.c_uint64, C.POINTER(C.c_float)]
    L.aw_trim_cache.restype = None
    L.aw_batch_create.argtypes = [vp, C.POINTER(AwParams), C.c_int, C.POINTER(AwPair), C.c_uint64, C.c_uint32, C.POINTER(vp)]
    L.aw_batch_launch.argtypes = [vp, vp, vp]
    L.aw_batch_fetch.argtypes = [vp, vp, RESULT_CB, vp]
    L.aw_batch_stats.argtypes = [vp, vp, C.POINTER(C.c_uint64)]
    L.aw_batch_kernel_ms.argtypes = [vp, vp, C.POINTER(C.c_float)]
    L.aw_batch_debug_cycles.argtypes = [vp, vp, C.POINTER(C.c_uint64)]
    L.aw_batch_destroy.argtypes = [vp, vp]
    L.aw_batch_destroy.restype = None
    L.aw_orient_pairs.argtypes = [vp, C.POINTER(AwPair), C.c_uint64, C.POINTER(C.c_uint8)]
    L.aw_get_sketch.argtypes = [vp, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
    L.aw_mash_jaccard_counts.argtypes = [vp, C.c_int, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.aw_aligner_new_affine.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.POINTER(vp)]
    L.aw_aligner_new_affine2p.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.POINTER(vp)]
    for f in (L.aw_aligner_set_alignment_scope, L.aw_aligner_set_alignment_span, L.aw_aligner_set_heuristic):
        f.argtypes = [vp, C.c_int]
    L.aw_aligner_get_memory_mode.argtypes = [vp]
    L.aw_aligner_align.argtypes = [vp, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32]
    L.aw_aligner_score.argtypes = [vp]
    L.aw_aligner_score.restype = C.c_int32
    L.aw_aligner_cigar.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.aw_aligner_cigar.restype = C.POINTER(C.c_uint8)
    L.aw_aligner_delete.argtypes = [vp]
    L.aw_aligner_delete.restype = None
    _lib = L
    return L


def check(status, where):
    if status != AW_OK:
        raise AllwaveError(status, where)


def make_params(match=0, mismatch=5, gap_open=8, gap_extend=2, gap2_open=24, gap2_extend=1):
    p = AwParams(match, mismatch, gap_open, gap_extend, 0, 0, 0, 0)
    if gap2_open is not None:
        p.gap2_open, p.has_gap2_open = gap2_open, 1
    if gap2_extend is not None:
        p.gap2_extend, p.has_gap2_extend = gap2_extend, 1
    return p


def make_pairs(pairs):
    arr = (AwPair * max(1, len(pairs)))()
    for i, (a, b) in enumerate(pairs):
        arr[i].query_idx, arr[i].target_idx = a, b
    return arr


def result_to_dict(r, want_bytes=True):
    d = {
        "query_idx": r.query_idx, "target_idx": r.target_idx,
        "query_start": r.query_start, "query_end": r.query_end,
        "target_start": r.target_start, "target_end": r.target_end,
        "is_reverse": bool(r.is_reverse), "status": r.status, "score": r.score,
        "num_matches": r.num_matches, "alignment_length": r.alignment_length,
        "cg": C.string_at(r.cg, r.cg_len).decode() if r.cg_len else "",
        "paf": C.string_at(r.paf, r.paf_len).decode() if r.paf_len else "",
        "cs": C.string_at(r.cs, r.cs_len).decode() if r.cs_len else "",
    }
    if want_bytes and r.cigar_len and r.cigar_bytes:
        d["cigar_bytes"] = C.string_at(r.cigar_bytes, r.cigar_len)
    else:
        d["cigar_bytes"] = b""
    return d


class Context:
    """one aw_ctx (one GPU)"""

    def __init__(self, device=0):
        L = lib()
        h = C.c_void_p()
        check(L.aw_create(device, C.byref(h)), "aw_create")
        self._h = h
        self.n = 0

    def close(self):
        if self._h:
            lib().aw_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        check(lib().aw_set_option(self._h, key.encode(), int(value)), f"aw_set_option({key})")

    def load_sequences(self, ids, seqs):
        n = len(seqs)
        sa = (C.c_char_p * max(1, n))(*seqs)
        la = (C.c_uint64 * max(1, n))(*[len(s) for s in seqs])
        ia = (C.c_char_p * max(1, n))(*[i.encode() if isinstance(i, str) else i for i in ids])
        check(lib().aw_load_sequences(self._h, n, sa, la, ia), "aw_load_sequences")
        self.n = n

    def align_pairs(self, params, pairs, orientation=AW_ORIENT_MASH, flags=0, callback=None):
        """e2e host API; returns list of result dicts (pair order) unless callback is given"""
        out = []
        want_bytes = bool(flags & AW_FLAG_CIGAR_BYTES)

        def _cb(rp, _u):
            d = result_to_dict(rp.contents, want_bytes)
            if callback is not None:
                return int(bool(callback(d)))
            out.append(d)
            return 0

        cb = RESULT_CB(_cb)
        arr = make_pairs(pairs)
        check(lib().aw_align_pairs(self._h, C.byref(params), orientation, arr, len(pairs), flags, cb, None), "aw_align_pairs")
        return out

    def align_stream(self, params, chunks, orientation=AW_ORIENT_MASH, flags=0, callback=None, block_callback=None):
        """aw_align_stream: `chunks` is an iterable of pair lists (the library pulls one at a time and keeps two in flight);
        callback(result_dict) and / or block_callback(bytes, n_lines) (needs AW_FLAG_PAF_BLOCKS); non-zero / True cancels"""
        it = iter(chunks)
        keep = {}
        want_bytes = bool(flags & AW_FLAG_CIGAR_BYTES)

        def _next(_u, out):
            try:
                ch = next(it)
            except StopIteration:
                return 0
            if not ch:
                return 0
            keep["arr"] = make_pairs(ch)  # must stay alive until the following call
            out[0] = C.cast(keep["arr"], C.POINTER(AwPair))
            return len(ch)

        def _cb(rp, _u):
            return int(bool(callback(result_to_dict(rp.contents, want_bytes))))

        def _blk(text, n, lines, _u):
            return int(bool(block_callback(C.string_at(text, n), lines)))

        src = CHUNK_SOURCE(_next)
        cb = RESULT_CB(_cb) if callback is not None else C.cast(None, RESULT_CB)
        blk = PAF_BLOCK_CB(_blk) if block_callback is not None else C.cast(None, PAF_BLOCK_CB)
        check(lib().aw_align_stream(self._h, C.byref(params), orientation, flags, src, None, cb, blk, None), "aw_align_stream")

    def estimate_divergence(self, pairs):
        arr = make_pairs(pairs)
        out = (C.c_float * max(1, len(pairs)))()
        check(lib().aw_estimate_divergence(self._h, arr, len(pairs), out), "aw_estimate_divergence")
        return [float(out[i]) for i in range(len(pairs))]

    def orient_pairs(self, pairs):
        arr = make_pairs(pairs)
        out = (C.c_uint8 * max(1, len(pairs)))()
        check(lib().aw_orient_pairs(self._h, arr, len(pairs), out), "aw_orient_pairs")
        return [int(out[i]) for i in range(len(pairs))]

    def get_sketch(self, idx, reverse_complement=False, canonical=False, k=15, size=1000):
        out = (C.c_uint64 * size)()
        n = C.c_uint32()
        check(lib().aw_get_sketch(self._h, idx, int(reverse_complement), int(canonical), k, size, out, C.byref(n)), "aw_get_sketch")
        return list(out[: n.value])

    def mash_jaccard_counts(self, k=15, size=1000):
        import numpy as np

        n = self.n
        inter = np.zeros((n, n), dtype=np.uint32)
        uni = np.zeros((n, n), dtype=np.uint32)
        check(lib().aw_mash_jaccard_counts(self._h, k, size, inter.ctypes.data_as(C.POINTER(C.c_uint32)),
                                           uni.ctypes.data_as(C.POINTER(C.c_uint32))), "aw_mash_jaccard_counts")
        return inter, uni


class Batch:
    """device-resident batch (aw_batch_*): what bench.py times"""

    def __init__(self, ctx, params, pairs, orientation=AW_ORIENT_MASH, flags=0):
        self.ctx = ctx
        self.flags = flags
        self._arr = make_pairs(pairs)
        h = C.c_void_p()
        check(lib().aw_batch_create(ctx._h, C.byref(params), orientation, self._arr, len(pairs), flags, C.byref(h)), "aw_batch_create")
        self._h = h

    def launch(self, stream=None):
        check(lib().aw_batch_launch(self.ctx._h, self._h, C.c_void_p(stream) if stream else None), "aw_batch_launch")

    def fetch(self, collect=True, callback=None):
        out = []
        want_bytes = bool(self.flags & AW_FLAG_CIGAR_BYTES)

        def _cb(rp, _u):
            if callback is not None:
                return int(bool(callback(rp.contents)))
            if collect:
                out.append(result_to_dict(rp.contents, want_bytes))
            return 0

        cb = RESULT_CB(_cb) if (collect or callback is not None) else C.cast(None, RESULT_CB)
        check(lib().aw_batch_fetch(self.ctx._h, self._h, cb, None), "aw_batch_fetch")
        return out

    def stats(self):
        s = (C.c_uint64 * 8)()
        check(lib().aw_batch_stats(self.ctx._h, self._h, s), "aw_batch_stats")
        keys = ["kernels_launched", "pairs_retried", "paf_bytes", "cigar_runs", "sum_block_len", "failed_pairs", "cells", "steps"]
        return dict(zip(keys, [int(x) for x in s]))

    def debug_cycles(self):
        s = (C.c_uint64 * 6)()
        check(lib().aw_batch_debug_cycles(self.ctx._h, self._h, s), "aw_batch_debug_cycles")
        return dict(zip(["phase1", "phase2", "base", "backtrace", "emit", "other"], [int(x) for x in s]))

    def kernel_ms(self):
        ms = C.c_float()
        check(lib().aw_batch_kernel_ms(self.ctx._h, self._h, C.byref(ms)), "aw_batch_kernel_ms")
        return float(ms.value)

    def close(self):
        if self._h:
            lib().aw_batch_destroy(self.ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Aligner:
    """lib_wfa2::AffineWavefronts-shaped single-pair aligner (aw_aligner_*)"""

    def __init__(self, ctx, mismatch, gap_open1, gap_ext1, gap_open2=None, gap_ext2=None, match=0, memory_mode=AW_MEMORY_ULTRALOW):
        h = C.c_void_p()
        if gap_open2 is None:
            check(lib().aw_aligner_new_affine(ctx._h, match, mismatch, gap_open1, gap_ext1, memory_mode, C.byref(h)), "aw_aligner_new_affine")
        else:
            check(lib().aw_aligner_new_affine2p(ctx._h, match, mismatch, gap_open1, gap_ext1, gap_open2, gap_ext2, memory_mode, C.byref(h)),
                  "aw_aligner_new_affine2p")
        self._h = h

    def set_alignment_scope(self, scope):
        """AW_SCOPE_SCORE: align() computes the score only and cigar() is empty; AW_SCOPE_ALIGNMENT (default): both"""
        check(lib().aw_aligner_set_alignment_scope(self._h, scope), "aw_aligner_set_alignment_scope")

    def align(self, pattern: bytes, text: bytes):
        return lib().aw_aligner_align(self._h, pattern, len(pattern), text, len(text))

    def score(self):
        return lib().aw_aligner_score(self._h)

    def cigar(self):
        n = C.c_uint64()
        p = lib().aw_aligner_cigar(self._h, C.byref(n))
        return C.string_at(p, n.value) if n.value else b""

    def close(self):
        if self._h:
            lib().aw_aligner_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
