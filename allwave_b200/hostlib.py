"""ctypes binding of liballwave_host.so: C exports (host_capi.cpp) of the C++ host mirror
(allwave_b200/host/allwave.hpp) of the reference's library surface."""
import ctypes as C
import os

from . import _cabi

_PKG = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_PKG, "liballwave_host.so")
_lib = None

KIND_NONE, KIND_RANDOM, KIND_AUTO, KIND_CONNECTIVITY, KIND_TREE = range(5)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise ImportError(f"{_SO} is missing: run __graft_entry__.build()")
        _cabi.lib()  # make sure liballwave_cuda.so is resolvable first
        L = C.CDLL(_SO)
        L.awh_last_message.restype = C.c_char_p
        L.awh_parse_scores.argtypes = [C.c_char_p, C.POINTER(_cabi.AwParams)]
        L.awh_parse_sparsification.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                               C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.awh_connectivity_probability.argtypes = [C.c_uint64, C.c_double]
        L.awh_connectivity_probability.restype = C.c_double
        L.awh_hash_str.argtypes = [C.c_char_p]
        L.awh_hash_str.restype = C.c_uint64
        L.awh_mode_from_params.argtypes = [C.POINTER(_cabi.AwParams)]
        L.awh_pair_list.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.c_int, C.c_double, C.c_uint64, C.c_uint64, C.c_double, C.c_int, C.c_int,
                                    C.POINTER(C.POINTER(C.c_uint64)), C.POINTER(C.c_uint64)]
        L.awh_build_knn_graph.argtypes = [C.POINTER(C.c_double), C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]
        L.awh_build_knn_graph.restype = C.POINTER(C.c_uint64)
        L.awh_free.argtypes = [C.c_void_p]
        L.awh_parse_ani_preset.argtypes = [C.c_char_p, C.c_char_p]
        L.awh_read_fasta.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.awh_read_fasta.restype = C.c_int64
        L.awh_run_job.argtypes = [C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_char_p, C.c_char_p, C.c_int, C.c_int,
                                  C.c_int, C.c_uint64, C.c_char_p, C.c_int, C.POINTER(C.c_double)]
        L.awh_test_cancel.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_uint64, C.c_uint64, C.c_char_p]
        L.awh_test_cancel.restype = C.c_int64
        L.awh_test_for_each.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_uint32, C.POINTER(C.c_int64), C.c_uint64]
        L.awh_test_for_each.restype = C.c_int64
        L.awh_validate_cigar.argtypes = [C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_char_p]
        L.awh_align_sequences.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_int32), C.c_int, C.POINTER(C.c_int32),
                                          C.POINTER(C.c_uint64), C.POINTER(C.c_void_p)]
        L.awh_partition_pairs.argtypes = [C.POINTER(C.c_uint64), C.c_uint64, C.POINTER(C.c_uint64), C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32)]
        _lib = L
    return _lib


def parse_scores(s):
    p = _cabi.AwParams()
    if lib().awh_parse_scores(s.encode(), C.byref(p)) != 0:
        raise ValueError(lib().awh_last_message().decode())
    return p


def parse_sparsification(s):
    kind, value, kn, kf, rf, kmer = C.c_int(), C.c_double(), C.c_uint64(), C.c_uint64(), C.c_double(), C.c_int()
    if lib().awh_parse_sparsification(s.encode(), C.byref(kind), C.byref(value), C.byref(kn), C.byref(kf), C.byref(rf), C.byref(kmer)) != 0:
        raise ValueError(lib().awh_last_message().decode())
    return dict(kind=kind.value, value=value.value, k_nearest=kn.value, k_farthest=kf.value, random_fraction=rf.value, kmer_size=kmer.value)


def pair_list(ids, kind=KIND_NONE, value=0.0, k_nearest=0, k_farthest=0, random_fraction=0.0, kmer_size=0, exclude_self=True, ctx=None):
    """AllPairIterator::with_options(...).get_pairs(); ctx (sequences loaded) is required for KIND_TREE"""
    n = len(ids)
    ia = (C.c_char_p * max(1, n))(*[i.encode() for i in ids])
    out = C.POINTER(C.c_uint64)()
    cnt = C.c_uint64()
    rc = lib().awh_pair_list(ctx._h if ctx is not None else None, n, ia, kind, value, k_nearest, k_farthest, random_fraction, kmer_size,
                             1 if exclude_self else 0, C.byref(out), C.byref(cnt))
    if rc != 0:
        raise RuntimeError(lib().awh_last_message().decode())
    pairs = [(out[2 * i], out[2 * i + 1]) for i in range(cnt.value)]
    lib().awh_free(out)
    return pairs


def build_knn_graph(matrix, k, farthest):
    n = len(matrix)
    flat = (C.c_double * max(1, n * n))(*[v for row in matrix for v in row])
    cnt = C.c_uint64()
    p = lib().awh_build_knn_graph(flat, n, k, 1 if farthest else 0, C.byref(cnt))
    out = [(p[2 * i], p[2 * i + 1]) for i in range(cnt.value)]
    lib().awh_free(p)
    return out


def partition_pairs(pairs, lens, n_parts):
    """allwave.hpp partition_pairs (the C++ multi-GPU sharding): list of n_parts pair lists, like partition.partition_pairs"""
    n = len(pairs)
    pa = (C.c_uint64 * max(1, 2 * n))(*[v for p in pairs for v in p])
    la = (C.c_uint64 * max(1, len(lens)))(*lens)
    out = (C.c_uint32 * max(1, n))()
    if lib().awh_partition_pairs(pa, n, la, len(lens), n_parts, out) != 0:
        raise RuntimeError(lib().awh_last_message().decode())
    shards = [[] for _ in range(max(1, n_parts))]
    for i, p in enumerate(pairs):
        shards[out[i]].append(tuple(p))
    return shards


def parse_ani_preset(s):
    """parse_ani_preset of the reference CLI (src/main.rs:83-124)"""
    buf = C.create_string_buffer(32)
    if lib().awh_parse_ani_preset(s.encode(), buf) != 0:
        raise ValueError(lib().awh_last_message().decode())
    return buf.value.decode()


def read_fasta(path, keep_prefixes="", exclude_prefixes=""):
    """read_fasta (+ -k / -e prefix filters) of the C++ host: (ids, total sequence length); .gz input needs zlib"""
    ids = C.c_void_p()
    tot = C.c_uint64()
    n = lib().awh_read_fasta(str(path).encode(), keep_prefixes.encode(), exclude_prefixes.encode(), C.byref(ids), C.byref(tot))
    if n < 0:
        raise RuntimeError(lib().awh_last_message().decode())
    joined = C.string_at(ids.value).decode()
    lib().awh_free(ids)
    return [x for x in joined.split("\n") if x != ""][:n] if n else [], tot.value


def run_job(ids, seqs, scores="0,5,8,2,24,1", sparsification="none", use_mash=True, first_device=0, n_gpus=1, max_pairs=0, out_path="", checksum=False):
    """the product path of `allwave --gpus N` on in-memory sequences (host_capi.cpp awh_run_job): contexts on n_gpus devices,
    pair list, streaming multi-GPU driver, PAF blocks.  Returns a dict with pairs, paf_bytes, seconds, setup_seconds,
    imbalance (max/mean GPU busy time) and, with checksum=True, an order-independent digest of the PAF lines."""
    n = len(seqs)
    ia = (C.c_char_p * max(1, n))(*[i.encode() for i in ids])
    sa = (C.c_char_p * max(1, n))(*seqs)
    la = (C.c_uint64 * max(1, n))(*[len(s) for s in seqs])
    out = (C.c_double * 6)()
    rc = lib().awh_run_job(n, ia, sa, la, scores.encode(), sparsification.encode(), 1 if use_mash else 0, first_device, n_gpus, max_pairs,
                           str(out_path).encode(), 1 if checksum else 0, out)
    if rc != 0:
        raise RuntimeError(lib().awh_last_message().decode())
    import struct

    digest = struct.unpack("<Q", struct.pack("<d", out[5]))[0]
    return dict(pairs=int(out[0]), paf_bytes=int(out[1]), seconds=out[2], setup_seconds=out[3], imbalance=out[4], digest=digest)


def cancel_probe(ctx, ids, lens, fail_at, chunk_pairs=0):
    """for_each_with_callback whose callback throws at result `fail_at`: (results seen, message) or (-1, "") if nothing was rethrown"""
    n = len(ids)
    ia = (C.c_char_p * max(1, n))(*[i.encode() for i in ids])
    la = (C.c_uint64 * max(1, n))(*lens)
    msg = C.create_string_buffer(128)
    seen = lib().awh_test_cancel(ctx._h, n, ia, la, fail_at, chunk_pairs, msg)
    return seen, msg.value.decode()


def for_each_rows(ctx, ids, lens, flags=0):
    """AllPairIterator::for_each_with_callback(cb, flags) over every ordered pair (default params, mash orientation): one dict per
    result with the numeric fields and the lengths of its CIGAR string and PAF line"""
    n = len(ids)
    ia = (C.c_char_p * max(1, n))(*[i.encode() for i in ids])
    la = (C.c_uint64 * max(1, n))(*lens)
    cap = n * n
    rows = (C.c_int64 * (8 * max(1, cap)))()
    k = lib().awh_test_for_each(ctx._h, n, ia, la, flags, rows, cap)
    if k < 0:
        raise RuntimeError(lib().awh_last_message().decode())
    keys = ["query_idx", "target_idx", "score", "is_reverse", "query_end", "target_end", "cg_len", "paf_len"]
    return [dict(zip(keys, rows[8 * i: 8 * i + 8])) for i in range(min(k, cap))]


def validate_cigar_alignment(cigar: bytes, query_len: int, reference_len: int):
    """wfa::validate_cigar_alignment (src/wfa.rs:105-176): None when valid, else the reference's message"""
    msg = C.create_string_buffer(160)
    rc = lib().awh_validate_cigar(cigar, len(cigar), query_len, reference_len, msg)
    return None if rc == 0 else msg.value.decode()


MODE_EDIT, MODE_AFFINE, MODE_AFFINE2P = 0, 1, 2


def align_sequences(ctx, pattern: bytes, text: bytes, mismatch, gap_opening1=0, gap_extension1=0, gap_opening2=0, gap_extension2=0, mode=MODE_AFFINE2P):
    """wfa::align_sequences (src/wfa.rs:178-258) through the C++ mirror -> dict(score, cigar, matches, mismatches, insertions, deletions,
    alignment_length); raises RuntimeError with the mirror's message on failure"""
    pen = (C.c_int32 * 5)(mismatch, gap_opening1, gap_extension1, gap_opening2, gap_extension2)
    score = C.c_int32()
    counts = (C.c_uint64 * 5)()
    cig = C.c_void_p()
    if lib().awh_align_sequences(ctx._h, pattern, len(pattern), text, len(text), pen, mode, C.byref(score), counts, C.byref(cig)) != 0:
        raise RuntimeError(lib().awh_last_message().decode())
    s = C.string_at(cig).decode()
    lib().awh_free(cig)
    return dict(score=score.value, cigar=s, matches=int(counts[0]), mismatches=int(counts[1]), insertions=int(counts[2]), deletions=int(counts[3]),
                alignment_length=int(counts[4]))
