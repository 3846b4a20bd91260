"""Score-only alignment (AW_FLAG_SCORE_ONLY, AW_SCOPE_SCORE): the optimal score of every pair without recursion, CIGAR or
PAF.  The optimal score is unique, so every score-only result is checked against the full alignment path of the GPU and
the CPU oracle's scores (and, on samples, the independent Gotoh DP)."""
import gzip
import json
import os
import random

import pytest

import allwave_b200 as aw
from allwave_b200 import synth
from test_gpu_round2 import CORES, DEFAULT, PENALTY_SETS, _cluster_ctx, _mutate, _sweep_group

gpu = pytest.mark.gpu
EDIT = dict(mismatch=1, gap_open=1, gap_extend=1, gap2_open=None, gap2_extend=None)


def _all_pairs(n):
    return [(i, j) for i in range(n) for j in range(n) if i != j]


def _rand_pairs(n, k, seed):
    rnd = random.Random(seed)
    pairs = []
    while len(pairs) < k:
        a, b = rnd.randrange(n), rnd.randrange(n)
        if a != b:
            pairs.append((a, b))
    return pairs


def _check_shape(res, seqs, pairs):
    """what a score-only result carries: indices, status, score, strand, the End2End span; no counts, CIGAR or text"""
    assert len(res) == len(pairs)
    for r, (q, t) in zip(res, pairs):
        assert (r["query_idx"], r["target_idx"]) == (q, t)
        assert r["status"] == 0, (q, t, r["status"])
        assert (r["query_start"], r["query_end"], r["target_start"], r["target_end"]) == (0, len(seqs[q]), 0, len(seqs[t]))
        assert (r["num_matches"], r["alignment_length"], r["cg"], r["paf"], r["cigar_bytes"]) == (0, 0, "", "", b"")


def _same(score_res, full_res):
    """status, score, strand and end coordinates of the score-only run equal those of the full alignment"""
    key = lambda r: (r["query_idx"], r["target_idx"], r["status"], r["score"], r["is_reverse"], r["query_start"], r["query_end"],
                     r["target_start"], r["target_end"])
    bad = [(key(a), key(b)) for a, b in zip(score_res, full_res) if key(a) != key(b)]
    assert not bad, f"{len(bad)}/{len(full_res)} pairs differ, first: {bad[:3]}"


def _oracle_scores(oracle, ids, seqs, pairs, pen, orientation):
    p = oracle.params(**pen)
    if orientation == aw.AW_ORIENT_FORWARD:
        return [oracle.wfa_align(p, seqs[q], seqs[t])[1] for q, t in pairs]
    return oracle.run_pairs(ids, seqs, pairs, p, use_mash=(orientation == aw.AW_ORIENT_MASH), threads=CORES)["scores"]


def _run(oracle, ctx, ids, seqs, pairs, pen, orientation=aw.AW_ORIENT_MASH, exp_scores=None, full=None):
    """score-only, full path (unless given) and oracle on the same pairs; returns the score-only results"""
    ctx.load_sequences(ids, seqs)
    params = aw.make_params(**pen)
    res = ctx.align_pairs(params, pairs, orientation=orientation, flags=aw.AW_FLAG_SCORE_ONLY)
    if full is None:
        full = ctx.align_pairs(params, pairs, orientation=orientation)
    _check_shape(res, seqs, pairs)
    _same(res, full)
    if exp_scores is None:
        exp_scores = _oracle_scores(oracle, ids, seqs, pairs, pen, orientation)
    bad = [(q, t, r["score"], s) for r, (q, t), s in zip(res, pairs, exp_scores) if r["score"] != s]
    assert not bad, f"{len(bad)}/{len(pairs)} scores differ from the oracle, first: {bad[:3]}"
    return res


def _gotoh_sample(oracle, res, seqs, pen, k, seed):
    p = oracle.params(**pen)
    for r in random.Random(seed).sample(res, min(k, len(res))):
        q, t = seqs[r["query_idx"]], seqs[r["target_idx"]]
        if r["is_reverse"]:
            q = oracle.reverse_complement(q)
        assert -r["score"] == oracle.gotoh_penalty(p, q, t)


# ---- 6. CPU: the flag and the scope constants are exported -----------------------------------------------------------
def test_flag_and_scope_exported():
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "allwave_cuda.h")).read()
    assert "#define AW_FLAG_SCORE_ONLY 16u" in hdr
    assert aw.AW_FLAG_SCORE_ONLY == aw._cabi.AW_FLAG_SCORE_ONLY == 16
    assert (aw.AW_SCOPE_SCORE, aw.AW_SCOPE_ALIGNMENT) == (0, 1)
    assert hasattr(aw.Aligner, "set_alignment_scope")


# ---- 1. sweep ----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("group", range(10))
def test_sweep_three_kernels(oracle, group):
    """2,000 seeded pairs per penalty set through the one-warp kernel (threads_per_cta 0: pairs up to 1 kb) and the chunked
    int16 kernels with 128 and 256 threads: scores equal the oracle's, everything else equals the full path with the default
    kernel choice (test_chunked_kernels.py holds the full path on the forced CTA sizes to the oracle)"""
    pen = PENALTY_SETS[group]
    ids, seqs, pairs = _sweep_group(9100 + group, npairs=2000)
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**pen), use_mash=True, threads=CORES)["scores"]
    full = None
    for tpc in (0, 128, 256):
        ctx = aw.Context(0)
        try:
            ctx.set_option("threads_per_cta", tpc)
            if full is None:
                ctx.load_sequences(ids, seqs)
                full = ctx.align_pairs(aw.make_params(**pen), pairs)
            res = _run(oracle, ctx, ids, seqs, pairs, pen, exp_scores=exp, full=full)
        finally:
            ctx.close()
    _gotoh_sample(oracle, res, seqs, pen, 100, group)


# ---- 2. edges ----------------------------------------------------------------------------------------------------------
@gpu
def test_edges(oracle, gpu_ctx):
    """empty sequences, identical sequences, lengths around the base-case length 100"""
    rnd = random.Random(15)
    base = bytes(rnd.choice(b"ACGT") for _ in range(300))
    seqs = [b"", b"A", b"ACGT", base, base, base[:150], base[150:], b"A" * 200, b"ACGT" * 40]
    for n in (99, 100, 101):
        a = bytes(rnd.choice(b"ACGT") for _ in range(n))
        seqs += [a, _mutate(rnd, a, 0.05)[:n].ljust(n, b"A"), _mutate(rnd, a, 0.2)]
    ids = ["e%d" % i for i in range(len(seqs))]
    for pen in (DEFAULT, EDIT):
        for orientation in (aw.AW_ORIENT_FORWARD, aw.AW_ORIENT_MASH):
            res = _run(oracle, gpu_ctx, ids, seqs, _all_pairs(len(seqs)), pen, orientation=orientation)
    assert (res[0]["query_end"], res[0]["target_end"]) == (0, 1)  # "" vs "A": one pure gap
    gpu_ctx.load_sequences(["a", "b"], [base, base])
    r = gpu_ctx.align_pairs(aw.make_params(**DEFAULT), [(0, 1)], flags=aw.AW_FLAG_SCORE_ONLY)[0]
    assert (r["status"], r["score"], r["is_reverse"], r["query_end"], r["target_end"]) == (0, 0, False, 300, 300)


@gpu
def test_scores_around_base_case_score(oracle, gpu_ctx):
    """scores on both sides of 250, where the top level switches between the base case and a breakpoint search"""
    rnd = random.Random(250)
    seqs = []
    for d in (0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.08):
        a = bytes(rnd.choice(b"ACGT") for _ in range(900))
        seqs += [a, _mutate(rnd, a, d)]
    ids = ["s%d" % i for i in range(len(seqs))]
    pairs = [(2 * i, 2 * i + 1) for i in range(len(seqs) // 2)] + [(2 * i + 1, 2 * i) for i in range(len(seqs) // 2)]
    res = _run(oracle, gpu_ctx, ids, seqs, pairs, DEFAULT, orientation=aw.AW_ORIENT_FORWARD)
    pens = [-r["score"] for r in res]
    assert min(pens) <= 250 < max(pens), pens


@gpu
def test_byte_kernel(oracle, gpu_ctx):
    """N and lower-case bytes take the byte (8-bit) kernels"""
    ids, seqs, _ = synth.generate(77, 5, 500, 0.04)
    seqs[1] = seqs[1][:100] + b"NNNNnnacgt" + seqs[1][110:]
    seqs[2] = seqs[2].lower()
    for orientation in (aw.AW_ORIENT_FORWARD, aw.AW_ORIENT_MASH):
        _run(oracle, gpu_ctx, ids, seqs, _all_pairs(5), DEFAULT, orientation=orientation)


@gpu
def test_match_score_bonus(oracle, gpu_ctx):
    """match_score < 0: the wavefront penalty P' on the shifted penalties converts to the user's penalty (P' + M (plen+tlen)) / 2"""
    ids, seqs, pairs = _sweep_group(978, nfam=24, members=4, maxlen=320, npairs=2500)
    for pen in (dict(match=-1, mismatch=4, gap_open=6, gap_extend=2, gap2_open=None, gap2_extend=None),
                dict(match=-2, mismatch=5, gap_open=8, gap_extend=2, gap2_open=24, gap2_extend=1),
                dict(match=-3, mismatch=2, gap_open=1, gap_extend=1, gap2_open=None, gap2_extend=None)):
        res = _run(oracle, gpu_ctx, ids, seqs, pairs, pen)
        assert any(r["score"] > 0 for r in res)
    ids2, seqs2, _ = synth.generate(12, 6, 9000, 0.04)
    _run(oracle, gpu_ctx, ids2, seqs2, _all_pairs(6), dict(match=-1, mismatch=5, gap_open=8, gap_extend=2, gap2_open=24, gap2_extend=1))


@gpu
def test_large_penalties_shared_memory_optin(oracle, gpu_ctx):
    """max_score_scope of 80..150 needs more than 48 KB of shared memory: the score kernels opt in like the full ones"""
    ids, seqs, _ = synth.generate(31, 6, 2000, 0.03)
    for pen in (dict(mismatch=5, gap_open=8, gap_extend=2, gap2_open=80, gap2_extend=1), dict(mismatch=3, gap_open=6, gap_extend=2, gap2_open=140, gap2_extend=1),
                dict(mismatch=90, gap_open=20, gap_extend=5, gap2_open=None, gap2_extend=None)):
        _run(oracle, gpu_ctx, ids, seqs, _all_pairs(6), pen)


# ---- 3. full size ------------------------------------------------------------------------------------------------------
@gpu
def test_c2_full_size(oracle, gpu_ctx):
    c, ids, seqs, _ = synth.config("C2", n=1000)
    _run(oracle, gpu_ctx, ids, seqs, _rand_pairs(1000, 256, 23), DEFAULT)


@gpu
def test_c5_full_size_mash_orientation(oracle, gpu_ctx):
    c, ids, seqs, rc = synth.config("C5", n=5000)
    res = _run(oracle, gpu_ctx, ids, seqs, _rand_pairs(5000, 256, 56), DEFAULT)
    assert any(r["is_reverse"] for r in res) and not all(r["is_reverse"] for r in res)
    for r in res:
        assert r["is_reverse"] == (rc[r["query_idx"]] != rc[r["target_idx"]])


@gpu
def test_c1_full_config(oracle, gpu_ctx):
    c, ids, seqs, _ = synth.config("C1")
    _run(oracle, gpu_ctx, ids, seqs, _all_pairs(16), DEFAULT)


@gpu
def test_int32_rows(oracle, gpu_ctx):
    """pairs just over the int16 storage bound (2*tlen+plen >= 32000) take the int32 chunked kernels"""
    ids, seqs, _ = synth.generate(4243, 2, 10800, 0.02)
    a, b = seqs
    for x, y in ((a[:10700], b[:10700]), (a[:10660], b[:10500])):
        p, t = len(x), len(y)
        assert 2 * t + p >= 32000 or 2 * p + t >= 32000 or 3 * (p + t) >= 63000  # outside plan_launch's int16 rule
        _run(oracle, gpu_ctx, ["x", "y"], [x, y], [(0, 1), (1, 0)], DEFAULT, orientation=aw.AW_ORIENT_FORWARD)


@gpu
@pytest.mark.parametrize("solo_len", [0, 3000])
def test_cluster_kernel(oracle, solo_len):
    """the cluster kernel (one pair per 8-CTA cluster): its top level is the cluster-wide part of the pair"""
    c, ids, seqs, _ = synth.config("C4", n=4, length=30000)
    pairs = [(0, 1), (1, 2), (2, 3), (3, 0), (0, 2)]
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**DEFAULT), use_mash=True, threads=CORES, fast=True)["scores"]
    ctx = _cluster_ctx(1000, solo_len)
    try:
        _run(oracle, ctx, ids, seqs, pairs, DEFAULT, exp_scores=exp)
        # pairs whose top level is a base case or one long gap
        rnd = random.Random(78)
        a = bytes(rnd.choice(b"ACGT") for _ in range(40000))
        s2 = [a, a, a[:25000], a[5000:], _mutate(rnd, a, 0.01)]
        p2 = [(0, 1), (0, 2), (2, 0), (3, 0), (0, 4)]
        _run(oracle, ctx, ["k%d" % i for i in range(5)], s2, p2, DEFAULT)
    finally:
        ctx.close()


@gpu
def test_c4_golden_pairs():
    """the 4 frozen C4 pairs (1 Mb haplotypes with SVs): score equals the golden score"""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c4_pairs.json.gz")
    gold = json.load(gzip.open(path, "rt"))
    c, ids, seqs, _ = synth.config("C4")
    pairs = [(g["q"], g["t"]) for g in gold["pairs"]]
    ctx = aw.Context(0)
    try:
        ctx.load_sequences(ids, seqs)
        res = ctx.align_pairs(aw.make_params(**DEFAULT), pairs, flags=aw.AW_FLAG_SCORE_ONLY)
        _check_shape(res, seqs, pairs)
        assert [r["score"] for r in res] == [g["score"] for g in gold["pairs"]]
    finally:
        ctx.close()


# ---- 4. modes and plumbing ---------------------------------------------------------------------------------------------
@gpu
def test_wfa_orientation(oracle, gpu_ctx):
    """AW_ORIENT_WFA: the two count-only orientation passes still run in full; the strand equals the full path's"""
    c, ids, seqs, rc = synth.config("C5", n=6, length=1200)
    res = _run(oracle, gpu_ctx, ids, seqs, _all_pairs(6), DEFAULT, orientation=aw.AW_ORIENT_WFA)
    for r in res:
        assert r["is_reverse"] == (rc[r["query_idx"]] != rc[r["target_idx"]])


@gpu
def test_retry_ladder(oracle):
    """a 48-diagonal first-try workspace: pairs report AW_EWORKSPACE on the device and go through the retry ladder"""
    ids, seqs, _ = synth.generate(77, 4, 3000, 0.08)
    pairs = _all_pairs(4)
    ctx = aw.Context(0)
    try:
        ctx.set_option("max_wavefront_width", 48)
        _run(oracle, ctx, ids, seqs, pairs, DEFAULT, orientation=aw.AW_ORIENT_FORWARD)
        b = aw.Batch(ctx, aw.make_params(**DEFAULT), pairs, orientation=aw.AW_ORIENT_FORWARD, flags=aw.AW_FLAG_SCORE_ONLY)
        b.launch()
        b.fetch(collect=False)
        st = b.stats()
        assert st["pairs_retried"] > 0 and st["failed_pairs"] == 0
        b.close()
    finally:
        ctx.close()


@gpu
def test_failure_without_sentinel(gpu_ctx):
    """with the ladder off a pair that does not fit fails as AW_EALIGN with score INT32_MAX and no sentinel line"""
    ids, seqs, _ = synth.generate(808, 4, 900, 0.08)
    seqs[3] = seqs[0]
    pairs = [(0, 1), (0, 3), (2, 1)]
    ctx = aw.Context(0)
    try:
        ctx.set_option("max_wavefront_width", 48)
        ctx.set_option("max_retry_attempts", 0)
        ctx.load_sequences(ids, seqs)
        res = ctx.align_pairs(aw.make_params(**DEFAULT), pairs, orientation=aw.AW_ORIENT_FORWARD, flags=aw.AW_FLAG_SCORE_ONLY)
        for r, (q, t) in zip(res, pairs):
            if (q, t) == (0, 3):
                assert (r["status"], r["score"], r["query_end"], r["target_end"]) == (0, 0, len(seqs[0]), len(seqs[0]))
                continue
            assert r["status"] == aw.AW_EALIGN and r["score"] == 2 ** 31 - 1
            assert (r["paf"], r["cg"], r["cigar_bytes"], r["num_matches"], r["alignment_length"]) == ("", "", b"", 0, 0)
    finally:
        ctx.close()


@gpu
def test_stream_several_chunks(oracle, gpu_ctx):
    """aw_align_stream pulls several chunks and keeps two batches in flight: results equal one aw_align_pairs call"""
    c, ids, seqs, _ = synth.config("C5", n=40, length=2000)
    pairs = _all_pairs(40)
    gpu_ctx.load_sequences(ids, seqs)
    params = aw.make_params(**DEFAULT)
    got = []
    gpu_ctx.align_stream(params, [pairs[i:i + 300] for i in range(0, len(pairs), 300)], flags=aw.AW_FLAG_SCORE_ONLY, callback=got.append)
    full = gpu_ctx.align_pairs(params, pairs)
    _check_shape(got, seqs, pairs)
    _same(got, full)
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**DEFAULT), use_mash=True, threads=CORES)["scores"]
    assert [r["score"] for r in got] == exp


@gpu
def test_cpp_host_for_each_with_callback(gpu_ctx):
    """AllPairIterator::for_each_with_callback(cb, AW_FLAG_SCORE_ONLY) of the C++ host: the flag reaches the stream, the
    callback copes with the missing CIGAR and PAF"""
    from allwave_b200 import hostlib as H

    c, ids, seqs, _ = synth.config("C5", n=12, length=3000)
    gpu_ctx.load_sequences(ids, seqs)
    lens = [len(s) for s in seqs]
    rows = H.for_each_rows(gpu_ctx, ids, lens, aw.AW_FLAG_SCORE_ONLY)
    full = H.for_each_rows(gpu_ctx, ids, lens, 0)
    assert len(rows) == len(full) == 12 * 11
    key = lambda r: (r["query_idx"], r["target_idx"])
    by = {key(r): r for r in full}
    for r in rows:
        f = by[key(r)]
        assert (r["score"], r["is_reverse"], r["query_end"], r["target_end"]) == (f["score"], f["is_reverse"], f["query_end"], f["target_end"])
        assert (r["query_end"], r["target_end"]) == (lens[r["query_idx"]], lens[r["target_idx"]])
        assert r["cg_len"] == r["paf_len"] == 0 and f["cg_len"] > 0 and f["paf_len"] > 0


@gpu
def test_forbidden_flag_combinations(gpu_ctx):
    ids, seqs, _ = synth.generate(3, 3, 500, 0.02)
    gpu_ctx.load_sequences(ids, seqs)
    params = aw.make_params(**DEFAULT)
    for extra in (aw.AW_FLAG_CIGAR_BYTES, aw.AW_FLAG_PAF_BLOCKS):
        flags = aw.AW_FLAG_SCORE_ONLY | extra
        with pytest.raises(aw.AllwaveError) as ei:
            gpu_ctx.align_pairs(params, [(0, 1)], flags=flags)
        assert ei.value.status == aw.AW_EINVAL and "AW_FLAG_SCORE_ONLY" in str(ei.value)
        with pytest.raises(aw.AllwaveError) as ei:
            gpu_ctx.align_stream(params, [[(0, 1)]], flags=flags, callback=lambda r: 0)
        assert ei.value.status == aw.AW_EINVAL
        with pytest.raises(aw.AllwaveError) as ei:
            aw.Batch(gpu_ctx, params, [(0, 1)], flags=flags)
        assert ei.value.status == aw.AW_EINVAL


@gpu
def test_aligner_score_scope(oracle, gpu_ctx):
    """Aligner with AW_SCOPE_SCORE: the alignment scope's score, an empty CIGAR; switching back restores the CIGAR"""
    ids, seqs, _ = synth.generate(32, 2, 3000, 0.05)
    for args, pen in (((5, 8, 2, 24, 1), DEFAULT), ((4, 6, 2), dict(mismatch=4, gap_open=6, gap_extend=2, gap2_open=None, gap2_extend=None))):
        al = aw.Aligner(gpu_ctx, *args)
        try:
            assert al.align(seqs[0], seqs[1]) == 0
            score, cigar = al.score(), al.cigar()
            st, sc, ops, _ = oracle.wfa_align(oracle.params(**pen), seqs[0], seqs[1])
            assert (score, cigar) == (sc, ops)
            al.set_alignment_scope(aw.AW_SCOPE_SCORE)
            assert al.align(seqs[0], seqs[1]) == 0
            assert al.score() == score and al.cigar() == b""
            assert al.align(b"", b"ACG") == 0
            gap = al.score()
            al.set_alignment_scope(aw.AW_SCOPE_ALIGNMENT)
            assert al.align(b"", b"ACG") == 0 and al.score() == gap and al.cigar() == b"III"
            assert al.align(seqs[0], seqs[1]) == 0
            assert (al.score(), al.cigar()) == (score, cigar)
        finally:
            al.close()


# ---- 5. work actually skipped ------------------------------------------------------------------------------------------
@gpu
def test_work_skipped(gpu_ctx):
    """on 1,024 C2 pairs the score-only launch computes at most 0.6x the cells and 0.3x the wavefront steps of the full
    launch (the CPU oracle counts 0.50 and 0.16 on these pairs): the recursion below the top level does not run"""
    c, ids, seqs, _ = synth.config("C2", n=1000)
    pairs = _rand_pairs(1000, 1024, 5)
    gpu_ctx.load_sequences(ids, seqs)
    params = aw.make_params(**DEFAULT)
    st, scores = {}, {}
    for name, flags in (("full", 0), ("score", aw.AW_FLAG_SCORE_ONLY)):
        b = aw.Batch(gpu_ctx, params, pairs, flags=flags)
        b.launch()
        scores[name] = [(r["status"], r["score"], r["is_reverse"]) for r in b.fetch()]
        st[name] = b.stats()
        b.close()
    assert scores["score"] == scores["full"]
    assert st["score"]["cells"] <= 0.6 * st["full"]["cells"], st
    assert st["score"]["steps"] <= 0.3 * st["full"]["steps"], st
    assert st["score"]["paf_bytes"] == st["score"]["cigar_runs"] == st["score"]["sum_block_len"] == 0
    assert st["score"]["failed_pairs"] == 0
