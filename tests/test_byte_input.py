"""Byte-exact input: N runs, soft-masked lower case and IUPAC codes.

Comparison is on raw bytes and case-sensitive (N == N, a != A), and reverse_complement upper-cases and maps every other byte
to N.  One non-ACGT byte anywhere in a context sends every pair of that context to the byte (BITS=8) kernels: a separate
engine with its own per-diagonal loop, edge tracking, 4-byte match extension and int16 scalar rows.  These tests hold every
kernel `dispatch_align` can pick to the CPU oracle on such input (KERNEL_CASES), compare the byte kernels with the 2-bit
kernels on the same clean pairs at full size, and check the sketch kernel at the edges of its selection."""
import gzip
import math
import os
import random
import re
import subprocess

import numpy as np
import pytest

import allwave_b200 as aw
from allwave_b200 import synth
from test_gpu_round2 import CORES, DEFAULT, PENALTY_SETS, _mutate, _sweep_group
from test_score_only import _check_shape, _run

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
API = os.path.join(ROOT, "allwave_b200", "csrc", "aw_api.cu")
EDIT = PENALTY_SETS[4]
AFFINE = PENALTY_SETS[3]       # -x 65: single-piece affine
O1_GT_O2 = PENALTY_SETS[5]     # o1 > o2, e2 > e1
IUPAC = b"RYKMSW"


# ---- dirty input -------------------------------------------------------------------------------------------------------
def _add_dirt(rnd, fam, events=None, keep_len=False):
    """the same loci of every member of a family of haplotypes: assembly-gap N runs of different lengths, blocks soft-masked
    in every member (they match) or in some members only (a != A), single IUPAC bytes.  keep_len: every N run replaces as
    many bases as it has, so lengths stay put."""
    fam = [bytearray(s) for s in fam]
    n_ev = events if events is not None else 1 + max(len(s) for s in fam) // 1500
    for _ in range(n_ev):
        r, rel, w = rnd.random(), rnd.random(), rnd.randint(1, 60)
        for s in fam:
            if not s:
                continue
            p = int(rel * len(s))
            if r < 0.3:
                s[p:p + w] = b"N" * (len(s[p:p + w]) if keep_len else rnd.randint(1, 3 * w))
            elif r < 0.55:
                s[p:p + w] = s[p:p + w].lower()
            elif r < 0.75:
                if rnd.random() < 0.5:
                    s[p:p + w] = s[p:p + w].lower()
            elif p < len(s) and rnd.random() < 0.7:
                s[p] = rnd.choice(IUPAC)
    return [bytes(s) for s in fam]


def _dirty_families(rnd, seqs, members, clip=None):
    """_add_dirt on each family block of `seqs`; one member of every third family lower-cased whole, one of every seventh
    family all N"""
    out = []
    for f in range(0, len(seqs), members):
        fam = _add_dirt(rnd, seqs[f:f + members])
        if (f // members) % 3 == 1:
            fam[-1] = fam[-1].lower()
        if (f // members) % 7 == 2:
            fam[-2] = b"N" * len(fam[-2])
        out += fam
    return [s[:clip] for s in out] if clip else out


def _is_clean(s):
    return not s.translate(None, b"ACGT")


# ---- the kernels dispatch_align can launch, and the inputs that reach each --------------------------------------------
def _define(name):
    src = open(API).read() + open(os.path.join(ROOT, "allwave_b200", "csrc", "aw_wfa.cuh")).read()
    return int(re.search(r"#define %s (\d+)" % name, src).group(1))


CLUSTER_SIZE, CLUSTER_NT, REGS = _define("AW_CLUSTER_SIZE"), _define("AW_CLUSTER_NT"), _define("AW_REGS")
B200_SMS = 148


def plan_kernel(max_p, max_t, all_clean, two, opts=None, npairs=1, sm_count=B200_SMS):
    """plan_launch's kernel choice (aw_api.cu) -> (NT, BITS, TWO, WS, cluster size) for a batch whose longest query / target
    are max_p / max_t, in a context that is clean (every loaded sequence upper-case ACGT) or not"""
    o = dict(threads_per_cta=0, ws16=1, cluster_min_len=200000, cluster_always=0)
    o.update(opts or {})
    maxlen = max(max_p, max_t)
    fits16 = bool(o["ws16"]) and 2 * max_t + max_p < 32000 and 2 * max_p + max_t < 32000 and 3 * (max_p + max_t) < 63000
    tpc = o["threads_per_cta"]
    nt = tpc or (32 if maxlen <= 1024 else (128 if all_clean and (fits16 or maxlen <= 50000) else 256))
    slots = max(1, sm_count * (65536 // (CLUSTER_NT * REGS)) // CLUSTER_SIZE)
    cluster = (o["cluster_min_len"] > 0 and all_clean and not fits16 and maxlen >= o["cluster_min_len"] and not tpc
               and (npairs <= 2 * slots or o["cluster_always"]))
    if cluster:
        nt = CLUSTER_NT
    if nt == 128 and not all_clean:
        nt = 256
    ws16 = fits16 and nt >= 64
    return (nt, 2 if all_clean else 8, bool(two), "short" if ws16 else "int", CLUSTER_SIZE if cluster else 1)


def _two(pen):
    return pen.get("gap2_open") is not None and pen.get("gap2_extend") is not None


TPC256 = dict(threads_per_cta=256)
INT32 = dict(ws16=0)
CLUSTER = dict(cluster_min_len=1000, cluster_always=1)
# (NT, BITS, TWO, WS, cluster) -> haplotypes (n, length, divergence), clean or dirty context, penalties, set_option values
KERNEL_CASES = {
    (32, 2, True, "int", 1): dict(n=8, length=700, d=0.05, clean=True, pen=DEFAULT, opts={}),
    (32, 2, False, "int", 1): dict(n=8, length=700, d=0.05, clean=True, pen=EDIT, opts={}),
    (32, 8, True, "int", 1): dict(n=8, length=700, d=0.05, clean=False, pen=DEFAULT, opts={}),
    (32, 8, False, "int", 1): dict(n=8, length=700, d=0.05, clean=False, pen=AFFINE, opts={}),
    (128, 2, True, "short", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=DEFAULT, opts={}),
    (128, 2, False, "short", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=AFFINE, opts={}),
    (128, 2, True, "int", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=DEFAULT, opts=INT32),
    (128, 2, False, "int", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=EDIT, opts=INT32),
    (256, 2, True, "short", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=DEFAULT, opts=TPC256),
    (256, 2, False, "short", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=AFFINE, opts=TPC256),
    (256, 2, True, "int", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=DEFAULT, opts=dict(TPC256, **INT32)),
    (256, 2, False, "int", 1): dict(n=5, length=4000, d=0.04, clean=True, pen=AFFINE, opts=dict(TPC256, **INT32)),
    (256, 8, True, "short", 1): dict(n=5, length=4000, d=0.04, clean=False, pen=DEFAULT, opts={}),
    (256, 8, False, "short", 1): dict(n=5, length=4000, d=0.04, clean=False, pen=EDIT, opts={}),
    (256, 8, True, "int", 1): dict(n=4, length=12000, d=0.02, clean=False, pen=DEFAULT, opts={}),
    (256, 8, False, "int", 1): dict(n=5, length=4000, d=0.04, clean=False, pen=AFFINE, opts=INT32),
    (CLUSTER_NT, 2, True, "int", CLUSTER_SIZE): dict(n=4, length=12000, d=0.02, clean=True, pen=DEFAULT, opts=CLUSTER),
    (CLUSTER_NT, 2, False, "int", CLUSTER_SIZE): dict(n=4, length=12000, d=0.02, clean=True, pen=AFFINE, opts=CLUSTER),
}


def _case_id(key):
    nt, bits, two, ws, cl = key
    return f"nt{nt}-b{bits}-{'two' if two else 'one'}-{ws}" + (f"-cluster{cl}" if cl > 1 else "")


def _case_inputs(key):
    """the seeded input set of one kernel case: ids, sequences, all directed pairs, penalties, options"""
    e = KERNEL_CASES[key]
    ids, seqs, _ = synth.generate(700 + sorted(KERNEL_CASES).index(key), e["n"], e["length"], e["d"], rc_prob=0.5)
    if not e["clean"]:
        rnd = random.Random(e["length"])
        seqs = _add_dirt(rnd, seqs)
        seqs[1] = seqs[1].lower()
    pairs = [(i, j) for i in range(e["n"]) for j in range(e["n"]) if i != j]
    return ids, seqs, pairs, e["pen"], e["opts"]


def _parsed_kernels():
    """{(mode, (NT, BITS, TWO, WS, cluster))} launched by dispatch_align in the default build (no -DAW_FAST_BUILD, no
    AW_NT_EXPERIMENT)"""
    src = open(API).read()
    body = src[src.index("cudaError_t dispatch_align("):]
    body = body[:body.index("\n}\n")]
    out = set()
    macro = re.search(r"#define AW_CASE\(NT_, BITS_, TWO_, WS_, W16_\)(.*?)\n#ifndef", body, re.S).group(1)
    assert "launch_align<NT_, BITS_, TWO_, WS_, 1, true>" in macro and "launch_align<NT_, BITS_, TWO_, WS_>" in macro
    for line in body.splitlines():
        m = re.match(r"\s*AW_CASE\((\w+), (\d+), (true|false), (int|short), (true|false)\)", line)
        if m and m.group(1) != "AW_NT_EXPERIMENT":
            nt, bits, two, ws, w16 = int(m.group(1)), int(m.group(2)), m.group(3) == "true", m.group(4), m.group(5) == "true"
            assert w16 == (ws == "short"), line
            out |= {("full", (nt, bits, two, ws, 1)), ("score", (nt, bits, two, ws, 1))}
    for m in re.finditer(r"launch_align<AW_CLUSTER_NT, (\d), (true|false), (int|short), AW_CLUSTER_SIZE(, true)?>", body):
        out.add(("score" if m.group(4) else "full", (CLUSTER_NT, int(m.group(1)), m.group(2) == "true", m.group(3), CLUSTER_SIZE)))
    return out


def test_kernel_case_table_covers_dispatch():
    """every kernel dispatch_align can launch, in full and score-only mode, has a parity case, and no case names a kernel
    that does not exist; plan_kernel maps each case's inputs to that case"""
    parsed = _parsed_kernels()
    assert len(parsed) == 2 * len(KERNEL_CASES)
    assert parsed == {(mode, k) for k in KERNEL_CASES for mode in ("full", "score")}
    for key in KERNEL_CASES:
        ids, seqs, pairs, pen, opts = _case_inputs(key)
        clean = all(_is_clean(s) for s in seqs)
        assert clean == KERNEL_CASES[key]["clean"], key
        max_p, max_t = max(len(seqs[q]) for q, _ in pairs), max(len(seqs[t]) for _, t in pairs)
        assert plan_kernel(max_p, max_t, clean, _two(pen), opts, npairs=len(pairs)) == key, key


def test_plan_kernel_thresholds():
    """the length rules plan_kernel restates: one warp up to 1 kb, int16 rows while every offset bound holds, byte kernels never
    use 128 threads or the cluster"""
    assert plan_kernel(1024, 1024, False, True) == (32, 8, True, "int", 1)
    assert plan_kernel(1025, 1000, False, True) == (256, 8, True, "short", 1)
    assert plan_kernel(10400, 10400, False, True) == (256, 8, True, "short", 1)
    assert plan_kernel(9000, 10800, False, False) == (256, 8, False, "short", 1)
    assert plan_kernel(10600, 10600, False, True) == (256, 8, True, "int", 1)  # 3 * (plen + tlen) >= 63000
    assert plan_kernel(10660, 10500, False, True) == (256, 8, True, "int", 1)
    assert plan_kernel(10700, 10700, True, True) == (128, 2, True, "int", 1)
    assert plan_kernel(60000, 60000, True, False) == (256, 2, False, "int", 1)
    assert plan_kernel(300000, 300000, True, True, npairs=4)[4] == CLUSTER_SIZE
    assert plan_kernel(300000, 300000, False, True, npairs=4) == (256, 8, True, "int", 1)


def test_dirty_generator():
    rnd = random.Random(1)
    ids, seqs, _ = synth.generate(5, 5, 3000, 0.03)
    d = _add_dirt(rnd, seqs, events=40)
    joined = b"".join(d)
    assert b"N" in joined and any(c in joined for c in IUPAC) and re.search(rb"[acgt]{5}", joined)
    assert not all(len(a) == len(b) for a, b in zip(d, seqs))
    k = _add_dirt(random.Random(2), seqs, events=40, keep_len=True)
    assert [len(s) for s in k] == [len(s) for s in seqs] and k != seqs


def test_fast_oracle_on_dirty_input(oracle):
    """the oracle's fast mode (8-byte extend, unchecked interior loop) gives the plain oracle's PAF, scores and cells on
    N / lower-case / IUPAC input"""
    rnd = random.Random(12)
    for (n, length, d, pen) in [(8, 600, 0.05, DEFAULT), (6, 300, 0.2, EDIT), (5, 2500, 0.03, AFFINE), (4, 7000, 0.04, DEFAULT),
                                (6, 1000, 0.02, O1_GT_O2)]:
        ids, seqs, _ = synth.generate(rnd.randrange(1 << 30), n, length, d, rc_prob=0.3)
        seqs = _add_dirt(rnd, seqs, events=8)
        seqs[0] = seqs[0].lower()
        seqs[-1] = b"N" * (length // 3)
        pairs = [(i, j) for i in range(n) for j in range(n) if i != j]
        p = oracle.params(**pen)
        a = oracle.run_pairs(ids, seqs, pairs, p, use_mash=True, threads=CORES)
        b = oracle.run_pairs(ids, seqs, pairs, p, use_mash=True, threads=CORES, fast=True)
        assert a["paf"] == b["paf"] and a["scores"] == b["scores"] and a["work"]["cells"] == b["work"]["cells"]


# ---- oracle parity of every kernel -------------------------------------------------------------------------------------
def _parity(oracle, ctx, ids, seqs, pairs, pen, fast=False, n_cigar=50, n_gotoh=0, seed=0):
    """full path (PAF, score, strand vs oracle.run_pairs with mash orientation; cigar_bytes vs oracle.wfa_align on a sample of
    forward pairs) and score-only path (_run) on the same pairs"""
    ctx.load_sequences(ids, seqs)
    params = aw.make_params(**pen)
    full = ctx.align_pairs(params, pairs, flags=aw.AW_FLAG_CIGAR_BYTES)
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**pen), use_mash=True, threads=CORES, fast=fast)
    bad = [(q, t, r["status"], r["score"], s, r["paf"][-60:], e[-60:]) for r, (q, t), e, s in zip(full, pairs, exp["paf"], exp["scores"])
           if r["status"] != 0 or r["paf"] != e or r["score"] != s]
    assert not bad, f"{len(bad)}/{len(pairs)} pairs differ from the oracle, first: {bad[:2]}"
    p = oracle.params(**pen)
    rnd = random.Random(seed)
    fwd = [r for r in full if not r["is_reverse"]]
    for r in rnd.sample(fwd, min(n_cigar, len(fwd))):
        st, sc, ops, _ = oracle.wfa_align(p, seqs[r["query_idx"]], seqs[r["target_idx"]])
        assert (st, sc, ops) == (0, r["score"], r["cigar_bytes"]), (r["query_idx"], r["target_idx"])
    for r in rnd.sample(full, min(n_gotoh, len(full))):
        q, t = seqs[r["query_idx"]], seqs[r["target_idx"]]
        if r["is_reverse"]:
            q = oracle.reverse_complement(q)
        assert -r["score"] == oracle.gotoh_penalty(p, q, t)
    _run(oracle, ctx, ids, seqs, pairs, pen, exp_scores=exp["scores"], full=full)
    return full


def _ctx(opts):
    ctx = aw.Context(0)
    for k, v in opts.items():
        ctx.set_option(k, v)
    return ctx


@gpu
@pytest.mark.parametrize("key", sorted(KERNEL_CASES), ids=_case_id)
def test_kernel_case_parity(oracle, key):
    """each kernel of the case table, full and score-only, on its own inputs"""
    ids, seqs, pairs, pen, opts = _case_inputs(key)
    ctx = _ctx(opts)
    try:
        _parity(oracle, ctx, ids, seqs, pairs, pen, n_cigar=6, n_gotoh=2)
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("group", range(10))
def test_one_warp_byte_kernels_sweep(oracle, gpu_ctx, group):
    """<32, 8, *>: 2,000 pairs of lengths 1..1024 with N runs, soft-masking, IUPAC bytes, whole lower-case and all-N members,
    under each of the ten penalty sets"""
    pen = PENALTY_SETS[group]
    ids, seqs, pairs = _sweep_group(9300 + group, nfam=40, members=5, maxlen=1000, npairs=2000)
    seqs = _dirty_families(random.Random(group), seqs, 5, clip=1024)
    assert max(len(s) for s in seqs) <= 1024 and not all(_is_clean(s) for s in seqs)
    assert plan_kernel(1024, 1024, False, _two(pen))[:2] == (32, 8)
    _parity(oracle, gpu_ctx, ids, seqs, pairs, pen, n_cigar=150, n_gotoh=60, seed=group)


@gpu
@pytest.mark.parametrize("pen", [DEFAULT, AFFINE, EDIT, O1_GT_O2], ids=["default", "affine", "edit", "o1_gt_o2"])
def test_byte_kernels_int16_rows(oracle, gpu_ctx, pen):
    """<256, 8, *, short>: dirty C2 / C5-shaped pairs of 1..10 kb, mixed strands"""
    ids, seqs, rc = synth.generate(61, 12, 5000, 0.04, rc_prob=0.5)
    rnd = random.Random(62)
    seqs = _dirty_families(rnd, seqs, 4)
    seqs[3] = seqs[3][:1100]
    seqs[7] = seqs[7] + seqs[7][:4500]
    assert plan_kernel(max(map(len, seqs)), max(map(len, seqs)), False, _two(pen))[:4] == (256, 8, _two(pen), "short")
    pairs = [(i, j) for i in range(12) for j in range(12) if i != j and (i + j) % 3 == 0]
    res = _parity(oracle, gpu_ctx, ids, seqs, pairs, pen, n_cigar=10)
    assert any(r["is_reverse"] for r in res) and not all(r["is_reverse"] for r in res)


@gpu
def test_byte_kernels_int32_rows(oracle, gpu_ctx):
    """<256, 8, *, int>: the int16 boundary lengths made dirty (lengths kept), C4-shaped pairs of 24..40 kb with SVs and N
    runs, one pair above 50 kb, and ws16=0 at a few kb"""
    ids, seqs, _ = synth.generate(4242, 2, 10800, 0.02)
    a, b = _add_dirt(random.Random(3), seqs, events=12, keep_len=True)
    for x, y in ((a[:10600], b[:10600]), (a[:10700], b[:10700]), (a[:10660], b[:10500]), (a[:9000], b[:10800])):
        for pen in (DEFAULT, AFFINE):
            _parity(oracle, gpu_ctx, ["x", "y"], [x, y], [(0, 1), (1, 0)], pen, n_cigar=1)
    c, ids, seqs, _ = synth.config("C4", n=4, length=32000)
    seqs = _add_dirt(random.Random(4), seqs, events=10)
    pairs = [(0, 1), (1, 2), (2, 3), (3, 0)]
    assert plan_kernel(max(map(len, seqs)), max(map(len, seqs)), False, True) == (256, 8, True, "int", 1)
    _parity(oracle, gpu_ctx, ids, seqs, pairs, DEFAULT, fast=True, n_cigar=0)
    rnd = random.Random(5)
    root = bytes(rnd.choice(b"ACGT") for _ in range(56000))
    big = _add_dirt(rnd, [root, _mutate(rnd, root, 0.004)], events=10)
    _parity(oracle, gpu_ctx, ["b0", "b1"], big, [(0, 1)], DEFAULT, fast=True, n_cigar=0)
    ids, seqs, _ = synth.generate(66, 4, 3000, 0.04, rc_prob=0.5)
    seqs = _add_dirt(random.Random(6), seqs)
    ctx = _ctx(INT32)
    try:
        for pen in (DEFAULT, AFFINE):
            _parity(oracle, ctx, ids, seqs, [(i, j) for i in range(4) for j in range(4) if i != j], pen, n_cigar=4)
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("opts", [TPC256, dict(TPC256, **INT32)], ids=["short", "int"])
def test_single_piece_256_thread_2bit(oracle, opts):
    """<256, 2, false, short|int>: clean single-piece pairs with threads_per_cta=256"""
    ids, seqs, _ = synth.generate(71, 8, 3000, 0.05, rc_prob=0.5)
    pairs = [(i, j) for i in range(8) for j in range(8) if i != j]
    ctx = _ctx(opts)
    try:
        for pen in (AFFINE, EDIT):
            _parity(oracle, ctx, ids, seqs, pairs, pen, n_cigar=6)
    finally:
        ctx.close()


# ---- the byte kernels against the 2-bit kernels at full size -----------------------------------------------------------
DIRT_ID, DIRT = "dirt", b"ACGTNNNNacgtRYKM" * 8


def _key(r):
    return (r["query_idx"], r["target_idx"], r["status"], r["score"], r["is_reverse"], r["query_start"], r["query_end"], r["target_start"],
            r["target_end"], r["num_matches"], r["alignment_length"], r["cg"], r["paf"], r["cigar_bytes"])


def _both_contexts(ids, seqs, pairs, pen=DEFAULT, opts=None, orientation=aw.AW_ORIENT_MASH):
    """the same clean pairs in a clean context (2-bit kernels) and in one that also holds a dirty sequence no pair uses
    (every pair on the byte kernels): full results and score-only results must be identical"""
    assert all(_is_clean(s) for s in seqs)
    params = aw.make_params(**pen)
    got = []
    for extra_ids, extra in (([], []), ([DIRT_ID], [DIRT])):
        ctx = _ctx(opts or {})
        try:
            ctx.load_sequences(ids + extra_ids, seqs + extra)
            full = ctx.align_pairs(params, pairs, orientation=orientation, flags=aw.AW_FLAG_CIGAR_BYTES)
            score = ctx.align_pairs(params, pairs, orientation=orientation, flags=aw.AW_FLAG_SCORE_ONLY)
        finally:
            ctx.close()
        _check_shape(score, seqs, pairs)
        got.append(([_key(r) for r in full], [_key(r) for r in score]))
    (fc, sc), (fd, sd) = got
    bad = [(a[:5], b[:5]) for a, b in zip(fc, fd) if a != b]
    assert not bad, f"{len(bad)}/{len(pairs)} full results differ between the 2-bit and byte kernels, first: {bad[:2]}"
    assert sc == sd
    return fc


def _rand_pairs(n, k, seed):
    rnd = random.Random(seed)
    out = []
    while len(out) < k:
        a, b = rnd.randrange(n), rnd.randrange(n)
        if a != b:
            out.append((a, b))
    return out


@gpu
def test_differential_c2_full_size():
    c, ids, seqs, _ = synth.config("C2")
    _both_contexts(ids, seqs, _rand_pairs(1000, 1024, 201))


@gpu
def test_differential_c5_full_size():
    c, ids, seqs, rc = synth.config("C5")
    res = _both_contexts(ids, seqs, _rand_pairs(5000, 512, 501))
    assert any(r[4] for r in res) and not all(r[4] for r in res)


@gpu
def test_differential_c1_full_config():
    c, ids, seqs, _ = synth.config("C1")
    _both_contexts(ids, seqs, [(i, j) for i in range(16) for j in range(16) if i != j])


@gpu
def test_differential_long_pairs():
    """five 40-kb C4-shaped pairs (<128, 2, true, int> against <256, 8, true, int>) and two 120-kb pairs (the cluster kernel
    against <256, 8, true, int>)"""
    c, ids, seqs, _ = synth.config("C4", n=6, length=40000)
    _both_contexts(ids, seqs, [(i, i + 1) for i in range(5)])
    c, ids, seqs, _ = synth.config("C4", n=3, length=120000)
    assert plan_kernel(120000, 120000, True, True, CLUSTER, npairs=2)[4] == CLUSTER_SIZE
    _both_contexts(ids, seqs, [(0, 1), (2, 1)], opts=dict(CLUSTER, solo_len=3000))


@gpu
def test_dirty_context_plumbing(oracle):
    """in a context holding one dirty sequence: the retry ladder, AW_ORIENT_WFA, PAF blocks of aw_align_stream and the failure
    sentinel give what the clean context gives"""
    c, ids, seqs, rc = synth.config("C5", n=10, length=1500)
    pairs = [(i, j) for i in range(10) for j in range(10) if i != j]
    params = aw.make_params(**DEFAULT)
    ref = _both_contexts(ids, seqs, pairs)
    # retry ladder: a 48-diagonal first-try workspace
    ctx = _ctx(dict(max_wavefront_width=48))
    try:
        ctx.load_sequences(ids + [DIRT_ID], seqs + [DIRT])
        b = aw.Batch(ctx, params, pairs, flags=aw.AW_FLAG_CIGAR_BYTES)
        b.launch()
        got = b.fetch()
        st = b.stats()
        b.close()
        assert st["pairs_retried"] > 0 and st["failed_pairs"] == 0
        assert [_key(r) for r in got] == ref
    finally:
        ctx.close()
    # wfa orientation
    _both_contexts(ids, seqs, pairs, orientation=aw.AW_ORIENT_WFA)
    ctx = aw.Context(0)
    try:
        ctx.load_sequences(ids + [DIRT_ID], seqs + [DIRT])
        res = ctx.align_pairs(params, pairs, orientation=aw.AW_ORIENT_WFA)
        assert all(r["is_reverse"] == (rc[r["query_idx"]] != rc[r["target_idx"]]) for r in res)
        # PAF blocks
        lines = [r["paf"] for r in ctx.align_pairs(params, pairs)]
        assert lines == [k[12] for k in ref]
        chunks = [pairs[i:i + 37] for i in range(0, len(pairs), 37)]
        blocks = []
        ctx.align_stream(params, chunks, flags=aw.AW_FLAG_PAF_BLOCKS, block_callback=lambda b, n: blocks.append(b) and False)
        assert b"".join(blocks).decode() == "".join(l + "\n" for l in lines)
    finally:
        ctx.close()
    # failure sentinel
    ids2, s2, _ = synth.generate(808, 4, 900, 0.08)
    s2[3] = s2[0]
    p2 = [(0, 1), (0, 3), (2, 1)]
    ctx = _ctx(dict(max_wavefront_width=48, max_retry_attempts=0))
    try:
        ctx.load_sequences(ids2 + [DIRT_ID], s2 + [DIRT])
        res = ctx.align_pairs(params, p2, orientation=aw.AW_ORIENT_FORWARD)
        for r, (q, t) in zip(res, p2):
            if (q, t) == (0, 3):
                assert r["status"] == 0 and r["cg"] == f"{len(s2[0])}="
                continue
            assert r["status"] == aw.AW_EALIGN and r["score"] == 2 ** 31 - 1 and r["cg"] == ""
            assert r["paf"] == f"{ids2[q]}\t{len(s2[q])}\t0\t0\t+\t{ids2[t]}\t{len(s2[t])}\t0\t0\t0\t0\t60\tgi:f:0.000000\tcg:Z:"
    finally:
        ctx.close()


# ---- a query much longer than its target -------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("opts", [{}, TPC256, dict(TPC256, **INT32)], ids=["default", "nt256", "nt256-int32"])
def test_long_query_short_target(oracle, opts):
    """an unrelated pair whose query is three times its target (a 785-bp tandem repeat against 255 bp, the pair of the
    -x 95 byte sweep that used to fail): the wavefront reaches diagonal -plen, far below -W/2 of the full-width row the
    retry ladder allocates.  It failed as AW_EALIGN on every rung while the diagonals were split evenly around 0.  Clean
    (2-bit) and dirty (byte) contexts, both orders, full and score-only, several penalty sets."""
    rnd = random.Random(785)
    q = b"CGTG" * 196 + b"C"
    t = _clean(rnd, 110) + b"N" * 60 + _clean(rnd, 85)
    long_t = _clean(rnd, 3000)
    pairs = [(0, 1), (1, 0), (2, 3), (3, 2)]
    for seqs in ([q, t, long_t, long_t[:700]], [q, t.replace(b"N", b"A"), long_t, long_t[:700]]):
        ids = ["q", "t", "lq", "lt"]
        for pen in (PENALTY_SETS[1], DEFAULT, AFFINE, EDIT):
            ctx = _ctx(opts)
            try:
                ctx.load_sequences(ids, seqs)
                res = ctx.align_pairs(aw.make_params(**pen), pairs, orientation=aw.AW_ORIENT_FORWARD, flags=aw.AW_FLAG_CIGAR_BYTES)
                exp = [oracle.wfa_align(oracle.params(**pen), seqs[a], seqs[b]) for a, b in pairs]
                assert [(r["status"], r["score"], r["cigar_bytes"]) for r in res] == [(0, sc, ops) for _, sc, ops, _ in exp], pen
                _run(oracle, ctx, ids, seqs, pairs, pen, orientation=aw.AW_ORIENT_FORWARD, exp_scores=[e[1] for e in exp], full=res)
            finally:
                ctx.close()


# ---- single-pair API ---------------------------------------------------------------------------------------------------
@gpu
def test_single_pair_api_dirty(oracle, gpu_ctx):
    """Aligner (both scopes) and the C++ mirror's align_sequences on lower-case / N / IUPAC pairs of 50 bp .. 12 kb"""
    from allwave_b200 import hostlib as H

    rnd = random.Random(90)
    cases = []
    for L in (50, 120, 700, 1500, 5000, 12000):
        a = bytes(rnd.choice(b"ACGT") for _ in range(L))
        x, y = _add_dirt(rnd, [a, _mutate(rnd, a, 0.04)], events=4 + L // 1000)
        cases.append((x, y))
    cases += [(cases[2][0].lower(), cases[2][1]), (b"N" * 300, cases[1][1]), (b"acgtRYKMSW" * 20, b"ACGTRYKMSW" * 20)]
    for args, pen in (((5, 8, 2, 24, 1), DEFAULT), ((4, 6, 2), dict(mismatch=4, gap_open=6, gap_extend=2, gap2_open=None, gap2_extend=None))):
        al = aw.Aligner(gpu_ctx, *args)
        try:
            for x, y in cases:
                st, sc, ops, _ = oracle.wfa_align(oracle.params(**pen), x, y)
                al.set_alignment_scope(aw.AW_SCOPE_ALIGNMENT)
                assert al.align(x, y) == 0 and (al.score(), al.cigar()) == (sc, ops), (len(x), len(y))
                al.set_alignment_scope(aw.AW_SCOPE_SCORE)
                assert al.align(x, y) == 0 and (al.score(), al.cigar()) == (sc, b"")
        finally:
            al.close()
    for mode, pen in ((H.MODE_EDIT, (3, 0, 0, 0, 0)), (H.MODE_AFFINE, (4, 6, 2, 0, 0)), (H.MODE_AFFINE2P, (5, 8, 2, 24, 1))):
        p = {H.MODE_EDIT: oracle.params(0, 3, 3, 3, None, None), H.MODE_AFFINE: oracle.params(0, 4, 6, 2, None, None),
             H.MODE_AFFINE2P: oracle.params(0, 5, 8, 2, 24, 1)}[mode]
        for x, y in cases:
            r = H.align_sequences(gpu_ctx, x, y, *pen, mode=mode)
            st, sc, ops, _ = oracle.wfa_align(p, x, y)
            assert st == 0 and r["score"] == sc and r["cigar"] == oracle.cigar_string(ops)
            assert (r["matches"], r["mismatches"], r["insertions"], r["deletions"]) == (ops.count(b"M"), ops.count(b"X"), ops.count(b"D"), ops.count(b"I"))


# ---- sketches, Jaccard, orientation, divergence ------------------------------------------------------------------------
KS = (1, 7, 8, 9, 15, 16, 31)
SIZES = (1, 7, 1000, 1024, 1025, 4096)


def _clean(rnd, n):
    return bytes(rnd.choice(b"ACGT") for _ in range(n))


def _sketch_set(k):
    """sequences at the edges of the sketch kernel for k-mer size k"""
    rnd = random.Random(k)
    seqs = [b"", _clean(rnd, max(0, k - 1)), _clean(rnd, k), _clean(rnd, k + 1)]
    for s in SIZES:  # s-1, s and s+1 valid k-mers: the take_all boundary of every sketch size
        for nk in (s - 1, s, s + 1):
            if nk <= 0:
                continue
            seqs.append(_clean(rnd, nk + k - 1))
            first = min(nk, 1 + nk // 2)  # the same count split by an N, inside a longer N-padded sequence
            seqs.append(b"N" * 37 + _clean(rnd, first + k - 1) + b"N" + _clean(rnd, nk - first + k - 1) + b"n" * 211)
    seqs += [b"N" * 2000, (_clean(rnd, k - 1) + b"N") * (3000 // k + 1) if k > 1 else b"N" * 3000, b"A" * 5000, b"AC" * 2500]
    a = _clean(rnd, 5000)
    dirty = _add_dirt(rnd, [a, _mutate(rnd, a, 0.03)], events=12)
    half = bytes(c | 0x20 if i % 2 else c for i, c in enumerate(a))
    pal = a[:1500] + bytes(reversed(a[:1500].translate(bytes.maketrans(b"ACGT", b"TGCA"))))
    seqs += dirty + [a.lower(), half, a, pal, _clean(rnd, 1000000)]
    if len(seqs) % 32 == 0:
        seqs.append(_clean(rnd, 333))
    return ["k%d_%d" % (k, i) for i in range(len(seqs))], seqs


@gpu
@pytest.mark.parametrize("k", KS)
def test_canonical_sketches_and_jaccard(oracle, gpu_ctx, k):
    """get_sketch (canonical) equals oracle.sketch at every sketch size, mash_jaccard_counts equals oracle.jaccard_counts"""
    ids, seqs = _sketch_set(k)
    assert len(seqs) % 32 != 0
    gpu_ctx.load_sequences(ids, seqs)
    for size in SIZES:
        exp = [oracle.sketch(s, k=k, size=size, canonical=True) for s in seqs]
        got = [gpu_ctx.get_sketch(i, canonical=True, k=k, size=size) for i in range(len(seqs))]
        bad = [(i, len(seqs[i]), len(g), len(e)) for i, (g, e) in enumerate(zip(got, exp)) if g != e]
        assert not bad, (k, size, bad[:4])
        if size in (7, 1000, 4096):
            inter, uni = gpu_ctx.mash_jaccard_counts(k=k, size=size)
            for i in range(len(seqs)):
                for j in range(i + 1, len(seqs)):
                    assert (int(inter[i, j]), int(uni[i, j])) == oracle.jaccard_counts(exp[i], exp[j]) == (int(inter[j, i]), int(uni[j, i])), (k, size, i, j)


@gpu
def test_stranded_sketches_orientation_divergence(oracle, gpu_ctx):
    """forward and reverse-complement sketches (k 15, size 1000), orient_pairs (ties fj == rj included) and estimate_divergence
    (a restatement of aw_divergence_kernel on the oracle's sketches, within one float32 ulp)"""
    ids, seqs = _sketch_set(15)
    gpu_ctx.load_sequences(ids, seqs)
    fwd = [oracle.sketch(s) for s in seqs]
    rev = [oracle.sketch(oracle.reverse_complement(s)) for s in seqs]
    for i in range(len(seqs)):
        assert gpu_ctx.get_sketch(i) == fwd[i], i
        assert gpu_ctx.get_sketch(i, reverse_complement=True) == rev[i], i
    small = [i for i, s in enumerate(seqs) if len(s) < 100000]
    pairs = [(q, t) for q in small[::2] for t in small if q != t]
    kfree = [i for i in small if not fwd[i]]
    pal = _palindrome_index(seqs)
    pairs += [(kfree[0], kfree[1]), (kfree[1], kfree[0])] + [(pal, t) for t in small if t != pal]
    assert gpu_ctx.orient_pairs(pairs) == [oracle.orientation_mash(seqs[q], seqs[t]) for q, t in pairs]
    est = gpu_ctx.estimate_divergence(pairs)
    for (q, t), g in zip(pairs, est):
        fi, fu = oracle.jaccard_counts(fwd[q], fwd[t])
        ri, ru = oracle.jaccard_counts(rev[q], fwd[t])
        j = max(fi / fu if fu else 0.0, ri / ru if ru else 0.0)
        d = 1.0 if j <= 0.0 else -math.log(2.0 * j / (1.0 + j)) / 15.0
        e = np.float32(min(max(d, 0.0), 1.0))
        ulps = abs(int(np.float32(g).view(np.int32)) - int(e.view(np.int32)))
        assert ulps <= 1, (q, t, g, float(e))
    assert est[pairs.index((kfree[0], kfree[1]))] == 1.0


def _palindrome_index(seqs):
    for i, s in enumerate(seqs):
        if len(s) == 3000 and s == s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA")):
            return i
    raise AssertionError("no reverse-complement palindrome in the set")


@gpu
def test_cli_dirty_fasta(oracle, tmp_path):
    """the CLI on a dirty FASTA, plain and gzipped: -p none gives the oracle's lines, --mash-matrix the oracle's table"""
    ids, seqs, _ = synth.generate(95, 6, 2500, 0.04, rc_prob=0.5)
    seqs = _add_dirt(random.Random(95), seqs, events=10)
    seqs[2] = seqs[2].lower()
    text = "".join(f">{i}\n{s.decode()}\n" for i, s in zip(ids, seqs))
    plain, gz = tmp_path / "in.fa", tmp_path / "in.fa.gz"
    plain.write_text(text)
    with gzip.open(gz, "wt") as f:
        f.write(text)
    exe = os.path.join(os.path.dirname(aw._cabi.so_path()), "allwave")
    pairs = [(i, j) for i in range(6) for j in range(6) if i != j]
    want = oracle.run_pairs(ids, seqs, pairs, oracle.params(**DEFAULT), use_mash=True, threads=CORES)["paf"]
    for fa in (plain, gz):
        out = tmp_path / "o.paf"
        subprocess.check_call([exe, "-i", str(fa), "-o", str(out), "-p", "none", "-x", "90%", "--no-progress"])
        assert out.read_text().splitlines() == want, fa
        rows = subprocess.run([exe, "-i", str(fa), "--mash-matrix"], capture_output=True, text=True, check=True).stdout.splitlines()
        assert rows[0].split("\t") == ["sequence"] + ids and len(rows) == 7
        sk = [oracle.sketch(s, canonical=True) for s in seqs]
        for i in range(6):
            row = rows[1 + i].split("\t")
            assert row[0] == ids[i]
            for j in range(6):
                exp = 0.0
                if i != j:
                    inter, uni = oracle.jaccard_counts(sk[i], sk[j])
                    jac = inter / uni if uni else 0.0
                    exp = 1.0 if jac <= 0.0 else (-1.0 / 15.0) * math.log(2.0 * jac / (1.0 + jac))
                assert row[1 + j] == f"{exp:.6f}", (i, j)
