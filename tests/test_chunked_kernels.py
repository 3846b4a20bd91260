"""The chunked 2-bit alignment kernels (<128|256, 2, *, short|int>) under every penalty set, on mixed-length batches and
at the int16 limits.

plan_launch picks one kernel per batch from the batch's longest pair, so a single long pair sends every short pair beside
it to the chunked kernels: their vector cell loop, arithmetic trimming, rescans, block-maxima overlap scan, int16 null
drift and warp-parallel leaves.  The sweeps of test_gpu_round2 never get there (every pair <= 1 kb runs on the one-warp
kernel).  Here a *carrier* -- one pair of two identical clean sequences, one diagonal for the aligner -- is appended to a
batch of short pairs and its length alone picks the kernel.  Every comparison is bit-exact against the CPU oracle: PAF
line, score and strand of every pair, CIGAR bytes on a sample of forward pairs, the Gotoh DP on a sample, and the
score-only path on the same pairs."""
import random
import re

import pytest

import allwave_b200 as aw
from allwave_b200 import synth
from test_byte_input import _ctx, _parity, _two, plan_kernel
from test_gpu_round2 import CORES, DEFAULT, PENALTY_SETS, _mutate, _sweep_group
from test_score_only import _check_shape, _same

gpu = pytest.mark.gpu
AFFINE = PENALTY_SETS[3]       # -x 65: single piece, e = 1
EDIT = PENALTY_SETS[4]
O_ZERO = PENALTY_SETS[8]       # o = 0
# match < 0: the three bonus sets of test_match_score_bonus
BONUS_SETS = [dict(match=-1, mismatch=4, gap_open=6, gap_extend=2, gap2_open=None, gap2_extend=None),
              dict(match=-2, mismatch=5, gap_open=8, gap_extend=2, gap2_open=24, gap2_extend=1),
              dict(match=-3, mismatch=2, gap_open=1, gap_extend=1, gap2_open=None, gap2_extend=None)]
GROUPS = PENALTY_SETS + BONUS_SETS


def _clean(rnd, n):
    return bytes(rnd.choice(b"ACGT") for _ in range(n))


# ---- routes: the carrier appended to a batch, the options, and the kernel plan_launch gives the batch ------------------
CARRIER_LENS = (2000, 11000, 60000)
# name -> (carrier length or None, set_option values, (NT, BITS, WS) of the launch)
ROUTES = {
    "c2k": (2000, {}, (128, 2, "short")),
    "c11k": (11000, {}, (128, 2, "int")),      # 3 * (11000 + 11000) >= 63000
    "c60k": (60000, {}, (256, 2, "int")),      # > 50 kb, below cluster_min_len
    "nt256": (None, dict(threads_per_cta=256), (256, 2, "short")),  # no natural route reaches it
}
# the int16 and int32 128-thread routes again, with the retry ladder off and a 64 MB history arena: every pair of these
# batches has a full-width first-try workspace (W = full_w while max_p + max_t <= 65536), so none may report AW_EWORKSPACE
FIRST_TRY = dict(max_retry_attempts=0, hist_mb=64)
ROUTES["c2k-first-try"] = (2000, FIRST_TRY, (128, 2, "short"))
ROUTES["c11k-first-try"] = (11000, FIRST_TRY, (128, 2, "int"))


def _edge_pool(rnd):
    """sequences and pairs at the edges: empty and 1-bp sequences, every length 1..40, both sides of the 16-base 2-bit word
    (15/16/17, 31/32/33), of the base-case length 100 and of 256; related, unrelated and pure-gap pairs"""
    seqs, pairs = [b"", b"A"], [(0, 1), (1, 0)]
    for L in list(range(1, 41)) + [15, 16, 17, 31, 32, 33, 99, 100, 101, 255, 256, 257]:
        a = _clean(rnd, L)
        b = _mutate(rnd, a, rnd.choice([0.05, 0.2])) or b"C"
        i = len(seqs)
        seqs += [a, b, _clean(rnd, L), a[: L // 2], a + _clean(rnd, 1 + L // 3)]
        pairs += [(i, i + 1), (i + 1, i), (i, i + 2), (i, 0), (0, i), (i, i + 3), (i + 3, i), (i + 4, i)]
    return seqs, pairs


def _group_inputs(group):
    """one sweep group of ~4,000 pairs (lengths 1..400 and then some), the edge pool, and the three carriers, loaded
    together: ids, seqs, the shared pairs, and {carrier length: carrier pair}"""
    ids, seqs, pairs = _sweep_group(9500 + group, npairs=4000)
    rnd = random.Random(group)
    e_seqs, e_pairs = _edge_pool(rnd)
    n = len(seqs)
    seqs = seqs + e_seqs
    pairs = pairs + [(n + a, n + b) for a, b in e_pairs]
    carriers = {}
    for L in CARRIER_LENS:
        c = _clean(random.Random(L), L)
        carriers[L] = (len(seqs), len(seqs) + 1)
        seqs += [c, c]
    return ["w%05d" % i for i in range(len(seqs))], seqs, pairs, carriers


def _route_pairs(name, pairs, carriers):
    L = ROUTES[name][0]
    return pairs + ([carriers[L]] if L else [])


def _route_kernel(name, seqs, pairs, two):
    L, opts, _ = ROUTES[name]
    max_p, max_t = max(len(seqs[q]) for q, _ in pairs), max(len(seqs[t]) for _, t in pairs)
    return plan_kernel(max_p, max_t, True, two, opts, npairs=len(pairs))


def test_carrier_routes():
    """CPU: each carrier (or forced CTA size) sends the whole batch to the kernel its route names, for one- and two-piece
    penalties, and the batch without a carrier would have run on the one-warp kernel"""
    for group in (0, 4):
        ids, seqs, pairs, carriers = _group_inputs(group)
        short = max(max(len(seqs[q]), len(seqs[t])) for q, t in pairs)
        assert short <= 1024 and short < min(CARRIER_LENS)
        for two in (True, False):
            assert _route_kernel("c2k", seqs, pairs, two) == (32, 2, two, "int", 1)
            for name, (_, _, (nt, bits, ws)) in ROUTES.items():
                assert _route_kernel(name, seqs, _route_pairs(name, pairs, carriers), two) == (nt, bits, two, ws, 1), (name, two)
    assert {_two(p) for p in GROUPS} == {True, False}


def _batch(ctx, pen, pairs, flags):
    b = aw.Batch(ctx, aw.make_params(**pen), pairs, flags=flags)
    try:
        b.launch()
        res = b.fetch()
        st = b.stats()
    finally:
        b.close()
    return res, st


def _group_id(g):
    return "pen%d" % g if g < len(PENALTY_SETS) else "bonus%d" % (g - len(PENALTY_SETS))


@gpu
@pytest.mark.parametrize("group", range(len(GROUPS)), ids=_group_id)
def test_mixed_length_sweep(oracle, group):
    """~4,300 short and edge pairs on every chunked route under one penalty set: full results (PAF, score, strand) against
    the oracle for every pair, CIGAR bytes on 100 forward pairs, Gotoh on 50, score-only against both; the first-try routes
    must align every pair on their first attempt"""
    pen = GROUPS[group]
    ids, seqs, pairs, carriers = _group_inputs(group)
    every = pairs + [carriers[L] for L in CARRIER_LENS]
    exp = oracle.run_pairs(ids, seqs, every, oracle.params(**pen), use_mash=True, threads=CORES)
    exp_of = {pq: (line, s) for pq, line, s in zip(every, exp["paf"], exp["scores"])}
    p = oracle.params(**pen)
    rnd = random.Random(group)
    ops_of = {}
    gotoh = rnd.sample(range(len(pairs)), 50)
    for name in ROUTES:
        rp = _route_pairs(name, pairs, carriers)
        ctx = _ctx(ROUTES[name][1])
        try:
            ctx.load_sequences(ids, seqs)
            full, st = _batch(ctx, pen, rp, aw.AW_FLAG_CIGAR_BYTES)
            score, st_s = _batch(ctx, pen, rp, aw.AW_FLAG_SCORE_ONLY)
        finally:
            ctx.close()
        bad = [(q, t, r["status"], r["score"], exp_of[(q, t)][1], r["paf"][-60:], exp_of[(q, t)][0][-60:])
               for r, (q, t) in zip(full, rp) if r["status"] != 0 or (r["paf"], r["score"]) != exp_of[(q, t)]]
        assert not bad, f"{name}: {len(bad)}/{len(rp)} pairs differ from the oracle, first: {bad[:2]}"
        _check_shape(score, seqs, rp)
        _same(score, full)
        if name.endswith("first-try"):
            for s in (st, st_s):
                assert s["pairs_retried"] == 0 and s["failed_pairs"] == 0, (name, s)
        fwd = [i for i, r in enumerate(full[: len(pairs)]) if not r["is_reverse"]]
        for i in random.Random(group).sample(fwd, min(100, len(fwd))):
            q, t = pairs[i]
            if (q, t) not in ops_of:
                st_o, sc, ops, _ = oracle.wfa_align(p, seqs[q], seqs[t])
                ops_of[(q, t)] = (st_o, sc, ops)
            assert ops_of[(q, t)] == (0, full[i]["score"], full[i]["cigar_bytes"]), (name, q, t)
        for i in gotoh if not pen.get("match") else ():  # the Gotoh DP has no match bonus
            r = full[i]
            qs, ts = seqs[r["query_idx"]], seqs[r["target_idx"]]
            if r["is_reverse"]:
                qs = oracle.reverse_complement(qs)
            assert -r["score"] == oracle.gotoh_penalty(p, qs, ts), (name, pairs[i])


@gpu
@pytest.mark.parametrize("pen,inputs,bad", [
    (EDIT, lambda: _group_inputs(4)[:3], [(76, 79), (79, 76), (155, 109)]),
    (BONUS_SETS[1], lambda: _group_inputs(11)[:3], [(47, 41), (129, 119), (69, 47)]),
    (EDIT, lambda: _sweep_group(9104, npairs=2000), [(153, 96)]),
    (O_ZERO, lambda: _sweep_group(9108, npairs=2000), [(8, 83), (32, 59)]),
], ids=["edit-sweep", "bonus1-sweep", "edit-score-only-sweep", "o0-score-only-sweep"])
def test_256_thread_leaf_runs_through_retry(oracle, pen, inputs, bad):
    """divergent pairs of 40..610 bp whose warp-parallel leaves need more CIGAR runs than the eighth of the run buffer a
    256-thread CTA gives each leaf on the first try: they report AW_EWORKSPACE there, and the retry ladder must give the
    leaves room (it used to keep the run buffer at its first-try size, so these pairs failed on every rung as AW_EALIGN).
    The pairs come from this file's EDIT and match = -2 sweep groups and from test_sweep_three_kernels' EDIT and o = 0 groups."""
    ids, seqs, _ = inputs()
    exp = oracle.run_pairs(ids, seqs, bad, oracle.params(**pen), use_mash=True, threads=CORES)
    ctx = _ctx(dict(threads_per_cta=256))
    try:
        ctx.load_sequences(ids, seqs)
        res, st = _batch(ctx, pen, bad, aw.AW_FLAG_CIGAR_BYTES)
    finally:
        ctx.close()
    assert [(r["status"], r["paf"], r["score"]) for r in res] == [(0, e, s) for e, s in zip(exp["paf"], exp["scores"])]
    assert st["pairs_retried"] > 0 and st["failed_pairs"] == 0, st


# ---- the int16 limits --------------------------------------------------------------------------------------------------
# plan_launch keeps int16 rows while 2t + p < 32000, 2p + t < 32000 and 3(p + t) < 63000.  Each pair meets one bound (or two)
# with the least slack the lengths allow, and its partner misses it by one base.
LIMIT_PAIRS = [
    ((10499, 10499), "short"), ((10500, 10500), "int"),    # 3(p + t) = 62994 | 63000
    ((9999, 11000), "short"), ((10000, 11000), "int"),     # 2t + p = 31999 and 3(p + t) = 62997 | 32000
    ((11000, 9999), "short"), ((11000, 10000), "int"),     # 2p + t, the same the other way round
    ((3199, 14400), "short"), ((3200, 14400), "int"),      # 2t + p = 31999 | 32000: a short query against a long target
]


@gpu
@pytest.mark.parametrize("pen", [DEFAULT, EDIT, AFFINE, O_ZERO], ids=["default", "edit", "x65", "o0"])
def test_int16_limits(oracle, pen):
    """pairs of one seeded root at ~2 % divergence on both sides of every int16 bound: oracle parity (full and score-only),
    and the same results with int16 rows switched off"""
    rnd = random.Random(16000)
    root = _clean(rnd, 16000)
    mut = _mutate(rnd, root, 0.02)
    assert len(mut) >= 14400
    two = _two(pen)
    for (p, t), ws in LIMIT_PAIRS:
        assert plan_kernel(p, t, True, two) == (128, 2, two, ws, 1), (p, t)
        assert plan_kernel(p, t, True, two, dict(ws16=0)) == (128, 2, two, "int", 1)
        seqs = [root[:p], mut[:t]]
        got = []
        for opts in ({}, dict(ws16=0)):
            ctx = _ctx(opts)
            try:
                full = _parity(oracle, ctx, ["x", "y"], seqs, [(0, 1)], pen, fast=True, n_cigar=1 if not got else 0)
            finally:
                ctx.close()
            got.append([(r["status"], r["score"], r["is_reverse"], r["paf"], r["cigar_bytes"]) for r in full])
        assert got[0] == got[1], (p, t)


# ---- realistic depth ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("group", range(len(PENALTY_SETS)))
def test_c2_c5_shapes_every_penalty_set(oracle, gpu_ctx, group):
    """C2-shaped (10 kb, 5 %) and C5-shaped (5 kb, 3 %, mixed strands) pairs with the natural kernel choice: deep recursion,
    warp-parallel leaves and the overlap scan under every penalty set"""
    pen = PENALTY_SETS[group]
    for name, length in (("C2", 10000), ("C5", 5000)):
        c, ids, seqs, _ = synth.config(name, n=6, length=length)
        pairs = [(i, (i + d) % 6) for i in range(6) for d in (1, 2)]
        assert plan_kernel(max(map(len, seqs)), max(map(len, seqs)), True, _two(pen))[:2] == (128, 2)
        _parity(oracle, gpu_ctx, ids, seqs, pairs, pen, fast=True, n_cigar=1, seed=group)


# ---- gi:f rounding on exact ties ---------------------------------------------------------------------------------------
# (L, substitutions): m / L = (L - k) / L.  L = 128, 256: binary-exact ties (odd multiples of 1/128, e.g. 127/128 -> 0.992188,
# 125/128 -> 0.976562) and non-ties; L = 640, 3200: every odd m is a decimal tie that is not binary-exact, so the double
# decides; L = 10112 = 128 * 79: binary-exact ties at m = 79 * odd
TIE_CASES = [(128, k) for k in (1, 2, 3, 5)] + [(256, k) for k in (2, 6, 1, 3)] + [(640, k) for k in (1, 3, 5, 15)] + \
            [(3200, k) for k in (1, 3, 7, 25)] + [(10112, k) for k in (79, 237, 1, 2)]


@gpu
def test_identity_rounding_ties(oracle):
    """clean pairs with k spaced substitutions (x = 5 is below the cost of any gap pair, so the alignment is L columns with
    L - k matches): gi:f equals Python's '%.6f' of the exact double and the oracle's line, on the one-warp and chunked
    emitters"""
    rnd = random.Random(128)
    seqs, pairs = [], []
    for L, k in TIE_CASES:
        a = bytearray(_clean(rnd, L))
        b = bytearray(a)
        for i in range(k):
            pos = (i * L) // k + L // (2 * k)
            b[pos] = b"ACGT"[(b"ACGT".index(b[pos]) + 1 + rnd.randrange(3)) % 4]
        pairs.append((len(seqs), len(seqs) + 1))
        seqs += [bytes(a), bytes(b)]
    carriers = {}
    for L in (2000, 11000):
        c = _clean(random.Random(L), L)
        carriers[L] = (len(seqs), len(seqs) + 1)
        seqs += [c, c]
    ids = ["t%03d" % i for i in range(len(seqs))]
    small = [pq for pq, (L, _) in zip(pairs, TIE_CASES) if L <= 640]
    batches = [(small, (32, 2, True, "int", 1)), (pairs + [carriers[2000]], (128, 2, True, "short", 1)),
               (pairs + [carriers[11000]], (128, 2, True, "int", 1))]
    want = dict(zip(pairs, TIE_CASES))
    ctx = aw.Context(0)
    try:
        ctx.load_sequences(ids, seqs)
        for bp, kernel in batches:
            assert plan_kernel(max(len(seqs[q]) for q, _ in bp), max(len(seqs[t]) for _, t in bp), True, True) == kernel
            exp = oracle.run_pairs(ids, seqs, bp, oracle.params(**DEFAULT), use_mash=True, threads=CORES)["paf"]
            res, st = _batch(ctx, DEFAULT, bp, 0)
            for r, pq, e in zip(res, bp, exp):
                assert r["status"] == 0 and r["paf"] == e, (kernel, pq, r["paf"][-80:], e[-80:])
                if pq in want:
                    L, k = want[pq]
                    assert (r["num_matches"], r["alignment_length"], r["is_reverse"]) == (L - k, L, False), (L, k)
                    gi = re.search(r"\tgi:f:([0-9.]+)\t", r["paf"]).group(1)
                    assert gi == "%.6f" % ((L - k) / L), (kernel, L, k, gi)
    finally:
        ctx.close()
