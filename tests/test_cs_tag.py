"""The cs:Z: difference string (AW_FLAG_CS, AW_FLAG_CS_LONG, the CLI's --cs): minimap2's convention, built on the GPU.

The reference is the oracle's C restatement (tests/oracle_cs.c through tests/oracle_cs.py): `awo_cs_string` computes the
tag from WFA2 op letters (M X I D, one per column; I consumes a target base, D a query base) and the two sequences, and
`awo_alignment_to_paf_cs` appends it to the oracle's PAF line.  `py_cs_string` below restates the tag once more in Python,
as a cross-check of the C code.  The CPU tests hold the oracle to known answers and to its own alignments by round trip.
The GPU tests hold every route of the library to it: a line with the flag must be the same pair's line without the flag +
"\\tcs:Z:" + the oracle's tag of that line's CIGAR, whose line is the oracle's."""
import gzip
import json
import os
import random
import re
import subprocess

import pytest

import allwave_b200 as aw
from allwave_b200 import synth
import oracle_cs
from test_gpu_round2 import CORES, DEFAULT, EDIT, _mutate

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BONUS = dict(match=-2, mismatch=5, gap_open=8, gap_extend=2, gap2_open=24, gap2_extend=1)
PENS = {"default": DEFAULT, "edit": EDIT, "bonus": BONUS}
CS, CS_LONG = aw.AW_FLAG_CS, aw.AW_FLAG_CS | aw.AW_FLAG_CS_LONG


# ---- the reference, its cross-check and its inverses --------------------------------------------------------------------
def py_cs_string(ops: bytes, query: bytes, target: bytes, long_form=False) -> str:
    """the tag of the alignment `ops` (WFA2 letters) of the oriented query against the target, restated in Python"""
    out, q, t = [], 0, 0
    for m in re.finditer(rb"M+|X|I+|D+", ops):
        op, n = m.group()[:1], len(m.group())
        if op == b"M":
            out.append(b"=" + target[t:t + n].upper() if long_form else b":%d" % n)
            q, t = q + n, t + n
        elif op == b"X":
            out.append(b"*" + target[t:t + 1].lower() + query[q:q + 1].lower())
            q, t = q + 1, t + 1
        elif op == b"I":
            out.append(b"-" + target[t:t + n].lower())
            t += n
        else:
            out.append(b"+" + query[q:q + n].lower())
            q += n
    assert (q, t) == (len(query), len(target)), "the ops do not consume both sequences"
    return b"".join(out).decode("latin-1")


def cs_string(ops: bytes, query: bytes, target: bytes, long_form=False) -> str:
    """the oracle's tag (awo_cs_string), which the Python restatement must agree with"""
    tag = oracle_cs.cs_string(ops, query, target, long_form)
    assert tag == py_cs_string(ops, query, target, long_form)
    return tag


def cg_ops(cg: str) -> bytes:
    """the WFA2 op bytes of a cg:Z: value (PAF I = WFA2 D, PAF D = WFA2 I)"""
    letter = {"=": b"M", "X": b"X", "I": b"D", "D": b"I"}
    return b"".join(letter[op] * int(n) for n, op in re.findall(r"(\d+)([=XID])", cg))


def _tokens(tag):
    toks = re.findall(r"([=:*+\-])([^=:*+\-]*)", tag)
    assert "".join(k + v for k, v in toks) == tag, tag
    return toks


def tag_ops(tag) -> bytes:
    """the columns a tag describes, as WFA2 op bytes"""
    out = []
    for k, v in _tokens(tag):
        assert v, tag
        if k == ":":
            out.append(b"M" * int(v))
        elif k == "=":
            out.append(b"M" * len(v))
        elif k == "*":
            assert len(v) == 2, tag
            out.append(b"X")
        else:
            out.append((b"D" if k == "+" else b"I") * len(v))
    return b"".join(out)


def rebuild(tag, target=None):
    """(target, oriented query) from a long tag alone, or from a short tag and the target"""
    tt, qq, t = [], [], 0
    for k, v in _tokens(tag):
        if k == ":":
            seg = target[t:t + int(v)].decode("latin-1")
            tt.append(seg)
            qq.append(seg)
            t += int(v)
        elif k == "=":
            tt.append(v)
            qq.append(v)
            t += len(v)
        elif k == "*":
            tt.append(v[0])
            qq.append(v[1])
            t += 1
        elif k == "+":
            qq.append(v)
        else:
            tt.append(v)
            t += len(v)
    return "".join(tt), "".join(qq)


def check_tag(short, long_, ops, query, target):
    """both forms against the converter, their columns against ops, and the sequences they rebuild (up to case)"""
    assert short == cs_string(ops, query, target) and long_ == cs_string(ops, query, target, True)
    assert tag_ops(short) == ops and tag_ops(long_) == ops
    t, q = rebuild(long_)
    assert (t.upper(), q.upper()) == (target.decode("latin-1").upper(), query.decode("latin-1").upper())
    t, q = rebuild(short, target)
    assert (t.upper(), q.upper()) == (target.decode("latin-1").upper(), query.decode("latin-1").upper())


# ---- CPU: known answers --------------------------------------------------------------------------------------------------
KNOWN = [
    # (target, oriented query, cg:Z:, short, long)
    (b"ACGTACGTAA", b"ACGCACGGGTA", "3=1X3=2I1=1D1=", ":3*tc:3+gg:1-a:1", "=ACG*tc=ACG+gg=T-a=A"),
    (b"ACGTTGCA", b"ACGTTGCA", "8=", ":8", "=ACGTTGCA"),
    (b"", b"", "", "", ""),
    (b"", b"ACG", "3I", "+acg", "+acg"),
    (b"ACG", b"", "3D", "-acg", "-acg"),
    (b"AAGG", b"AACCT", "2=2I1X1D", ":2+cc*gt-g", "=AA+cc*gt-g"),
    (b"AGTA", b"CGAA", "1X1=1X1=", "*ac:1*ta:1", "*ac=G*ta=A"),
    (b"AGTCA", b"CTACA", "1X1X1X2=", "*ac*gt*ta:2", "*ac*gt*ta=CA"),
    (b"ACGTT", b"AGGCC", "1=2I2D2X", ":1+gg-cg*tc*tc", "=A+gg-cg*tc*tc"),
    (b"ACNTa", b"ACNTA", "4=1X", ":4*aa", "=ACNT*aa"),
    (b"acgtN", b"acgtN", "5=", ":5", "=ACGTN"),
    (b"ACRYT", b"AcRkT", "1=1X1=1X1=", ":1*cc:1*yk:1", "=A*cc=R*yk=T"),
]


def test_known_answers():
    """the worked example of the tag's definition, all-match, empty sides, pure gaps, runs of X, I next to D, and N,
    IUPAC, lower-case and case-only-mismatch bytes"""
    for target, query, cg, short, long_ in KNOWN:
        ops = cg_ops(cg)
        assert (cs_string(ops, query, target), cs_string(ops, query, target, True)) == (short, long_), cg
        check_tag(short, long_, ops, query, target)


def test_round_trip_oracle_alignments(oracle):
    """about 2,000 oracle alignments: random related and unrelated pairs of 0..300 bp under four penalty sets (two with a
    match bonus), mash orientation, which reverse-complements the query of about one pair in seven"""
    rnd = random.Random(2026)
    sets = [DEFAULT, EDIT, BONUS, dict(match=-1, mismatch=4, gap_open=6, gap_extend=2, gap2_open=None, gap2_extend=None)]
    n = n_rev = 0
    for k in range(2000):
        L = rnd.choice([0, 1, 2, 5, 16, 33, rnd.randint(1, 300)])
        a = bytes(rnd.choice(b"ACGT") for _ in range(L))
        b = _mutate(rnd, a, rnd.choice([0.0, 0.05, 0.2])) if rnd.random() < 0.8 else bytes(rnd.choice(b"ACGT") for _ in range(rnd.randint(0, 300)))
        if rnd.random() < 0.5:
            b = oracle.reverse_complement(b)
        p = oracle.params(**sets[k % len(sets)])
        r = oracle.align_pair(b, a, 0, 1, p, use_mash=True)
        query = oracle.reverse_complement(b) if r["is_reverse"] else b
        ops = r["cigar_bytes"]
        short, long_ = cs_string(ops, query, a), cs_string(ops, query, a, True)
        check_tag(short, long_, ops, query, a)
        assert cg_ops(oracle.cigar_string(ops)) == ops
        if k % 10 == 0:  # the oracle's PAF line with the cs column
            line = oracle.align_pair(b, a, 0, 1, p, use_mash=True, qname="q", tname="t")["paf"]
            for tag, lf in ((short, False), (long_, True)):
                assert oracle_cs.align_pair_paf(b, a, 0, 1, p, "q", "t", long_form=lf) == line + "\tcs:Z:" + tag
        n += 1
        n_rev += bool(r["is_reverse"])
    assert n == 2000 and n_rev > 200


# ---- CPU: the CLI's --cs ------------------------------------------------------------------------------------------------
def _exe():
    return os.path.join(ROOT, "allwave_b200", "allwave")


def test_cli_cs_arguments(tmp_path):
    """--cs=bogus is an argument error; --cs, --cs=short and --cs=long pass argument parsing and reach the device step"""
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nACGTACGT\n>b\nACGTACGA\n")
    bad = subprocess.run([_exe(), "-i", str(fa), "--cs=bogus"], capture_output=True, text=True)
    assert bad.returncode == 2 and "--cs" in bad.stderr
    if aw._cabi.lib().aw_device_count() > 0:
        return  # with a device the run goes on: test_cli_end_to_end covers it
    for arg in ("--cs", "--cs=short", "--cs=long"):
        r = subprocess.run([_exe(), "-i", str(fa), arg, "--no-progress"], capture_output=True, text=True)
        assert r.returncode == 1 and "usage" not in r.stderr and "device" in r.stderr.lower(), (arg, r.stderr)


# ---- GPU: helpers ---------------------------------------------------------------------------------------------------------
def _batch(ctx, pen, pairs, orientation, flags):
    b = aw.Batch(ctx, aw.make_params(**pen), pairs, orientation=orientation, flags=flags)
    try:
        b.launch()
        res = b.fetch()
        st = b.stats()
    finally:
        b.close()
    return res, st


def _oriented(seqs, r):
    q = seqs[r["query_idx"]]
    return synth_rc(q) if r["is_reverse"] else q


def synth_rc(s):
    import oracle_lib

    return oracle_lib.reverse_complement(s)


def _check_lines(seqs, plain, short, long_, ops=None):
    """every flagged line = the flagless line + the cs column of the tag of that line's CIGAR; r["cs"] is the tag and
    r["cg"] the flagless cg"""
    assert len(plain) == len(short) == len(long_)
    for k, (p, s, l) in enumerate(zip(plain, short, long_)):
        assert p["status"] == s["status"] == l["status"] == 0, (k, p["status"], s["status"], l["status"])
        q, t = _oriented(seqs, p), seqs[p["target_idx"]]
        o = cg_ops(p["cg"])
        if ops is not None:
            assert ops[k] == o
        want_s, want_l = cs_string(o, q, t), cs_string(o, q, t, True)
        assert s["paf"] == p["paf"] + "\tcs:Z:" + want_s, (k, s["paf"][-80:], want_s[-40:])
        assert l["paf"] == p["paf"] + "\tcs:Z:" + want_l, (k, l["paf"][-80:], want_l[-40:])
        assert (s["cs"], l["cs"]) == (want_s, want_l) and s["cg"] == l["cg"] == p["cg"]
        for r in (s, l):
            assert r["cigar_bytes"] == b"" and (r["score"], r["is_reverse"], r["query_end"], r["target_end"]) == \
                (p["score"], p["is_reverse"], p["query_end"], p["target_end"])


def _three(ctx, pen, pairs, orientation=aw.AW_ORIENT_MASH):
    plain, st0 = _batch(ctx, pen, pairs, orientation, aw.AW_FLAG_CIGAR_BYTES)
    short, st1 = _batch(ctx, pen, pairs, orientation, CS)
    long_, st2 = _batch(ctx, pen, pairs, orientation, CS_LONG)
    # paf_bytes counts the delivered lines alike with and without the tag (no newline outside block mode)
    for st, res in ((st0, plain), (st1, short), (st2, long_)):
        assert st["paf_bytes"] == sum(len(r["paf"]) for r in res), st
    return plain, short, long_, (st0, st1, st2)


def _oracle_lines(oracle, ids, seqs, pairs, pen, orientation, fast=False):
    if orientation == aw.AW_ORIENT_FORWARD:
        return None
    return oracle.run_pairs(ids, seqs, pairs, oracle.params(**pen), use_mash=orientation == aw.AW_ORIENT_MASH, threads=CORES, fast=fast)["paf"]


def _route_inputs(route):
    """(ids, seqs, pairs, set_option values) of one kernel route: short pairs alone run on the one-warp kernel, a 2 kb or
    11 kb carrier pair sends the batch to the int16 or int32 chunked 2-bit kernel, N / soft-masked bytes to the
    one-warp byte-compare kernel, and with a 2 kb soft-masked carrier to the 256-thread one, and the cluster options with
    20 kb pairs to the 8-CTA cluster kernel"""
    rnd = random.Random(ROUTES.index(route))
    seqs = []
    if route == "cluster":
        c, ids, seqs, _ = synth.config("C4", n=3, length=20000)
        return ids, seqs, [(0, 1), (1, 2), (2, 0)], dict(cluster_min_len=1000, cluster_always=1, solo_len=2000)
    for f in range(12):
        root = bytes(rnd.choice(b"ACGT") for _ in range(rnd.randint(1, 600)))
        fam = [root] + [_mutate(rnd, root, d)[:1000] or b"A" for d in (0.02, 0.1, 0.25)]
        if f % 2:
            fam[1] = synth_rc(fam[1])
        if route in ("byte", "byte_long"):
            fam[2] = fam[2][: len(fam[2]) // 2] + b"NNN" + fam[2][len(fam[2]) // 2:]
            fam[3] = fam[3].lower()
        seqs += fam
    pairs = [(i, j) for i in range(len(seqs)) for j in range(len(seqs)) if i != j and i // 4 == j // 4]
    pairs += [(rnd.randrange(len(seqs)), rnd.randrange(len(seqs))) for _ in range(40)]
    pairs = [(q, t) for q, t in pairs if q != t]
    carrier = {"int16": 2000, "int32": 11000}.get(route)
    if carrier:
        c = bytes(random.Random(carrier).choice(b"ACGT") for _ in range(carrier))
        pairs.append((len(seqs), len(seqs) + 1))
        seqs += [c, c]
    if route == "byte_long":
        c = bytes(random.Random(2000).choice(b"acgt") for _ in range(2000))
        pairs.append((len(seqs), len(seqs) + 1))
        seqs += [c, c]
    return ["r%03d" % i for i in range(len(seqs))], seqs, pairs, {}


ROUTES = ["one_warp", "int16", "int32", "byte", "cluster", "byte_long"]
ORIENTS = {"mash": aw.AW_ORIENT_MASH, "wfa": aw.AW_ORIENT_WFA, "forward": aw.AW_ORIENT_FORWARD}


def test_route_inputs_pick_their_kernels():
    """CPU: each route's inputs reach the kernel it is named after"""
    from test_byte_input import plan_kernel

    for route in ROUTES:
        ids, seqs, pairs, opts = _route_inputs(route)
        clean = all(re.fullmatch(rb"[ACGT]*", s) for s in seqs)
        mp, mt = max(len(seqs[q]) for q, _ in pairs), max(len(seqs[t]) for _, t in pairs)
        nt, bits, _, ws, cl = plan_kernel(mp, mt, clean, True, opts, npairs=len(pairs))
        want = {"one_warp": (32, 2, "int", 1), "int16": (128, 2, "short", 1), "int32": (128, 2, "int", 1), "byte": (32, 8, "int", 1),
                "cluster": (512, 2, "int", 8), "byte_long": (256, 8, "short", 1)}[route]
        assert (nt, bits, ws, cl) == want, (route, (nt, bits, ws, cl))


# ---- GPU: every route, penalty set and orientation mode -----------------------------------------------------------------
@gpu
@pytest.mark.parametrize("route", ROUTES)
def test_routes_against_oracle(oracle, route):
    ids, seqs, pairs, opts = _route_inputs(route)
    ctx = aw.Context(0)
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        ctx.load_sequences(ids, seqs)
        for pname, pen in PENS.items():
            for oname, orient in ORIENTS.items():
                if route == "cluster" and (pname, oname) not in (("default", "mash"), ("edit", "wfa"), ("bonus", "forward")):
                    continue  # 20 kb pairs: one penalty set per orientation mode
                plain, short, long_, _ = _three(ctx, pen, pairs, orient)
                exp = _oracle_lines(oracle, ids, seqs, pairs, pen, orient, fast=route == "cluster")
                if exp is not None:
                    assert [r["paf"] for r in plain] == exp, (route, pname, oname)
                    if route != "cluster":  # a sample of whole tagged lines from the oracle's own PAF writer
                        p = oracle.params(**pen)
                        for k in random.Random(2).sample(range(len(pairs)), 25):
                            q, t = pairs[k]
                            for res, lf in ((short, False), (long_, True)):
                                want = oracle_cs.align_pair_paf(seqs[q], seqs[t], q, t, p, ids[q], ids[t], long_form=lf,
                                                                use_mash=orient == aw.AW_ORIENT_MASH)
                                assert res[k]["paf"] == want, (route, pname, oname, q, t)
                else:  # forward: the CIGAR of a sample against the oracle's aligner
                    p = oracle.params(**pen)
                    for r in random.Random(1).sample(plain, min(20, len(plain))):
                        st, sc, ops, _ = oracle.wfa_align(p, seqs[r["query_idx"]], seqs[r["target_idx"]])
                        assert (st, sc, ops) == (0, r["score"], r["cigar_bytes"])
                _check_lines(seqs, plain, short, long_, ops=[r["cigar_bytes"] for r in plain])
    finally:
        ctx.close()


# ---- GPU: full size ------------------------------------------------------------------------------------------------------
def _rand_pairs(n, k, seed):
    rnd = random.Random(seed)
    out = []
    while len(out) < k:
        a, b = rnd.randrange(n), rnd.randrange(n)
        if a != b:
            out.append((a, b))
    return out


@gpu
@pytest.mark.parametrize("name,n,seed", [("C2", 1000, 22), ("C5", 5000, 55)])
def test_full_size_256_pairs(oracle, gpu_ctx, name, n, seed):
    c, ids, seqs, _ = synth.config(name, n=n)
    pairs = _rand_pairs(n, 256, seed)
    gpu_ctx.load_sequences(ids, seqs)
    plain, short, long_, _ = _three(gpu_ctx, DEFAULT, pairs)
    assert [r["paf"] for r in plain] == _oracle_lines(oracle, ids, seqs, pairs, DEFAULT, aw.AW_ORIENT_MASH)
    _check_lines(seqs, plain, short, long_)
    if name == "C5":
        assert any(r["is_reverse"] for r in plain) and not all(r["is_reverse"] for r in plain)


@gpu
def test_c4_pair_of_1mb():
    """the first pair of the frozen C4 golden results (two 1 Mb haplotypes): the tag against the golden line's own CIGAR,
    through the converter and by round trip; the line before the column is the golden line"""
    path = os.path.join(ROOT, "tests", "golden", "c4_pairs.json.gz")
    if not os.path.exists(path):
        pytest.skip("tests/golden/c4_pairs.json.gz has not been generated")
    g = json.load(gzip.open(path, "rt"))["pairs"][0]
    c, ids, seqs, _ = synth.config("C4")
    ctx = aw.Context(0)
    try:
        ctx.load_sequences(ids, seqs)
        got = {f: ctx.align_pairs(aw.make_params(**DEFAULT), [(g["q"], g["t"])], flags=f)[0] for f in (CS, CS_LONG)}
    finally:
        ctx.close()
    s, l = got[CS], got[CS_LONG]
    assert s["paf"] == g["paf"] + "\tcs:Z:" + s["cs"] and l["paf"] == g["paf"] + "\tcs:Z:" + l["cs"]
    cg = re.search(r"\tcg:Z:(\S*)", g["paf"]).group(1)
    assert s["cg"] == l["cg"] == cg
    ops = cg_ops(cg)
    q, t = _oriented(seqs, s), seqs[g["t"]]
    assert len(ops) > 10 ** 6
    check_tag(s["cs"], l["cs"], ops, q, t)


# ---- GPU: streaming, retry ladder, failures, flags ---------------------------------------------------------------------
@gpu
def test_stream_blocks_with_cs(oracle):
    """aw_align_stream with AW_FLAG_PAF_BLOCKS | AW_FLAG_CS over several chunks: the blocks, concatenated, are the per-pair
    lines of aw_align_pairs with the flag, in pair order; also on the per-line path the retry ladder takes"""
    c, ids, seqs, rc = synth.config("C5", n=24, length=1500)
    pairs = [(i, j) for i in range(24) for j in range(24) if i != j]
    chunks = [pairs[i:i + 97] for i in range(0, len(pairs), 97)]
    p = aw.make_params(**DEFAULT)
    for width in (None, 48):
        ctx = aw.Context(0)
        try:
            if width:
                ctx.set_option("max_wavefront_width", width)
            ctx.load_sequences(ids, seqs)
            for flags in (CS, CS_LONG):
                per_pair = ctx.align_pairs(p, pairs, flags=flags)
                lines = [r["paf"] for r in per_pair]
                got, seen = [], []
                ctx.align_stream(p, chunks, flags=aw.AW_FLAG_PAF_BLOCKS | flags, block_callback=lambda b, n: got.append(b) and False,
                                 callback=lambda d: seen.append(d["paf"]) and False)
                text = b"".join(got).decode()
                if width:
                    assert sorted(text.splitlines()) == sorted(lines)
                else:
                    assert text == "".join(l + "\n" for l in lines) and len(got) == len(chunks)
                assert seen == lines
            plain = ctx.align_pairs(p, pairs)
            short, long_ = ctx.align_pairs(p, pairs, flags=CS), ctx.align_pairs(p, pairs, flags=CS_LONG)
            _check_lines(seqs, plain, short, long_)
        finally:
            ctx.close()
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**DEFAULT), use_mash=True, threads=CORES)["paf"]
    assert [r["paf"] for r in plain] == exp


@gpu
def test_retried_pairs_carry_tags(oracle):
    """a narrow first-try workspace sends divergent pairs through the retry ladder: their lines carry correct tags too"""
    ids, seqs, _ = synth.generate(808, 8, 900, 0.08, rc_prob=0.5)
    pairs = [(i, j) for i in range(8) for j in range(8) if i != j]
    ctx = aw.Context(0)
    try:
        ctx.set_option("max_wavefront_width", 48)
        ctx.load_sequences(ids, seqs)
        plain, short, long_, stats = _three(ctx, DEFAULT, pairs)
        assert all(st["pairs_retried"] > 0 and st["failed_pairs"] == 0 for st in stats), stats
        assert [r["paf"] for r in plain] == _oracle_lines(oracle, ids, seqs, pairs, DEFAULT, aw.AW_ORIENT_MASH)
        _check_lines(seqs, plain, short, long_)
    finally:
        ctx.close()


@gpu
def test_failure_sentinel_ends_in_empty_tag(gpu_ctx):
    """with the ladder off, a pair that does not fit its workspace becomes the failure sentinel, which ends in "\\tcs:Z:";
    the pair that fits carries its tag"""
    ids, seqs, _ = synth.generate(808, 4, 900, 0.08)
    seqs[3] = seqs[0]
    pairs = [(0, 1), (0, 3), (2, 1)]
    ctx = aw.Context(0)
    try:
        ctx.set_option("max_wavefront_width", 48)
        ctx.set_option("max_retry_attempts", 0)
        ctx.load_sequences(ids, seqs)
        for flags, tag in ((CS, f":{len(seqs[0])}"), (CS_LONG, "=" + seqs[0].decode())):
            for mode in ("pairs", "blocks"):
                if mode == "pairs":
                    res = ctx.align_pairs(aw.make_params(**DEFAULT), pairs, orientation=aw.AW_ORIENT_FORWARD, flags=flags)
                    lines = [r["paf"] for r in res]
                else:
                    got = []
                    ctx.align_stream(aw.make_params(**DEFAULT), [pairs], orientation=aw.AW_ORIENT_FORWARD, flags=aw.AW_FLAG_PAF_BLOCKS | flags,
                                     block_callback=lambda b, n: got.append(b) and False)
                    lines = b"".join(got).decode().splitlines()
                for k, (q, t) in enumerate(pairs):
                    if (q, t) == (0, 3):
                        assert lines[k].endswith(f"\tcg:Z:{len(seqs[0])}=\tcs:Z:{tag}")
                        continue
                    assert lines[k] == f"{ids[q]}\t{len(seqs[q])}\t0\t0\t+\t{ids[t]}\t{len(seqs[t])}\t0\t0\t0\t0\t60\tgi:f:0.000000\tcg:Z:\tcs:Z:"
                    if mode == "pairs":
                        assert res[k]["status"] == aw.AW_EALIGN and res[k]["cs"] == "" and res[k]["cg"] == ""
    finally:
        ctx.close()


@gpu
def test_forbidden_flag_combinations(gpu_ctx):
    """the tag is a PAF column: AW_EINVAL with AW_FLAG_NO_PAF and AW_FLAG_SCORE_ONLY, from every entry point"""
    ids, seqs, _ = synth.generate(5, 3, 300, 0.05)
    gpu_ctx.load_sequences(ids, seqs)
    p = aw.make_params(**DEFAULT)
    for flags in (CS | aw.AW_FLAG_NO_PAF, CS | aw.AW_FLAG_SCORE_ONLY, aw.AW_FLAG_CS_LONG | aw.AW_FLAG_SCORE_ONLY, aw.AW_FLAG_CS_LONG | aw.AW_FLAG_NO_PAF):
        for call in (lambda: aw.Batch(gpu_ctx, p, [(0, 1)], flags=flags), lambda: gpu_ctx.align_pairs(p, [(0, 1)], flags=flags),
                     lambda: gpu_ctx.align_stream(p, [[(0, 1)]], flags=flags, callback=lambda d: False)):
            with pytest.raises(aw.AllwaveError) as ei:
                call()
            assert ei.value.status == aw.AW_EINVAL, flags
    # CS_LONG alone implies CS
    r = gpu_ctx.align_pairs(p, [(0, 1)], flags=aw.AW_FLAG_CS_LONG)[0]
    assert r["cs"] and r["cs"][0] in "=*+-" and r["paf"].endswith("\tcs:Z:" + r["cs"])


# ---- GPU: the CLI end to end -------------------------------------------------------------------------------------------
@gpu
def test_cli_end_to_end(oracle, tmp_path):
    """allwave -i FASTA --cs / --cs=long on sequences of both strands: the oracle's lines + the cs column of each line's
    CIGAR; with two devices, --gpus 2 gives the same lines"""
    c, ids, seqs, rc = synth.config("C5", n=8, length=1200)
    assert any(rc) and not all(rc)
    fa = tmp_path / "small.fa"
    fa.write_text("".join(f">{i}\n{s.decode()}\n" for i, s in zip(ids, seqs)))
    pairs = [(i, j) for i in range(8) for j in range(8) if i != j]
    exp = oracle.run_pairs(ids, seqs, pairs, oracle.params(**DEFAULT), use_mash=True, threads=CORES)["paf"]
    by_names = {(ids[q], ids[t]): (q, t) for q, t in pairs}
    runs = [[]] + ([["--gpus", "2"]] if aw._cabi.lib().aw_device_count() >= 2 else [])
    for arg, long_form in (("--cs", False), ("--cs=long", True)):
        for extra in runs:
            out = tmp_path / "o.paf"
            subprocess.check_call([_exe(), "-i", str(fa), "-o", str(out), "-p", "none", "--no-progress", arg] + extra)
            lines = out.read_text().splitlines()
            assert len(lines) == len(exp)
            want = {}
            for line in exp:
                f = line.split("\t")
                q, t = by_names[(f[0], f[5])]
                qs = synth_rc(seqs[q]) if f[4] == "-" else seqs[q]
                cg = re.search(r"\tcg:Z:(\S*)", line).group(1)
                want[(f[0], f[5])] = line + "\tcs:Z:" + cs_string(cg_ops(cg), qs, seqs[t], long_form)
            assert sorted(lines) == sorted(want.values()), (arg, extra)
            if not extra:
                assert [l.split("\t")[:6:5] for l in lines] == [l.split("\t")[:6:5] for l in exp]
