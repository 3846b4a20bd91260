#!/usr/bin/env python
"""bench.py -- aligned pairs/s of the allwave alignment hot path on B200 (BASELINE.json metric).

Default workload (config.workload): BASELINE config 2 -- 1,000 x 10 kb synthetic sequences at 5 % per-haplotype
divergence, `-p none` (999,000 directed pairs), scores 0,5,8,2,24,1, mash orientation.  `--config C1..C5` selects the
other BASELINE configs (SURVEY 8d generator, same seeds).  A "step" is one pass of the whole hot path (orientation ->
biWFA -> CIGAR -> PAF text) over one batch of `--batch` pairs per GPU drawn from that config's pair list.

  --scaling weak (default, the driver's contract): every rank aligns its own shard of world*batch pairs, no collective.
  --scaling strong: ONE process drives the product path (allwave --gpus N = AllPairIterator over N contexts with a shared
            chunk queue, liballwave_host.so) over a FIXED pair list on --gpus N devices: total pairs / wall time.

  value     device-resident: sequences + pair list already in HBM, kernels launched on the timed stream, PAF text left in HBM.
  e2e       through the host-facing C-ABI calls the CLI makes (aw_load_sequences + aw_align_stream with PAF blocks) with HOST
            buffers: H2D of sequences and pairs and D2H of every PAF line inside the timed region.
  roofline  the alignment kernel alone (CUDA events around it on the launch stream) against the measured HBM copy
            bandwidth, with SURVEY 8(d)'s algorithmic bytes per pair.
  cpu_baseline / --impl reference
            the CPU restatement of the allwave/WFA2 path (oracle/, "port": the Rust reference cannot be built in this
            image), all host threads, on a bounded sample of the same pairs (in the N=1 line only).
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# per config: description, scores, -p strategy, default pairs per GPU per step, CPU sample (pairs per core), dtype of the wavefront rows
CONFIGS = {
    "C1": dict(desc="C1: 16 x 10 kb, 1% divergence per haplotype, -p none (240 directed pairs), -s 0,5,8,2,24,1, mash orientation",
               scores=(0, 5, 8, 2, 24, 1), spars="none", batch=240, cpu_pairs_per_core=15, dtype="int16"),
    "C2": dict(desc="C2: 1000 x 10 kb, 5% divergence per haplotype, -p none (999,000 directed pairs), -s 0,5,8,2,24,1, mash orientation",
               scores=(0, 5, 8, 2, 24, 1), spars="none", batch=14208, cpu_pairs_per_core=8, dtype="int16"),  # 24 pairs per resident CTA: short tail
    "C3": dict(desc="C3: 1415 x 150 bp reads, 2% divergence, -p none (2,000,810 directed pairs), -s 0,1,1,1, mash orientation",
               scores=(0, 1, 1, 1, None, None), spars="none", batch=2000810, cpu_pairs_per_core=20000, dtype="int32"),
    "C4": dict(desc="C4: 200 x 1 Mb haplotypes, 0.1-2% divergence + SVs, -p giant:0.99 (~1,970 pairs), -s 0,5,8,2,24,1, mash orientation",
               scores=(0, 5, 8, 2, 24, 1), spars="giant:0.99", batch=16, cpu_pairs_per_core=0, dtype="int32"),  # 16 pairs: one per cluster, ~40 s per step
    "C5": dict(desc="C5: 5000 x 5 kb, 3% divergence, 50% reverse-complemented, -p tree:2:1:0.1 (~2.51 M pairs), -s 0,5,8,2,24,1, mash orientation",
               scores=(0, 5, 8, 2, 24, 1), spars="tree:2:1:0.1", batch=37888, cpu_pairs_per_core=64, dtype="int16"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="weak: pairs per GPU per step (0 = the config's default)")
    ap.add_argument("--pairs", type=int, default=0, help="strong: pairs of the fixed job (0 = default)")
    ap.add_argument("--nseq", type=int, default=0, help="number of sequences (0 = the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = steps")
    ap.add_argument("--out-paf", default="", help="strong: also write the PAF here")
    ap.add_argument("--no-checksum", action="store_true", help="strong: skip the extra (untimed) pass that computes the order-independent PAF digest")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="weak: after the timed steps, write the results of the last one as DIR/<name>.npy (see OutputDump)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.scaling != "weak"):
        ap.error("--dump-outputs needs --impl b200 --scaling weak")
    return args


def config_sequences(name, nseq):
    from allwave_b200 import synth

    c, ids, seqs, _ = synth.config(name, n=nseq or None)
    return ids, seqs


def config_pair_list(name, ids, seqs, ctx=None):
    """the config's full directed pair list, exactly what the CLI would align (src/iterator.rs:37-77)"""
    from allwave_b200 import hostlib as H

    spars = CONFIGS[name]["spars"]
    n = len(ids)
    if spars == "none":
        return None  # implicit: every (i, j), i != j -- sampled arithmetically
    sp = H.parse_sparsification(spars)
    return H.pair_list(ids, sp["kind"], value=sp["value"], k_nearest=sp["k_nearest"], k_farthest=sp["k_farthest"], random_fraction=sp["random_fraction"],
                       kmer_size=sp["kmer_size"], ctx=ctx)


def job_pairs(nseq, total, full=None):
    """deterministic sample of the pair list: every stride-th pair"""
    npairs_all = nseq * (nseq - 1) if full is None else len(full)
    total = min(total, npairs_all)
    stride = max(1, npairs_all // max(1, total))
    out = []
    for t in range(total):
        idx = (t * stride) % npairs_all
        if full is not None:
            out.append(tuple(full[idx]))
            continue
        i, r = divmod(idx, nseq - 1)
        j = r if r < i else r + 1
        out.append((i, j))
    return out


def algorithmic_bytes(seqs, pairs, paf_bytes):
    # SURVEY 8(d): ceil(n/4) + ceil(m/4) + 16 (pair descriptor) + len(PAF line) per pair
    b = paf_bytes
    for q, t in pairs:
        b += (len(seqs[q]) + 3) // 4 + (len(seqs[t]) + 3) // 4 + 16
    return b


def kernel_source_hash():
    """identifies the kernel sources a profile belongs to (profiles/ncu_summary.json carries the same stamp)"""
    h = hashlib.sha1()
    for f in ("aw_wfa.cuh", "aw_common.cuh", "aw_sketch.cuh"):
        h.update(open(os.path.join(ROOT, "allwave_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


class OutputDump:
    """What a caller of the timed path receives for each pair (aw_result, through aw_batch_fetch), collected from the fetch of
    the last timed step and written as float64 / float32 .npy files, at most LIMIT bytes in all, so that two builds can be
    compared output for output on the same inputs:

      pair_index                 position of each dumped pair in the pair list of the step
      <field>                    one aw_result field per file (FIELDS), one row per dumped pair
      paf_sample_index           positions of the pairs whose PAF line is dumped
      paf_sample_offsets         start of each of those lines in paf_sample_bytes (one more entry than lines)
      paf_sample_bytes           the lines' bytes (float32 codes 0..255)

    Every pair is dumped when there are at most MAX_ROWS, else a sample drawn with a fixed seed; the PAF text is dumped for a
    fixed-seed sample of MAX_PAF_LINES of those pairs, as many as fit in the remaining bytes."""

    FIELDS = ("query_idx", "target_idx", "query_start", "query_end", "target_start", "target_end", "is_reverse", "status", "score",
              "num_matches", "alignment_length", "paf_len")
    LIMIT = 64 << 20
    MAX_ROWS = 1 << 18
    MAX_PAF_LINES = 1024

    def __init__(self, npairs):
        import numpy as np

        rng = np.random.default_rng(0)
        rows = np.arange(npairs) if npairs <= self.MAX_ROWS else np.sort(rng.choice(npairs, self.MAX_ROWS, replace=False))
        paf_rows = np.sort(rng.choice(rows, min(len(rows), self.MAX_PAF_LINES), replace=False))
        self.rows, self.paf_rows = rows, paf_rows
        self.take = np.zeros(npairs, dtype=bool)
        self.take[rows] = True
        self.take_paf = np.zeros(npairs, dtype=bool)
        self.take_paf[paf_rows] = True
        self.n, self.vals, self.paf = 0, [], []

    def add(self, r):
        """aw_result callback of Batch.fetch, called once per pair in pair order; returns 0 (do not cancel)"""
        import ctypes as C

        i = self.n
        self.n += 1
        if self.take[i]:
            self.vals.append(tuple(getattr(r, f) for f in self.FIELDS))
            if self.take_paf[i]:
                self.paf.append(C.string_at(r.paf, r.paf_len) if r.paf_len else b"")
        return 0

    def write(self, out_dir):
        import numpy as np

        if self.n != len(self.take):
            raise SystemExit(f"--dump-outputs: the fetch delivered {self.n} results for {len(self.take)} pairs")
        vals = np.asarray(self.vals, dtype=np.float64).reshape(len(self.rows), len(self.FIELDS))
        arrays = {"pair_index": self.rows.astype(np.float64)}
        arrays.update((f, vals[:, j].copy()) for j, f in enumerate(self.FIELDS))
        # bytes left for the PAF text (float32 codes) after the other arrays, the sample's index and offsets and the .npy headers
        room = (self.LIMIT - sum(a.nbytes for a in arrays.values()) - 16 * (len(self.paf_rows) + 1) - (1 << 16)) // 4
        lines, used = [], 0
        for line in self.paf:
            if used + len(line) > room:
                break
            lines.append(line)
            used += len(line)
        arrays["paf_sample_index"] = self.paf_rows[: len(lines)].astype(np.float64)
        arrays["paf_sample_offsets"] = np.concatenate([[0], np.cumsum([len(x) for x in lines])]).astype(np.float64)
        arrays["paf_sample_bytes"] = np.frombuffer(b"".join(lines), dtype=np.uint8).astype(np.float32)
        assert sum(a.nbytes for a in arrays.values()) <= self.LIMIT
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_sample_pairs(cfg, pairs, cores):
    per_core = CONFIGS[cfg]["cpu_pairs_per_core"]
    return pairs[: max(2, per_core * cores)] if per_core else []


def run_reference(args, rank, world):
    """--impl reference: the CPU restatement (oracle/) on all host threads; rank 0 only."""
    if rank != 0:
        return
    import oracle_lib as O

    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    ids, seqs = config_sequences(args.config, args.nseq)
    if cfg["spars"] == "none":
        full = None
    else:  # the pair list of the sparsified configs comes from the oracle here (no GPU on this path)
        kinds = {"giant": O.SPARS_GIANT, "tree": O.SPARS_TREE}
        parts = cfg["spars"].split(":")
        if parts[0] == "giant":
            full = O.pair_list(ids, seqs, kind=kinds["giant"], fraction=float(parts[1]))
        else:
            full = O.pair_list(ids, seqs, kind=kinds["tree"], fraction=float(parts[3]), k_nearest=int(parts[1]), k_farthest=int(parts[2]))
    per_core = cfg["cpu_pairs_per_core"] or 1
    per_step = max(2, per_core * cores) if args.config != "C4" else 2
    pairs = job_pairs(len(seqs), per_step, full)
    p = O.params(*cfg["scores"])
    for _ in range(min(args.warmup, 1)):
        O.run_pairs(ids, seqs, pairs[: max(1, min(len(pairs), cores // 2))], p, use_mash=True, threads=cores, fast=True)
    t0 = time.perf_counter()
    block = 0
    for _ in range(args.steps):
        r = O.run_pairs(ids, seqs, pairs, p, use_mash=True, threads=cores, fast=True)
        block += r["sum_block_len"]
    dt = time.perf_counter() - t0
    value = len(pairs) * args.steps / dt
    line = {
        "impl": "reference", "metric": "aligned pairs/s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": cfg["desc"], "pairs_per_step": len(pairs),
                   "note": "CPU restatement of the allwave/WFA2 path (oracle/, PARITY UNPINNED vs WFA2-lib); the Rust reference cannot be built here"},
        "gbp_per_s": block / dt / 1e9,
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": f"{len(pairs)} pairs of the {args.config} pair list per step x {args.steps} steps (fast mode of the port)"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_strong(args):
    """one process, N GPUs, the product path: AllPairIterator::for_each_paf_block over N contexts (shared chunk queue)"""
    import allwave_b200 as aw
    from allwave_b200 import hostlib as H

    cfg = CONFIGS[args.config]
    if aw._cabi.lib().aw_device_count() < args.gpus:
        raise SystemExit(f"--scaling strong --gpus {args.gpus}: only {aw._cabi.lib().aw_device_count()} devices visible")
    ids, seqs = config_sequences(args.config, args.nseq)
    scores = ",".join(str(s) for s in cfg["scores"] if s is not None)
    default_pairs = {"C1": 240, "C2": 151552, "C3": 2000810, "C4": 0, "C5": 600000}[args.config]  # 0 = the whole pair list
    max_pairs = args.pairs or default_pairs
    sampler = ClockSampler(0)
    runs = []
    if args.warmup:  # one warm-up pass on a small prefix: allocations, sketches, instruction caches
        H.run_job(ids, seqs, scores=scores, sparsification=cfg["spars"], n_gpus=args.gpus, max_pairs=max(1, max_pairs // 16) if max_pairs else 8 * args.gpus)
    for _ in range(args.steps):
        runs.append(H.run_job(ids, seqs, scores=scores, sparsification=cfg["spars"], n_gpus=args.gpus, max_pairs=max_pairs, out_path=args.out_paf))
    clocks = sampler.stop()
    chk = {"digest": 0} if args.no_checksum else H.run_job(ids, seqs, scores=scores, sparsification=cfg["spars"], n_gpus=args.gpus, max_pairs=max_pairs, checksum=True)
    secs = [r["seconds"] for r in runs]
    pairs = runs[0]["pairs"]
    value = pairs * len(runs) / sum(secs)
    line = {
        "metric": "aligned pairs/s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(secs) / len(runs), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
        "config": {"workload": cfg["desc"], "pairs_total": pairs, "path": "one process: AllPairIterator::for_each_paf_block over N contexts, shared cost-ordered chunk queue, "
                   "two batches in flight per GPU, PAF blocks to the host (allwave --gpus N)", "l2": "per-launch working set exceeds the 126 MB L2; no explicit flush"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 8 * pairs, "d2h_bytes_per_step": runs[0]["paf_bytes"] + 112 * pairs, "steps": len(runs)},
        "paf_bytes": runs[0]["paf_bytes"], "paf_digest": None if args.no_checksum else "%016x" % chk["digest"], "gpu_imbalance_max_over_mean": max(r["imbalance"] for r in runs),
        "setup_seconds": runs[0]["setup_seconds"], "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
        "gpu_launches": None,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.scaling == "strong":
        if world > 1:
            raise SystemExit("--scaling strong is a single-process run: use `python bench.py --scaling strong --gpus N` without torchrun")
        run_strong(args)
        return

    import torch
    import torch.distributed as dist

    import allwave_b200 as aw
    from allwave_b200 import partition

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_gpus = world
    cfg = CONFIGS[args.config]
    scores = cfg["scores"]
    ids, seqs = config_sequences(args.config, args.nseq)
    params = aw.make_params(*scores)

    ctx = aw.Context(local_rank)
    ctx.load_sequences(ids, seqs)
    full = config_pair_list(args.config, ids, seqs, ctx)
    n_all = len(seqs) * (len(seqs) - 1) if full is None else len(full)
    B = args.batch or cfg["batch"] or (4 * 148)
    B = min(B, max(1, n_all // world))
    # whole job = world*B pairs; host-side greedy (LPT) partition by predicted cost (length x estimated divergence), no collective
    job = job_pairs(len(seqs), B * world, full)
    div = ctx.estimate_divergence(job) if world > 1 else None
    shards = partition.partition_pairs(job, [len(s) for s in seqs], world, divergence=div)
    pairs = shards[rank]
    batch = aw.Batch(ctx, params, pairs, orientation=aw.AW_ORIENT_MASH, flags=0)
    stream = torch.cuda.current_stream()
    sh = stream.cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also builds the sketches once: they stay resident like the sequences) ----
    for _ in range(args.warmup):
        batch.launch(sh)
    torch.cuda.synchronize()
    if args.warmup:  # a batch that was never launched has nothing to fetch
        batch.fetch(collect=False)
    launches_per_step = 2  # orientation kernel + alignment kernel (memsets are not kernels of ours)

    # ---- timed: device-resident ----
    sampler = ClockSampler(local_rank)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    ev0.record(stream)
    for _ in range(args.steps):
        batch.launch(sh)
        kernel_ms.append(batch.kernel_ms())
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    dump = OutputDump(len(pairs)) if args.dump_outputs else None
    batch.fetch(collect=False, callback=dump.add if dump else None)
    st = batch.stats()
    if st["failed_pairs"]:
        raise SystemExit(f"{st['failed_pairs']} pairs failed on the GPU path")
    retried = st["pairs_retried"]
    if dump:
        dump.write(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"))

    # ---- timed: end to end through the host-facing C-ABI call, host buffers ----
    e2e_steps = args.e2e_steps or args.steps
    acc = {"paf_bytes": 0, "n": 0}
    import ctypes as C

    # the call the CLI makes: aw_align_stream with AW_FLAG_PAF_BLOCKS -- every batch comes back as one block of
    # newline-terminated PAF lines in pair order (host memory); the chunks are what aw_align_pairs would cut as well
    def _blk(text, nbytes, nlines, _u):
        acc["paf_bytes"] += nbytes - nlines
        acc["n"] += nlines
        return 0

    blk = aw._cabi.PAF_BLOCK_CB(_blk)
    arr = aw._cabi.make_pairs(pairs)
    chunk = 65536
    if max(len(x) for x in seqs) <= 1024:  # reads: the product path's rule (allwave_b200/host/allwave.hpp, drive()): 65,536 .. 262,144 pairs per chunk
        n_chunks = max(1, -(-len(pairs) // 262144), min(12, len(pairs) // 65536))
        chunk = -(-len(pairs) // n_chunks)
    cursor = {"pos": 0}

    def _next(_u, out):
        b = cursor["pos"]
        if b >= len(pairs):
            return 0
        cnt = min(chunk, len(pairs) - b)
        out[0] = C.cast(C.byref(arr, b * C.sizeof(aw._cabi.AwPair)), C.POINTER(aw._cabi.AwPair))
        cursor["pos"] = b + cnt
        return cnt

    src = aw._cabi.CHUNK_SOURCE(_next)
    L = aw._cabi.lib()
    ctx2 = aw.Context(local_rank)
    n = len(seqs)
    sa = (C.c_char_p * n)(*seqs)
    la = (C.c_uint64 * n)(*[len(s) for s in seqs])
    ia = (C.c_char_p * n)(*[i.encode() for i in ids])

    def e2e_step():
        t_a = time.perf_counter()
        aw._cabi.check(L.aw_load_sequences(ctx2._h, n, sa, la, ia), "aw_load_sequences")
        t_b = time.perf_counter()
        cursor["pos"] = 0
        aw._cabi.check(L.aw_align_stream(ctx2._h, C.byref(params), aw.AW_ORIENT_MASH, aw.AW_FLAG_PAF_BLOCKS, src, None, C.cast(None, aw._cabi.RESULT_CB), blk, None),
                       "aw_align_stream")
        if os.environ.get("AW_BENCH_TRACE"):
            print(f"[e2e] load {1e3 * (t_b - t_a):.1f} ms, align_stream {1e3 * (time.perf_counter() - t_b):.1f} ms", file=sys.stderr)

    e2e_step()  # warm-up (allocations)
    acc.update(paf_bytes=0, n=0)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    paf_bytes_step = acc["paf_bytes"] // max(1, e2e_steps)
    h2d = sum(len(s) for s in seqs) + 8 * len(pairs) + sum(len(i) for i in ids)
    d2h = paf_bytes_step + 112 * len(pairs)
    ctx2.close()

    # ---- reduce over ranks: max time, summed work ----
    t = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    w = torch.tensor([len(pairs), st["sum_block_len"], st["cells"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    ms_max, e2e_ms_max = float(t[0]), float(t[1])
    pairs_total, block_total, cells_total = float(w[0]), float(w[1]), float(w[2])

    if rank == 0:
        value = pairs_total * args.steps / (ms_max / 1e3)
        e2e_value = pairs_total * e2e_steps / (e2e_ms_max / 1e3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        k_ms = sum(kernel_ms) / len(kernel_ms)
        algo = algorithmic_bytes(seqs, pairs, st["paf_bytes"])
        achieved = algo / (k_ms / 1e3) / 1e9
        # dram bytes of the dominant kernel from the committed ncu capture -- only if it was taken with these kernel sources
        # and this workload; scaled per pair to the batch of this run
        traffic, traffic_note = None, "no ncu capture of this kernel build / workload in profiles/ncu_summary.json"
        try:
            summ = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))
            ak = summ.get("align_kernel", {})
            if summ.get("kernel_source_hash") == kernel_source_hash() and summ.get("config", "C2") == args.config and ak.get("pairs_per_launch"):
                traffic = ak["dram_bytes_per_launch"] / ak["pairs_per_launch"] * len(pairs)
                traffic_note = (f"ncu --set full capture {summ.get('tag')} ({ak['pairs_per_launch']} pairs per launch), scaled per pair; in that capture: "
                                f"dram throughput {ak.get('dram_throughput_pct', 0):.1f} % of peak, issue slots active {ak.get('issue_active_pct', 0):.1f} %, "
                                f"{ak.get('inst_executed', 0) / ak['pairs_per_launch'] / 1e6:.0f} M warp instructions per pair")
        except Exception:
            pass
        line = {
            "metric": "aligned pairs/s", "value": value, "unit": "pairs/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
            "config": {"workload": cfg["desc"], "pairs_per_gpu_per_step": len(pairs), "nseq": len(seqs),
                       "partition": f"host LPT over {world} GPUs by length x estimated divergence, no collective",
                       "l2": "per-launch working set (wavefront rings + history) exceeds the 126 MB L2; no explicit flush",
                       "parity_note": "oracle = CPU restatement of WFA2-lib biWFA; PARITY UNPINNED against the real WFA2-lib (not on disk)"},
            "gbp_per_s": block_total * args.steps / (ms_max / 1e3) / 1e9,
            "cells_per_s": cells_total * args.steps / (ms_max / 1e3),
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps},
            "gpu_launches": launches_per_step * args.steps, "pairs_retried_per_step": retried,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                         "kernel": "aw_align_kernel", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": algo,
                         "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                         "note": "compulsory HBM traffic of this path is tiny (SURVEY 8d): the kernel is bound by memory latency + integer issue, see profiles/"},
        }
        sample = cpu_sample_pairs(args.config, pairs, os.cpu_count() or 1)
        if not args.no_cpu_baseline and sample and world == 1:  # the CPU leg belongs to the N=1 line only (idle ranks would share its cores)
            import oracle_lib as O

            cores = os.cpu_count() or 1
            # the baseline leg runs the restatement in its fast mode (free lists, unchecked interior loop, 8-byte extend: what a
            # WFA2-lib build does); the parity check below uses the plain checker path, whose speed is reported as well
            rf = O.run_pairs(ids, seqs, sample, O.params(*scores), use_mash=True, threads=cores, fast=True)
            r = O.run_pairs(ids, seqs, sample, O.params(*scores), use_mash=True, threads=cores)
            line["cpu_baseline"] = {"value": len(sample) / rf["seconds"], "unit": "pairs/s", "cores": cores, "kind": "port",
                                    "sample": f"first {len(sample)} pairs of rank 0's shard, {cores} threads, {rf['seconds']:.1f} s (fast mode of the port)",
                                    "checker_value": len(sample) / r["seconds"], "fast_equals_checker": rf["paf"] == r["paf"]}
            # parity of the same pairs, GPU vs CPU restatement, outside every timed region
            gres = ctx.align_pairs(params, sample, orientation=aw.AW_ORIENT_MASH)
            same = sum(1 for g, c in zip(gres, r["paf"]) if g["paf"] == c)
            line["parity"] = {"pairs_checked": len(sample), "paf_identical": same, "scores_identical": sum(1 for g, s in zip(gres, r["scores"]) if g["score"] == s)}
            if same != len(sample):
                line["parity"]["FAILED"] = True
        print(json.dumps(line), flush=True)
    batch.close()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
