"""What the cs:Z: tag costs: no tag, AW_FLAG_CS and AW_FLAG_CS_LONG on the device-resident batch bench.py times (same config,
seed and batch size, mash orientation, aw_batch_*).  The three batches live in one process; after warm-up the modes alternate
launch by launch.  One JSON line per config: pairs/s and step ms of each mode (medians), the delivered PAF bytes per pair,
whether every pair's line with the tag starts with its line without it, and the GPU's name and power limit read in the same
run.

usage: python tools/cs_probe.py [--configs C2,C3,C5] [--rounds 5] [--warmup 2] [--out DIR]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the config tables and pair sampling of the benchmark itself)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def probe(name, rounds, warmup):
    import torch

    import allwave_b200 as aw

    cfg = bench.CONFIGS[name]
    ids, seqs = bench.config_sequences(name, 0)
    ctx = aw.Context(0)
    ctx.load_sequences(ids, seqs)
    full_list = bench.config_pair_list(name, ids, seqs, ctx)
    n_all = len(seqs) * (len(seqs) - 1) if full_list is None else len(full_list)
    pairs = bench.job_pairs(len(seqs), min(cfg["batch"], n_all), full_list)
    params = aw.make_params(*cfg["scores"])
    flags = {"none": 0, "short": aw.AW_FLAG_CS, "long": aw.AW_FLAG_CS | aw.AW_FLAG_CS_LONG}
    modes = {m: aw.Batch(ctx, params, pairs, orientation=aw.AW_ORIENT_MASH, flags=f) for m, f in flags.items()}
    for b in modes.values():
        for _ in range(warmup):
            b.launch()
        torch.cuda.synchronize()
        b.fetch(collect=False)
    ms = {m: [] for m in modes}
    # one step = every kernel of one launch (orientation, alignment, and the tag and re-layout kernels of the tag modes) on
    # the context's stream; the host clock stops after a device-wide synchronise
    for _ in range(rounds):
        for m, b in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b.launch()
            torch.cuda.synchronize()
            ms[m].append((time.perf_counter() - t0) * 1e3)
    out = dict(config=name, pairs=len(pairs), rounds=rounds)
    lines = {}
    for m, b in modes.items():
        got = []
        b.fetch(collect=False, callback=lambda r: got.append((r.status, bytes(r.paf[: r.paf_len]))) and 0)
        st = b.stats()
        lines[m] = got
        med = statistics.median(ms[m])
        out[m] = dict(pairs_per_s=round(len(pairs) / (med / 1e3), 1), step_ms_median=round(med, 3), step_ms=[round(x, 3) for x in ms[m]],
                      paf_bytes_per_pair=round(st["paf_bytes"] / len(pairs), 1), failed_pairs=st["failed_pairs"], pairs_retried=st["pairs_retried"])
        b.close()
    out["lines_extend_untagged"] = all(
        (s0, s1, s2) == (0, 0, 0) and l1.startswith(l0 + b"\tcs:Z:") and l2.startswith(l0 + b"\tcs:Z:")
        for (s0, l0), (s1, l1), (s2, l2) in zip(lines["none"], lines["short"], lines["long"]))
    for m in ("short", "long"):
        out[m]["rate_vs_none"] = round(out[m]["pairs_per_s"] / out["none"]["pairs_per_s"], 4)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C3,C5")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="", help="directory for cs_<config>.json (one JSON line each)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("cs_probe.py needs a B200: the product path has no CPU fallback")
    for name in args.configs.split(","):
        line = dict(probe(name, args.rounds, args.warmup), **gpu_info())
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"cs_{name}.json"), "w") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
