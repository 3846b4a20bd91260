"""Score-only vs full alignment on the device-resident batch bench.py times (same config, seed and batch size, mash
orientation, aw_batch_*).  Both batches live in one process; after warm-up the two modes alternate launch by launch.
One JSON line per config: pairs/s and kernel ms of each mode (medians), cells and steps per pair, whether every pair's
status, score and strand agree, and the GPU's name and power limit read in the same run.

usage: python tools/score_only_probe.py [--configs C2,C5,C3] [--rounds 5] [--warmup 2] [--out profiles/r03_runs]"""
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
    modes = {"full": aw.Batch(ctx, params, pairs, orientation=aw.AW_ORIENT_MASH, flags=0),
             "score": aw.Batch(ctx, params, pairs, orientation=aw.AW_ORIENT_MASH, flags=aw.AW_FLAG_SCORE_ONLY)}
    for b in modes.values():
        for _ in range(warmup):
            b.launch()
        torch.cuda.synchronize()
        b.fetch(collect=False)
    ms = {m: [] for m in modes}
    kms = {m: [] for m in modes}
    # one step = every kernel of one launch (orientation + alignment) on the context's stream; the host clock stops after a
    # device-wide synchronise
    for _ in range(rounds):
        for m, b in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b.launch()
            torch.cuda.synchronize()
            ms[m].append((time.perf_counter() - t0) * 1e3)
            kms[m].append(b.kernel_ms())
    out = dict(config=name, pairs=len(pairs), rounds=rounds)
    results = {}
    for m, b in modes.items():
        got = []
        b.fetch(collect=False, callback=lambda r: got.append((r.status, r.score, r.is_reverse)) and 0)
        st = b.stats()
        results[m] = got
        med = statistics.median(ms[m])
        out[m] = dict(pairs_per_s=round(len(pairs) / (med / 1e3), 1), step_ms_median=round(med, 3), step_ms=[round(x, 3) for x in ms[m]],
                      kernel_ms_median=round(statistics.median(kms[m]), 3), cells_per_pair=st["cells"] / len(pairs),
                      steps_per_pair=st["steps"] / len(pairs), failed_pairs=st["failed_pairs"], pairs_retried=st["pairs_retried"])
        b.close()
    out["scores_equal"] = results["full"] == results["score"]
    out["speedup_pairs_per_s"] = round(out["score"]["pairs_per_s"] / out["full"]["pairs_per_s"], 3)
    out["cells_ratio"] = round(out["score"]["cells_per_pair"] / out["full"]["cells_per_pair"], 4)
    out["steps_ratio"] = round(out["score"]["steps_per_pair"] / out["full"]["steps_per_pair"], 4)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C5,C3")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="", help="directory for score_only_<config>.json (one JSON line each)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("score_only_probe.py needs a B200: the product path has no CPU fallback")
    for name in args.configs.split(","):
        line = dict(probe(name, args.rounds, args.warmup), **gpu_info())
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"score_only_{name}.json"), "w") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
