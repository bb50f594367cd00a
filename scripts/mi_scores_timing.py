"""Timing of the batched rank-1 divergence (csrc/mi_batch.cu, engine.rank1_divergence_scores) against the per-split route
(engine.rank1_divergence: spb_table_marginals + spb_mi_table, one split at a time), on seeded inputs of bench_inputs:

  (a) 12 taxa x 10^6 sites (bench workload c2's input), all 2,035 splits: batched call and per-split loop;
  (b) 20 taxa x 10^6 sites, 10^4 random covering splits (bench_inputs.random_splits_idx, default_rng seed 5): both;
  (c) 64 taxa x 10^6 sites, the 61 splits of the true tree plus 195 random ones: batched call only (the per-split route
      reads uint64 keys and stops at 31 taxa).

Every shape is run once before it is timed; a timed call is bracketed by device synchronises and the best of `--reps`
calls is kept.  Reported: ms per call, split scores per second, and (split, pattern) inserts + lookups per second (two
inserts in pass 1 and two lookups in pass 2 per pair), plus the largest |batched - per-split| relative to the score.

    python scripts/mi_scores_timing.py [--sites 1000000] [--reps 3] [--out profiles/r5_mi_scores_timing.json]

Prints one JSON object with the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench_inputs as BI  # noqa: E402
import splitp_b200 as sp  # noqa: E402

eng = sp.engine


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def timed(fn, reps):
    fn()  # warm-up of this shape
    torch.cuda.synchronize()
    best, out = float("inf"), None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3, out


def per_split(table, splits):
    return torch.cat([eng.rank1_divergence(table, a, b).reshape(1) for a, b in splits])


def true_splits(n):
    """Non-trivial splits of bench_inputs' balanced n-taxon tree, as row positions (rows are in sorted-name order)."""
    parent, names = BI.balanced_parents(n)
    row = {name: i for i, name in enumerate(BI.taxa_of(names))}
    below = {node: {row[name]} for node, name in names.items()}
    for node in range(len(parent) - 1, 0, -1):
        below.setdefault(parent[node], set()).update(below.get(node, set()))
    out, seen = [], set()
    for node in range(1, len(parent)):
        side = frozenset(below[node])
        canon = min(side, frozenset(range(n)) - side, key=lambda s: sorted(s))
        if 1 < len(side) < n - 1 and canon not in seen:
            seen.add(canon)
            out.append((sorted(side), sorted(set(range(n)) - side)))
    return out


def case(table, splits, reps, loop):
    P = int(table.compact()[0].shape[0]) if isinstance(table, eng.WideTable) else table.num
    ms, got = timed(lambda: eng.rank1_divergence_scores(table, splits), reps)
    pairs = P * len(splits)
    res = {"splits": len(splits), "patterns": P, "batched_ms": ms, "batched_split_scores_per_s": len(splits) / (ms * 1e-3),
           "batched_inserts_lookups_per_s": 4 * pairs / (ms * 1e-3)}
    if loop:
        lms, ref = timed(lambda: per_split(table, splits), 1)
        g, r = got.cpu().numpy(), ref.cpu().numpy()
        res.update({"per_split_ms": lms, "per_split_split_scores_per_s": len(splits) / (lms * 1e-3), "speedup": lms / ms,
                    "max_rel_diff": float(np.max(np.abs(g - r) / np.maximum(np.abs(r), 1e-300)))})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mi_scores_timing.py needs a CUDA device")
    res = {"gpu": gpu_info(), "sites": args.sites, "reps": args.reps}
    codes = BI.simulate_codes(12, 0.05, "JC", args.sites, 2)
    table = eng.count_patterns(eng.pack(codes))
    res["a_12taxa_all_splits"] = case(table, BI.all_splits_idx(12), args.reps, True)
    codes = BI.simulate_codes(20, 0.05, "JC", args.sites, 3)
    table = eng.count_patterns(eng.pack(codes))
    res["b_20taxa_10k_random"] = case(table, BI.random_splits_idx(20, 10_000, seed=5), args.reps, True)
    codes = BI.simulate_codes(64, 0.05, "JC", args.sites, 4)
    wide, valid, n, N = eng.pack_wide(codes)
    table = eng.count_patterns_wide(wide, valid, n, N)
    splits = true_splits(64) + BI.random_splits_idx(64, 195, seed=5)
    res["c_64taxa_true_plus_random"] = case(table, splits, args.reps, False)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
