"""Timing of bootstrap trees (batch.bootstrap_trees: every replicate's erickson_SVD(Method.subflattening) agglomerated in
lockstep on the device, csrc/agglomerate.cu) on seeded inputs of bench_inputs, B = 100 replicates each:

  20 taxa x 10^6 sites, 32 taxa x 10^6 sites, 64 taxa x 10^5 sites (balanced tree, JC, branch length 0.05).

Per case:
  - the whole bootstrap_trees call (host clock bracketed by device synchronises, after one untimed call with B = 2);
  - its phases, from a separate run of engine.bootstrap_tree_masks with a PhaseTimer (CUDA events): "resample" (replicate
    counts + compaction + per-replicate table copies), "tables" (pair tables of the counts + triple tables), "score" (the
    multi-table scoring launches) and "step" (the agglomeration step kernel), with the library's launch count;
  - the host loop it replaces, for `--host-reps` replicates: expanding replicate b into a {pattern: probability} mapping
    and erickson_SVD(Alignment(mapping, taxa), method=Method.subflattening) on it, per replicate, plus whether that tree's
    informative splits equal the lockstep tree's.

    python scripts/bootstrap_trees_timing.py [--out profiles/r7_bootstrap_trees_timing.json] [--host-reps 2]

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
import splitp_b200.batch  # noqa: E402,F401
from splitp_b200.alignment import Alignment  # noqa: E402
from splitp_b200.phylogenetics import erickson_SVD  # noqa: E402

eng = sp.engine
SEED = 2024
B = 100


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def counted(codes):
    n = codes.shape[0]
    if n <= eng.NARROW_MAX_TAXA:
        return eng.count_patterns(eng.pack(codes))
    return eng.count_patterns_wide(*eng.pack_wide(codes))


def mapping_of(tb, n):
    keys = tb.keys.cpu().numpy().view(np.uint64)
    counts = tb.counts.cpu().numpy().view(np.uint32).astype(np.int64)
    sh = 2 * (n - 1 - np.arange(n))
    if keys.ndim == 1:
        codes = ((keys[:, None] >> sh.astype(np.uint64)) & np.uint64(3)).astype(np.uint8)
    else:
        lo = (keys[:, 0:1] >> np.minimum(sh, 62).astype(np.uint64)) & np.uint64(3)
        hi = (keys[:, 1:2] >> np.maximum(sh - 64, 0).astype(np.uint64)) & np.uint64(3)
        codes = np.where(sh >= 64, hi, lo).astype(np.uint8)
    strings = np.frombuffer(b"ACGT", dtype=np.uint8)[codes].view(f"S{n}").ravel()
    N = counts.sum()
    return {s.decode(): int(c) / N for s, c in zip(strings, counts)}


def informative(tree):
    return {frozenset(s) for s in tree if min(len(s[0]), len(s[1])) >= 2}


def case(n, sites, host_reps):
    codes = BI.simulate_codes(n, 0.05, "JC", sites, n)
    taxa = sp.batch._default_taxa(n)
    res = {"taxa": n, "sites": sites, "replicates": B}
    sp.batch.bootstrap_trees(codes, replicates=2, seed=SEED)
    ms, out = wall(lambda: sp.batch.bootstrap_trees(codes, replicates=B, seed=SEED))
    res["bootstrap_trees_ms"] = ms
    res["bootstrap_trees_ms_per_tree"] = ms / (B + 1)
    res["mean_support"] = float(out.support.mean())
    count_ms, table = wall(lambda: counted(codes))
    res["count_ms"] = count_ms
    first = min(range(n), key=lambda i: taxa[i])
    timer = eng.PhaseTimer()
    launches = int(eng.lib.spb_launch_count())
    ms, (masks, _) = wall(lambda: eng.bootstrap_tree_masks(table, B, SEED, first, timer))
    res["launches"] = int(eng.lib.spb_launch_count()) - launches
    res["timed_tree_masks_ms"] = ms
    res["phases_ms"] = {k: v[0] for k, v in timer.totals().items()}
    res["phase_spans"] = {k: v[1] for k, v in timer.totals().items()}
    host = []
    for b, tb in enumerate(eng.bootstrap_tables(table, host_reps, SEED)):
        t0 = time.perf_counter()
        mapping = mapping_of(tb, n)
        t1 = time.perf_counter()
        tree = erickson_SVD(Alignment(mapping, taxa), taxa=taxa, method=sp.Method.subflattening)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        host.append({"replicate": b, "patterns": len(mapping), "mapping_ms": (t1 - t0) * 1e3, "erickson_svd_ms": (t2 - t1) * 1e3,
                     "informative_splits_equal": informative(tree) == informative(out.replicate_trees[b])})
    res["host_loop"] = host
    res["host_erickson_svd_ms_per_replicate"] = float(np.mean([h["erickson_svd_ms"] for h in host]))
    res["host_mapping_ms_per_replicate"] = float(np.mean([h["mapping_ms"] for h in host]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bootstrap_trees_timing.py needs a CUDA device")
    res = {"gpu": gpu_info(), "seed": SEED}
    for n, sites in ((20, 1_000_000), (32, 1_000_000), (64, 100_000)):
        res[f"t{n}_s{sites}"] = case(n, sites, args.host_reps)
        print(json.dumps(res[f"t{n}_s{sites}"]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
