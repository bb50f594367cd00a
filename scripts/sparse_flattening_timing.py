"""Timing of the sparse flattening route (csrc/sparse.cu, engine.sparse_flattening_scores):

  * 20 taxa x 10^6 simulated sites: a batch each of 10|10, 5|15 and 2|18 splits;
  * 64 taxa x 10^6 simulated sites: 32|32 and 8|56 splits;
  * a whole erickson_SVD(Method.flattening) at 20 taxa x 10^5 sites.

Per batch: the plan (ranking of the projections + the CSR / CSC sorts), the solver (small Gram + scorer, or the block-Krylov
cycles), both as CUDA-event spans of one call, the whole call (host clock around a call that ends in a device synchronise),
and one F (F^T Q) product (spb_sparse_product, CUDA events, mean over repeated launches).  The product's bytes are counted
from the shapes: the index / value arrays and offsets of both groupings, one 64-byte gather per non-zero in each stage and
the 64-byte outputs.  It is a gather: every non-zero reads a random 64-byte row, so it is bound by the latency of these
gathers (L2 for rows that stay cached), and bytes over time is reported against the 7.7 TB/s HBM peak only as a ratio.

    python scripts/sparse_flattening_timing.py [--sites 1000000] [--erickson-sites 100000] [--out FILE]

Prints one JSON object with the GPU's name and power limit beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import splitp_b200 as sp  # noqa: E402

eng = sp.engine
HBM_PEAK = 7.7e12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def codes_of(n, N, seed):
    tree = sp.trees.balanced_tree(n, 0.1)
    return sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=seed)


def side_splits(n, a, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        perm = rng.permutation(n)
        out.append((sorted(perm[:a].tolist()), sorted(perm[a:].tolist())))
    return out


def product_time(plans, reps=20):
    k = -(-max(p.k for p in plans) // eng.SPARSE_K_ALIGN) * eng.SPARSE_K_ALIGN
    a = eng.sparse_batch_arrays(plans, k)
    B = len(plans)
    ws = eng._empty(int(eng.lib.spb_sparse_product_ws(k, B, a["ncols"], a["nnz"])), torch.float64)
    Q = torch.randn((B, 8, k), dtype=torch.float64, device=eng.device())
    AQ = torch.empty_like(Q)
    args = (eng._p(a["row_off"]), eng._p(a["row_col"]), eng._p(a["row_val"]), eng._p(a["col_off"]), eng._p(a["col_row"]),
            eng._p(a["col_val"]), a["ncols"], a["nnz"], k, B, eng._p(Q), eng._p(AQ), eng._p(ws), eng._st())
    eng.call("spb_sparse_product", *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.call("spb_sparse_product", *args)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nnz, rows, cols = a["nnz"], B * k, a["ncols"]
    # transpose (read Q, write Qt), per stage: offsets, index + value per non-zero, a 64-byte gather per non-zero, 64-byte outputs
    moved = 2 * 64 * rows + 8 * (rows + cols) + 2 * nnz * (4 + 8 + 64) + 64 * (rows + cols)
    return {"k_padded": k, "nnz": nnz, "ncols": cols, "product_ms": ms, "bytes_model": moved,
            "bytes_per_s": moved / (ms * 1e-3), "share_of_hbm_peak": moved / (ms * 1e-3) / HBM_PEAK}


def time_batch(table, splits):
    eng.sparse_flattening_scores(table, splits[:1])  # module load / first launches
    torch.cuda.synchronize()
    timer = eng.PhaseTimer()
    t0 = time.perf_counter()
    scores = eng.sparse_flattening_scores(table, splits, timer=timer)
    torch.cuda.synchronize()
    whole = (time.perf_counter() - t0) * 1e3
    phases = {name: {"ms": ms, "spans": n} for name, (ms, n, _) in timer.totals().items()}
    plans = [eng.sparse_plan(table, *s) for s in splits]
    out = {"splits": len(splits), "k": [p.k for p in plans], "C": [p.C for p in plans], "whole_ms": whole, "phases": phases,
           "scores": scores.cpu().numpy().tolist()}
    out.update(product_time(plans))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--erickson-sites", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "sites": args.sites}
    codes = codes_of(20, args.sites, seed=1)
    t0 = time.perf_counter()
    table = eng.count_patterns(eng.pack(codes))
    torch.cuda.synchronize()
    res["t20"] = {"patterns": table.num, "count_ms": (time.perf_counter() - t0) * 1e3}
    for a, count in ((10, 4), (5, 8), (2, 16)):
        res["t20"][f"{a}|{20 - a}"] = time_batch(table, side_splits(20, a, count, seed=a))
    codes = codes_of(64, args.sites, seed=2)
    wide, valid, n, N = eng.pack_wide(codes)
    keys, counts = eng.count_patterns_wide(wide, valid, n, N).compact()
    wtab = eng.WidePatternTable(n, keys, counts.to(torch.float64))
    res["t64"] = {"patterns": wtab.num}
    for a, count in ((32, 2), (8, 4)):
        res["t64"][f"{a}|{64 - a}"] = time_batch(wtab, side_splits(64, a, count, seed=a))
    codes = codes_of(20, args.erickson_sites, seed=3).cpu().numpy()
    U, cnt = np.unique(codes.T, axis=0, return_counts=True)
    mapping = {"".join("ACGT"[c] for c in row): int(k) for row, k in zip(U, cnt)}
    sp.erickson_SVD({p: v for p, v in list(mapping.items())[:50]} | {"A" * 20: 1}, method=sp.Method.flattening)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    chosen = sp.erickson_SVD(mapping, method=sp.Method.flattening)
    torch.cuda.synchronize()
    res["erickson20"] = {"sites": args.erickson_sites, "patterns": len(mapping), "seconds": time.perf_counter() - t0,
                         "steps": len(chosen)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
