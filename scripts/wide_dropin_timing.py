"""Timing of the 32..64-taxon mapping routes at 64 taxa (10^5 and 10^6 simulated sites by default):

  * host encode_patterns of the {pattern: probability} dict, and table_from_mapping (encode + upload) on a cache miss;
  * the pair-table kernel spb_pair_tables_wide (CUDA events, mean over repeated launches after a warm-up);
  * subflattening + split_score of one 32|32 split (host clock around calls that end in a device synchronise);
  * a whole erickson_SVD(Method.subflattening) (host clock).

    python scripts/wide_dropin_timing.py [--sites 100000 1000000] [--out FILE]

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


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def wall(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return out


def mapping_of(n, N, seed):
    """{pattern: count / N} of a simulated alignment (generate_alignment's values), built with the vectorised decode."""
    tree = sp.trees.balanced_tree(n, 0.1)
    codes = sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=seed)
    wide, valid, n, N = eng.pack_wide(codes)
    keys, counts = eng.count_patterns_wide(wide, valid, n, N).compact()
    pats = eng.decode_keys(keys.cpu().numpy().view(np.uint64), n)
    vals = (counts.cpu().numpy().astype(np.float64) / float(N)).tolist()
    return tree, dict(zip(pats, vals))


def run(n, N, reps):
    tree, mapping = mapping_of(n, N, seed=5)
    res = {"taxa": n, "sites": N, "patterns": len(mapping)}
    pats = list(mapping.keys())
    res["host_encode_patterns_ms"] = wall(lambda: eng.encode_patterns(pats), 3)
    res["table_from_mapping_cache_miss_ms"] = wall(lambda: eng.table_from_mapping(dict(mapping)), 3)
    table = eng.table_from_mapping(mapping)
    N_tab = torch.empty((n, n, 4, 4), dtype=torch.float64, device="cuda")
    ws = torch.empty(max(int(eng.lib.spb_pair_tables_wide_ws(table.num, n)), 1), dtype=torch.float64, device="cuda")

    def pair_kernel():
        eng.call("spb_pair_tables_wide", eng._p(table.keys), eng._p(table.values), table.num, n, eng._p(N_tab), eng._p(ws), eng._st())

    for _ in range(3):
        pair_kernel()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        pair_kernel()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    work = 2.0 * table.num * (4 * n) ** 2  # dense E^T diag(v) E flops (both triangles; the kernel does the upper block triangle)
    res["pair_tables_wide_kernel_ms"] = ms
    res["pair_tables_wide_dense_equiv_tflops"] = work / (ms * 1e-3) / 1e12
    aln = sp.Alignment(mapping, tree.taxa)
    split = (tree.taxa[:32], tree.taxa[32:])
    sp.split_score(sp.subflattening(split, aln))  # warm-up (table cached from here on)
    res["subflattening_plus_split_score_ms"] = wall(lambda: sp.split_score(sp.subflattening(split, aln)), 5)
    t = time.perf_counter()
    picks = sp.erickson_SVD(aln, taxa=list(tree.taxa), method=sp.Method.subflattening)
    torch.cuda.synchronize()
    res["erickson_svd_subflattening_ms"] = (time.perf_counter() - t) * 1e3
    true = {frozenset(map(frozenset, s)) for s in tree.splits()}
    res["erickson_true_splits_recovered"] = f"{len(true & {frozenset(map(frozenset, s)) for s in picks})}/{len(true)}"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=64)
    ap.add_argument("--sites", type=int, nargs="+", default=[100_000, 1_000_000])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_dropin_timing.py needs a CUDA device")
    out = {"gpu": gpu_info(), "runs": [run(args.taxa, N, args.reps) for N in args.sites]}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
