"""Timing of split scores and erickson_SVD trees along site windows (batch.window_scores / window_trees) against the host
loop they replace (slice the alignment, then one score_splits / erickson_SVD call per window), on seeded inputs of
bench_inputs (balanced tree, JC, branch length 0.05):

  subflattening  20 taxa x 10^7 sites, windows of 10^5 sites with step 5 10^4 (199 windows), the tree's 17 informative
                 splits plus 10^3 random ones; 64 taxa x 10^6 sites, the same windows (19), tree splits + 10^3 random ones
  trees          window_trees at the same two sizes
  flattening, mutual information   12 taxa x 10^6 sites, the same windows (19), the tree's splits + 10^3 random ones

Per case: the window call (host clock bracketed by device synchronises, after one untimed warm-up call on a short
prefix), the host loop over `--host-windows` of its windows (scaled to all windows; for trees it includes building each
window's {pattern: probability} mapping), and whether the outputs of those
windows agree (bitwise for subflattening, mutual information and trees; within max(1e-9, 64 eps / score^2) for
flattening).  It also times the segment kernel alone (spb_pair_tables_segments over the windows' cuts, CUDA events around the
launches only) next to one pair_kernel pass over the whole alignment (spb_pair_tables).

    python scripts/window_scores_timing.py [--out profiles/r8_window_scores_timing.json] [--host-windows 4]

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
import splitp_b200.batch as batch  # noqa: E402
from splitp_b200.alignment import Alignment  # noqa: E402
from splitp_b200.phylogenetics import erickson_SVD  # noqa: E402

eng = sp.engine
M = sp.Method


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


def events(fn, reps=5):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def mapping_of(codes):
    """{pattern: count / sites} of a code matrix without unusable sites: erickson_SVD's input."""
    cols, counts = np.unique(codes.T, axis=0, return_counts=True)
    lut = np.array(list("ACGT"))
    return {"".join(lut[c]): int(k) / codes.shape[1] for c, k in zip(cols, counts)}


def tree_splits(n):
    from tests.test_gpu_bootstrap_trees import true_splits
    taxa, truth = true_splits(n)
    index = {t: i for i, t in enumerate(taxa)}
    return [([index[t] for t in a], [index[t] for t in b]) for a, b in truth]


def agree(got, ref, tol):
    if not tol:
        return bool(np.array_equal(got.view(np.uint64), ref.view(np.uint64)))
    ok = ~np.isnan(ref)
    bound = np.maximum(1e-9, 64 * np.finfo(float).eps / np.maximum(ref[ok], 1e-300) ** 2)
    return bool(np.array_equal(np.isnan(got), np.isnan(ref))
                and (np.abs(got[ok] - ref[ok]) <= bound * np.maximum(np.abs(ref[ok]), 1e-300)).all())


def score_case(n, N, method, host_windows, width=100_000, step=50_000, seed=2024):
    codes = BI.simulate_codes(n, 0.05, "JC", N, seed)
    splits = tree_splits(n) + BI.random_splits_idx(n, 1000, seed)
    wins = batch.sliding_windows(N, width, step)
    batch.window_scores(codes[:, :3 * width], splits, batch.sliding_windows(3 * width, width, step), method)  # warm-up
    ms, got = wall(lambda: batch.window_scores(codes, splits, wins, method))
    picks = np.linspace(0, len(wins) - 1, host_windows).astype(int)
    host_ms, same = [], True
    for w in picks:
        b, e = wins[w]
        t, ref = wall(lambda: batch.score_splits(np.ascontiguousarray(codes[:, b:e]), splits, method))
        host_ms.append(t)
        same &= agree(got[w], ref, method == M.flattening)
    per = float(np.median(host_ms))
    return {"taxa": n, "sites": N, "windows": len(wins), "width": width, "step": step, "splits": len(splits),
            "method": str(method), "window_scores_ms": ms, "host_loop_ms_per_window": per, "host_loop_ms_all_windows": per * len(wins),
            "speedup": per * len(wins) / ms, "host_windows_checked": len(picks), "outputs_agree": bool(same)}


def tree_case(n, N, host_windows, width=100_000, step=50_000, seed=2024):
    codes = BI.simulate_codes(n, 0.05, "JC", N, seed)
    wins = batch.sliding_windows(N, width, step)
    taxa = batch._default_taxa(n)
    batch.window_trees(codes[:, :3 * width], batch.sliding_windows(3 * width, width, step))  # warm-up
    ms, trees = wall(lambda: batch.window_trees(codes, wins))
    picks = np.linspace(0, len(wins) - 1, host_windows).astype(int)
    host_ms, same = [], True
    for w in picks:
        b, e = wins[w]
        t, host = wall(lambda: erickson_SVD(Alignment(mapping_of(codes[:, b:e]), taxa), taxa=taxa, method=M.subflattening))
        host_ms.append(t)
        same &= {frozenset(s) for s in trees[w]} == {frozenset(s) for s in host}
    per = float(np.median(host_ms))
    return {"taxa": n, "sites": N, "windows": len(wins), "width": width, "step": step, "window_trees_ms": ms,
            "host_loop_ms_per_window": per, "host_loop_ms_all_windows": per * len(wins), "speedup": per * len(wins) / ms,
            "host_windows_checked": len(picks), "same_splits": bool(same)}


def segment_pass(n, N, width=100_000, step=50_000, seed=2024):
    """Kernel launches only: the rows, the bounds and the raw row are allocated and uploaded once, then the two entry points
    are timed back to back (their counts accumulate; the time does not depend on the values)."""
    codes = BI.simulate_codes(n, 0.05, "JC", N, seed)
    aln = eng.pack(codes, want_sm=False)
    ends = np.unique(batch.sliding_windows(N, width, step).reshape(-1))
    S, words = len(ends) - 1, int(eng.lib.spb_pair_raw_words(n))
    d_ends = torch.from_numpy(ends).to(eng.device())
    rows, raw = eng._zeros((S, words), torch.int64), eng._zeros(words, torch.int64)
    seg = events(lambda: eng.call("spb_pair_tables_segments", eng._p(aln.planes), eng._p(aln.valid), n, aln.plane_words,
                                  eng._p(d_ends), S, eng._p(rows), eng._st()), reps=20)
    whole = events(lambda: eng.call("spb_pair_tables", eng._p(aln.planes), eng._p(aln.valid), n, aln.plane_words, 0,
                                    aln.plane_words, eng._p(raw), eng._st()), reps=20)
    return {"taxa": n, "sites": N, "segments": S, "segment_kernel_ms": seg, "pair_kernel_whole_ms": whole,
            "note": "CUDA events over 20 launches each (after one warm-up), kernel launches only"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-windows", type=int, default=4)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "scores": [], "trees": [], "segment_pass": []}
    for n, N in ((20, 10_000_000), (64, 1_000_000)):
        res["scores"].append(score_case(n, N, M.subflattening, args.host_windows))
        res["trees"].append(tree_case(n, N, args.host_windows))
        res["segment_pass"].append(segment_pass(n, N))
    for method in (M.flattening, M.mutual_information):
        res["scores"].append(score_case(12, 1_000_000, method, args.host_windows))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
