"""Timing of bootstrap split scores along site windows (batch.window_bootstrap_scores) and of the count-row rank-1
divergence behind its mutual-information path (engine.rank1_divergence_count_rows: spb_mi_row_slots + spb_mi_row_scores),
on seeded inputs of bench_inputs (balanced tree, JC).

  (a) "count_rows": the divergences of ~200 random covering splits for B = 100 bootstrap count rows of one 10^5-site
      table at 12 / 20 / 40 / 64 taxa: the count-row kernel (side tables built once, all rows in a few launches) against
      rank1_divergence_scores on each replicate's compacted table (the route bootstrap_scores took before), CUDA events
      around the scoring only (count rows and compacted tables are built beforehand), and whether the scores are equal.
  (b) "windows": window_bootstrap_scores over 19 windows of 10^5 sites (step 5 10^4) of a 10^6-site alignment, each
      method, against a loop of bootstrap_scores on the slices with each window's seed (timed on `--host-windows` windows
      and scaled to 19); 20 taxa with B = 100 and 64 taxa with B = 20, 16 random covering splits.
  (c) "bootstrap_scores": bootstrap_scores (B = 100) against the per-replicate loop it replaced (bootstrap_tables, then
      pair_tables_from_table + subflatten_scores, or rank1_divergence_scores, on each table after the same counting),
      run alternately, for subflattening and mutual information: the c2 input (12 taxa, branch length 0.05, 10^6 sites,
      all 2,035 splits) and 20 taxa x 10^6 sites with 200 random covering splits.

Wall times are host clocks bracketed by device synchronises, after a warm-up call.

    python scripts/window_bootstrap_scores_timing.py [--out profiles/r10_window_bootstrap_scores_timing.json]
                                                     [--host-windows 3] [--repeats 3]

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
from splitp_b200.enums import Method  # noqa: E402

eng = sp.engine
SEED = 2024
SITES, WIDTH, STEP = 1_000_000, 100_000, 50_000


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


def events(fn, reps=3):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, out


def covering_splits(n, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        perm = rng.permutation(n)
        k = int(rng.integers(1, n))
        out.append((sorted(perm[:k].tolist()), sorted(perm[k:].tolist())))
    return out


def counted(codes):
    if codes.shape[0] <= eng.NARROW_MAX_TAXA:
        return eng.count_patterns(eng.pack(codes))
    return eng.count_patterns_wide(*eng.pack_wide(codes))


def count_rows_case(n, B=100, S=200, sites=100_000):
    table = counted(BI.simulate_codes(n, 0.05, "JC", sites, n))
    splits = covering_splits(n, S, n)
    src = eng.bootstrap_sources([table], [SEED])[0]
    keys, counts, _, N, _ = src
    P = int(counts.shape[0])
    rows = eng._bootstrap_rows(src, 0, B, own=False)
    tabs = list(eng.bootstrap_tables(table, B, SEED))
    new_ms, new = events(lambda: eng.rank1_divergence_count_rows(keys, lambda r0, r1: rows[r0:r1], B, n, float(N), splits,
                                                                 row_cap=min(P, N)))
    old_ms, old = events(lambda: torch.stack([eng.rank1_divergence_scores(tb, splits) for tb in tabs]))
    return {"taxa": n, "sites": sites, "patterns": P, "replicates": B, "splits": S, "count_rows_ms": new_ms,
            "per_replicate_ms": old_ms, "speedup": old_ms / new_ms,
            "equal": bool(torch.equal(new.view(torch.int64), old.view(torch.int64)))}


def windows_case(n, B, host_windows, S=16):
    codes = BI.simulate_codes(n, 0.05, "JC", SITES, n)
    wins = batch.sliding_windows(SITES, WIDTH, STEP)
    W = int(wins.shape[0])
    splits = covering_splits(n, S, 3 * n)
    out = {"taxa": n, "sites": SITES, "windows": W, "window_sites": WIDTH, "window_step": STEP, "replicates": B, "splits": S}
    for m in (Method.subflattening, Method.mutual_information, Method.flattening):
        batch.window_bootstrap_scores(codes, splits, wins[:2], m, replicates=2, seed=SEED)  # warm-up
        ms, got = wall(lambda: batch.window_bootstrap_scores(codes, splits, wins, m, replicates=B, seed=SEED))
        loop, equal = [], True
        for w, (b, e) in enumerate(wins[:host_windows].tolist()):
            sl = np.ascontiguousarray(codes[:, b:e])
            t, want = wall(lambda: batch.bootstrap_scores(sl, splits, m, B, seed=eng.window_bootstrap_seed(SEED, b, e)))
            loop.append(t)
            equal &= bool(np.array_equal(got[w].view(np.int64), want.view(np.int64)))
        out[m.name] = {"window_bootstrap_scores_ms": ms, "bootstrap_scores_loop_ms": float(np.median(loop)) * W,
                       "loop_windows_timed": len(loop), "equal": equal}
    return out


def parent_route(codes, splits, method, B, seed):
    """bootstrap_scores as the parent commit computed it: the same counting, then one scorer call per replicate table."""
    ss = batch.SplitScorer(splits, None, method)
    table = ss._count(codes)
    out = eng._empty((B, len(splits)), torch.float64)
    for b, tb in enumerate(eng.bootstrap_tables(table, B, seed)):
        if method == Method.subflattening:
            out[b] = eng.subflatten_scores(eng.pair_tables_from_table(tb, as_counts=True), *ss.masks)
        else:
            out[b] = eng.rank1_divergence_scores(tb, ss.idx_all)
    return out.cpu().numpy()


def bootstrap_scores_case(name, codes, splits, B, repeats):
    out = {"input": name, "taxa": int(codes.shape[0]), "sites": int(codes.shape[1]), "splits": len(splits), "replicates": B}
    for m in (Method.subflattening, Method.mutual_information):
        batch.bootstrap_scores(codes[:, :10_000], splits, m, 2, SEED)  # warm-up
        parent_route(codes[:, :10_000], splits, m, 2, SEED)
        new, old, equal = [], [], True
        for _ in range(repeats):  # alternately
            t, a = wall(lambda: batch.bootstrap_scores(codes, splits, m, B, SEED))
            new.append(t)
            t, b = wall(lambda: parent_route(codes, splits, m, B, SEED))
            old.append(t)
            equal &= bool(np.array_equal(a.view(np.int64), b.view(np.int64)))
        out[m.name] = {"this_commit_ms": float(np.median(new)), "parent_route_ms": float(np.median(old)),
                       "this_commit_all_ms": new, "parent_route_all_ms": old, "equal": equal}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_window_bootstrap_scores_timing.json"))
    ap.add_argument("--host-windows", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    res = {"gpu": gpu_info()}
    res["count_rows"] = [count_rows_case(n) for n in (12, 20, 40, 64)]
    print(json.dumps(res["count_rows"]), flush=True)
    res["windows"] = [windows_case(20, 100, args.host_windows), windows_case(64, 20, args.host_windows)]
    print(json.dumps(res["windows"]), flush=True)
    c2 = BI.simulate_codes(12, 0.05, "JC", SITES, 2)  # bench.py c2: seed 2
    res["bootstrap_scores"] = [
        bootstrap_scores_case("c2", c2, BI.all_splits_idx(12), 100, args.repeats),
        bootstrap_scores_case("t20", BI.simulate_codes(20, 0.05, "JC", SITES, 20), covering_splits(20, 200, 20), 100, args.repeats),
    ]
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
