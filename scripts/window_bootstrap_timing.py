"""Timing of bootstrap trees along site windows (batch.window_bootstrap_trees: every window's tree and its replicates'
trees agglomerated in lockstep, the pair tables of each window's count rows from spb_pair_tables_count_rows) on seeded
inputs of bench_inputs (balanced tree, JC, branch length 0.05), windows of 10^5 sites with step 5 10^4 (19 windows):

  20 taxa x 10^6 sites, B = 100 replicates;   64 taxa x 10^6 sites, B = 20 replicates.

Per case:
  - the whole window_bootstrap_trees call (host clock bracketed by device synchronises, after an untimed warm-up call);
  - its phases from a separate run of the same stages with a PhaseTimer (CUDA events): "count" (pack + counting every
    window), then engine.bootstrap_tree_masks_multi's "resample", "pair tables" (spb_pair_tables_count_rows), "triple
    tables" (transform + triple tables), "score" and "step", the library's launch count, and the host time of turning the
    masks into erickson_SVD's split format and of the support (numpy on the masks);
  - the counted work of the pair tables, (non-zero counts of every window's B + 1 rows) x n (n + 1) / 2 cell increments, and
    its rate over the "pair tables" phase (the count-row kernel up to engine.COUNT_ROWS_MAX_TAXA taxa, the compacted
    single-table route above);
  - for the first window, the count-row kernel (its increments/s) against the single-table route on the same B + 1 rows
    (spb_pair_tables_weighted up to 31 taxa, spb_pair_tables_wide above, on each replicate's compacted table as
    SubflattenTables.add builds it), CUDA events around the pair-table launches only, and whether the tables are equal;
  - the host loop the call replaces: bootstrap_trees on the slice of each of `--host-windows` windows with the window's
    seed (median, times the number of windows), and whether those entries are equal.

Before the cases, the pair tables of one table's 101 count rows (10^5 simulated sites) at 12 to 64 taxa through the
count-row kernel and through the single-table routes (the numbers behind engine.COUNT_ROWS_MAX_TAXA).

    python scripts/window_bootstrap_timing.py [--out profiles/r9_window_bootstrap_timing.json] [--host-windows 3]
                                              [--routes-only]

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
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def count_windows(codes, wins):
    """The window tables window_bootstrap_trees counts."""
    n = codes.shape[0]
    if n <= eng.NARROW_MAX_TAXA:
        aln = eng.pack(codes)
        return [eng.count_patterns(aln, b, e) for b, e in wins.tolist()]
    wide, valid, _, N = eng.pack_wide(codes)
    return [eng.count_patterns_wide(wide, valid, n, N, b, e) for b, e in wins.tolist()]


def single_table_route(table, B, seed, n):
    """The replicate tables of the single-table route and a function that builds their pair tables N."""
    keys, counts = eng._counted(table)
    _, N = eng._bootstrap_prefix(counts)
    tabs = [eng._table_of_counts(table, keys, counts, N)] + list(eng.bootstrap_tables(table, B, seed))
    out = eng._empty((B + 1, n, n, 4, 4), torch.float64)

    def run():
        for r, tb in enumerate(tabs):
            vals = tb.counts.to(torch.float64)  # pair_tables_from_table's values: counts below 2^31 here
            if n <= eng.NARROW_MAX_TAXA:
                out[r].zero_()
                eng.call("spb_pair_tables_weighted", eng._p(tb.keys), eng._p(vals), tb.num, n, eng._p(out[r]), eng._st())
            else:
                ws = eng._empty(max(int(eng.lib.spb_pair_tables_wide_ws(tb.num, n)), 1), torch.float64)
                eng.call("spb_pair_tables_wide", eng._p(tb.keys), eng._p(vals), tb.num, n, eng._p(out[r]), eng._p(ws), eng._st())
        return out
    return run


def case(n, B, host_windows):
    codes = BI.simulate_codes(n, 0.05, "JC", SITES, n)
    wins = batch.sliding_windows(SITES, WIDTH, STEP)
    W = int(wins.shape[0])
    taxa = batch._default_taxa(n)
    res = {"taxa": n, "sites": SITES, "windows": W, "window_sites": WIDTH, "window_step": STEP, "replicates": B}
    batch.window_bootstrap_trees(codes, wins[:2], replicates=2, seed=SEED)  # warm-up
    ms, out = wall(lambda: batch.window_bootstrap_trees(codes, wins, replicates=B, seed=SEED))
    res["window_bootstrap_trees_ms"] = ms
    res["ms_per_window"] = ms / W
    res["mean_support"] = float(np.mean([o.support.mean() for o in out]))

    # phases of the same stages
    timer = eng.PhaseTimer()
    launches = int(eng.lib.spb_launch_count())
    with timer.span("count"):
        tables = count_windows(codes, wins)
    seeds = [eng.window_bootstrap_seed(SEED, b, e) for b, e in wins.tolist()]
    first = min(range(n), key=lambda i: taxa[i])
    ms, (masks, _) = wall(lambda: eng.bootstrap_tree_masks_multi(tables, B, seeds, first, timer))
    res["launches"] = int(eng.lib.spb_launch_count()) - launches
    res["timed_tree_masks_ms"] = ms
    res["phases_ms"] = {k: v[0] for k, v in timer.totals().items()}
    res["phase_spans"] = {k: v[1] for k, v in timer.totals().items()}
    t0 = time.perf_counter()
    trees = batch._trees_of_masks(masks, taxa)
    t1 = time.perf_counter()
    support = [batch._support(masks[w], None, n) for w in range(W)]
    t2 = time.perf_counter()
    res["host_split_names_ms"] = (t1 - t0) * 1e3
    res["host_support_ms"] = (t2 - t1) * 1e3
    res["split_masks_converted"] = int(masks.size)
    assert trees[0] == out[0].tree and np.array_equal(support[0], out[0].support)

    # counted work of the pair tables (count-row kernel: one increment per non-zero count and taxon pair i <= j)
    srcs = eng.bootstrap_sources(tables, seeds)
    nnz = []
    for src in srcs:
        rows = eng._bootstrap_rows(src, 0, B + 1)
        nnz.append(int(torch.count_nonzero(rows).item()))
        del rows
    pairs = n * (n + 1) // 2
    res["pair_tables_route"] = "count rows" if n <= eng.COUNT_ROWS_MAX_TAXA else "compacted rows, spb_pair_tables_wide"
    res["count_rows_nonzero"] = sum(nnz)
    res["count_rows_patterns"] = int(sum(int(s[1].shape[0]) for s in srcs)) * (B + 1)
    res["pair_table_increments"] = sum(nnz) * pairs
    res["pair_table_increments_per_s"] = sum(nnz) * pairs / (res["phases_ms"]["pair tables"] * 1e-3)

    # the count-row kernel against the single-table route on window 0's rows
    rows = eng._bootstrap_rows(srcs[0], 0, B + 1)
    new = lambda: eng.pair_tables_count_rows(srcs[0][0], rows, n)  # noqa: E731
    old = single_table_route(tables[0], B, seeds[0], n)
    k_ms = events(new)
    res["window0"] = {"patterns": int(srcs[0][1].shape[0]), "rows": B + 1, "nonzero": nnz[0],
                      "count_rows_kernel_ms": k_ms, "count_rows_increments_per_s": nnz[0] * pairs / (k_ms * 1e-3),
                      "single_table_route_ms": events(old),
                      "tables_equal": bool(torch.equal(new().view(torch.int64), old().view(torch.int64)))}
    del rows, srcs, tables

    # the host loop it replaces
    host = []
    for w in np.linspace(0, W - 1, host_windows).astype(int).tolist():
        b, e = wins[w].tolist()
        sl = np.ascontiguousarray(codes[:, b:e])
        ms_w, r = wall(lambda: batch.bootstrap_trees(sl, B, seed=eng.window_bootstrap_seed(SEED, b, e)))
        host.append({"window": w, "bootstrap_trees_ms": ms_w, "equal": r.tree == out[w].tree and r.replicate_trees ==
                     out[w].replicate_trees and bool(np.array_equal(r.support, out[w].support))})
    res["host_loop"] = host
    res["host_loop_ms_estimate"] = float(np.median([h["bootstrap_trees_ms"] for h in host])) * W
    return res


def route_by_taxa(n, B=100, sites=100_000):
    """The pair tables of one table's B + 1 count rows (10^5 simulated sites) through the count-row kernel, the
    single-table route on the pre-compacted replicate tables, and (32..64 taxa) the compaction + spb_pair_tables_wide route
    bootstrap_group_tables takes above engine.COUNT_ROWS_MAX_TAXA: CUDA events, 3 calls each after a warm-up."""
    codes = BI.simulate_codes(n + n % 2, 0.05, "JC", sites, n)[:n]
    table = count_windows(codes, np.array([[0, sites]]))[0]
    src = eng.bootstrap_sources([table], [SEED])[0]
    rows = eng._bootstrap_rows(src, 0, B + 1)
    new = lambda: eng.pair_tables_count_rows(src[0], rows, n)  # noqa: E731
    old = single_table_route(table, B, SEED, n)
    res = {"taxa": n, "sites": sites, "rows": B + 1, "patterns": int(src[1].shape[0]),
           "nonzero": int(torch.count_nonzero(rows).item()), "count_rows_kernel_ms": events(new),
           "single_table_route_ms": events(old), "tables_equal": bool(torch.equal(new().view(torch.int64), old().view(torch.int64)))}
    if n >= 32:
        comp = lambda: eng._pair_tables_compacted_rows(src[0], rows, n)  # noqa: E731
        res["compacted_rows_route_ms"] = events(comp)
        res["compacted_rows_equal"] = bool(torch.equal(comp().view(torch.int64), old().view(torch.int64)))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-windows", type=int, default=3)
    ap.add_argument("--routes-only", action="store_true", help="only the pair-table routes by taxon count")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("window_bootstrap_timing.py needs a CUDA device")
    res = {"gpu": gpu_info(), "seed": SEED}
    res["routes_by_taxa"] = []
    for n in (12, 20, 24, 31, 32, 36, 40, 44, 48, 56, 64):
        res["routes_by_taxa"].append(route_by_taxa(n))
        print(json.dumps(res["routes_by_taxa"][-1]), file=sys.stderr, flush=True)
    for n, B in (() if args.routes_only else ((20, 100), (64, 20))):
        res[f"t{n}_b{B}"] = case(n, B, args.host_windows)
        print(json.dumps(res[f"t{n}_b{B}"]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
