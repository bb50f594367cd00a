"""Dense count flattenings (engine.CountScorer) against the sparse route (engine.sparse_flattening_scores) on the largest
size classes of 15 and 16 taxa, on both sides of 32,768 distinct patterns (above it the tensor-core Gram of these classes
splits its K dimension and needs a workspace of rows_pad^2 int64 per matrix of a launch).

Inputs: the alignments of tests/test_gpu_score_limits.py (balanced Jukes-Cantor tree, branch length 0.02, plus uniformly
random sites).  Per (alignment, class): 4 random splits scored by each route once to warm up, then timed over 3 calls
(host clock around calls that end in a device synchronise), with the peak of device memory allocated during the calls.
The dense route is the scorer's per-class path (CountScorer._score_group), whatever route score_many picks for the class.
A route that cannot allocate its buffers is reported with its error.

    python scripts/dense_flattening_limits_timing.py [--out FILE]

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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench_inputs as BI  # noqa: E402
import splitp_b200 as sp  # noqa: E402

eng = sp.engine
CASES = [(15, 40_000, 8_000), (15, 60_000, 33_000), (16, 40_000, 8_000), (16, 60_000, 30_000)]  # (n, tree sites, random sites)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip().splitlines()[:1]}


def codes_of(n, N, random_sites, seed):
    codes = BI.simulate_codes(n + n % 2, 0.02, "JC", N, seed)[:n]
    noise = np.random.default_rng(seed + 1).integers(0, 4, size=(n, random_sites), dtype=np.uint8)
    return np.ascontiguousarray(np.concatenate([codes, noise], axis=1))


def side_splits(n, a, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        perm = rng.permutation(n)
        out.append((sorted(perm[:a].tolist()), sorted(perm[a:].tolist())))
    return out


def dense(scorer, splits, a):
    if scorer._batch_bytes is None:
        scorer._batch_bytes = min(48 << 30, torch.cuda.mem_get_info()[0] // 3)
    out = torch.empty(len(splits), dtype=torch.float64, device=eng.device())
    scorer._score_group(splits, a, list(range(len(splits))), out, 512, scorer._batch_bytes)
    return out


def timed(fn, reps=3):
    try:
        fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        t0 = time.perf_counter()
        for _ in range(reps):
            out = fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / reps
        return {"ms_per_call": round(ms, 3), "peak_extra_gib": round((torch.cuda.max_memory_allocated() - base) / 2**30, 2)}, out
    except Exception as exc:  # noqa: BLE001  (an allocation failure or a geometry the kernels refuse is a result here)
        torch.cuda.synchronize()
        return {"error": f"{type(exc).__name__}: {str(exc).splitlines()[0][:200]}"}, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows = []
    for n, N, noise in CASES:
        codes = codes_of(n, N, noise, 100 + n)
        table = eng.count_patterns(eng.pack(codes))
        for a in range(5, n // 2 + 1):
            splits = side_splits(n, a, 4, 10 * n + a)
            scorer = eng.CountScorer(table)
            d, d_out = timed(lambda: dense(scorer, splits, a))
            del scorer
            torch.cuda.empty_cache()
            s, s_out = timed(lambda: eng.sparse_flattening_scores(table, splits))
            row = {"taxa": n, "patterns": table.num, "class": f"{a}|{n - a}", "splits": len(splits), "dense": d, "sparse": s}
            if d_out is not None and s_out is not None:
                row["max_rel_diff"] = float(((d_out - s_out).abs() / s_out.abs()).max())
            rows.append(row)
            print(json.dumps(row), flush=True)
            torch.cuda.empty_cache()
    res = {"gpu": gpu_info(), "rows": rows}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
