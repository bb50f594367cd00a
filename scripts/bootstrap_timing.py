"""Timing of bootstrap split scores (csrc/bootstrap.cu, engine.bootstrap_tables, batch.bootstrap_scores) on seeded inputs of
bench_inputs:

  (a) c2: 12 taxa x 10^6 sites (bench workload c2's input), all 2,035 flattening splits, B = 100 replicates;
  (b) c3: 20 taxa x 10^7 sites (bench workload c3's input, GTR), all 524,267 subflattening splits, B = 20;
  (c) c2's input, mutual information of all 2,035 splits, B = 100.

Per workload: CUDA-event time of the resampling kernel for all B replicates in one call (draws / s), of the compaction of
those B count rows, the host-clock time of bootstrap_scores (bracketed by device synchronises) and of score_splits on the
original alignment, each after one untimed run of the same shape (for bootstrap_scores: B = 2).  "scoring per replicate" is
(bootstrap_scores - resampling - compaction) / B.  Atomics issued by the resampling kernel after the warp aggregation are
counted with the host model (tests/bootstrap_reference.py) over the first `--model-reps` replicates.

    python scripts/bootstrap_timing.py [--out profiles/r6_bootstrap_timing.json] [--sites-c3 10000000]

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
from tests import bootstrap_reference as BR  # noqa: E402

eng = sp.engine
SEED = 2024


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
    """Best CUDA-event time (ms) of fn() over `reps` runs after one warm-up."""
    fn()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def resampling(codes, B, model_reps):
    table = eng.count_patterns(eng.pack(codes))
    keys, counts = table.keys.contiguous(), table.counts.contiguous()
    prefix, N = eng._bootstrap_prefix(counts)
    P = int(counts.shape[0])
    rows = torch.empty((B, P), dtype=torch.int32, device=keys.device)
    draw_ms = events(lambda: eng.call("spb_bootstrap_counts", eng._p(prefix), P, N, SEED, 0, B, eng._p(rows), eng._st()))
    cap = B * min(P, N)
    ok, oc = torch.empty(cap, dtype=torch.int64, device=keys.device), torch.empty(cap, dtype=torch.int32, device=keys.device)
    off = torch.empty(B + 1, dtype=torch.int64, device=keys.device)
    ws = torch.empty(int(eng.lib.spb_bootstrap_compact_ws(P, B)), dtype=torch.int64, device=keys.device)
    compact_ms = events(lambda: eng.call("spb_bootstrap_compact", eng._p(rows), eng._p(keys), 1, P, B, eng._p(ok), eng._p(oc), cap,
                                         eng._p(off), eng._p(ws), eng._st()))
    host = counts.cpu().numpy().view(np.uint32).astype(np.int64)
    atomics = [BR.atomics_after_aggregation(BR.draws(host, SEED, b)) for b in range(model_reps)]
    nnz = (off[1:] - off[:-1]).double().mean().item()
    return {"patterns": P, "sites": N, "replicates": B, "draws": B * N,
            "resample_ms": draw_ms, "resample_ms_per_replicate": draw_ms / B, "draws_per_s": B * N / (draw_ms * 1e-3),
            "atomics_per_replicate_model": float(np.mean(atomics)), "atomics_per_draw_model": float(np.mean(atomics)) / N,
            "model_replicates": model_reps,
            "compact_ms": compact_ms, "compact_ms_per_replicate": compact_ms / B, "mean_patterns_per_replicate": nnz}


def workload(codes, splits, method, B, model_reps):
    res = resampling(codes, B, model_reps)
    m = getattr(sp.Method, method)
    sp.batch.score_splits(codes, splits, m)
    res["score_splits_ms"] = min(wall(lambda: sp.batch.score_splits(codes, splits, m))[0] for _ in range(3))
    sp.batch.bootstrap_scores(codes, splits, m, replicates=2, seed=SEED)
    ms, out = wall(lambda: sp.batch.bootstrap_scores(codes, splits, m, replicates=B, seed=SEED))
    scoring = (ms - res["resample_ms"] - res["compact_ms"]) / B
    res.update({"splits": len(splits), "method": method, "bootstrap_scores_ms": ms, "bootstrap_ms_per_replicate": ms / B,
                "scoring_ms_per_replicate": scoring, "resample_share_of_scoring": res["resample_ms_per_replicate"] / scoring,
                "finite_scores": bool(np.isfinite(out).all())})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sites-c3", type=int, default=10_000_000)
    ap.add_argument("--model-reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bootstrap_timing.py needs a CUDA device")
    res = {"gpu": gpu_info(), "seed": SEED}
    c2 = BI.simulate_codes(12, 0.05, "JC", 1_000_000, 2)
    res["a_c2_flattening"] = workload(c2, BI.all_splits_idx(12), "flattening", 100, args.model_reps)
    res["c_c2_mutual_information"] = workload(c2, BI.all_splits_idx(12), "mutual_information", 100, args.model_reps)
    c3 = BI.simulate_codes(20, 0.05, "GTR", args.sites_c3, 3)
    res["b_c3_subflattening"] = workload(c3, BI.all_splits_idx(20), "subflattening", 20, 1)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
