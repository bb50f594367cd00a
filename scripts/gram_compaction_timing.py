"""Per-class Gram timing of CountScorer.score_many with column ranks (S0 holds the occupied columns only) on the c2 input:
12 taxa, JC, branch length 0.05, 10^6 sites, seed 2 (bench_inputs.simulate_codes), all 2,035 splits.

For every size class: the Gram launches (CUDA events around each launch through CountScorer.gram_hook, summed), the rank pass
(spb_col_ranks_batch of the same batches, CUDA events, run again outside score_many), the occupied columns per split
(min / mean / max) and the executed tensor-core or dp4a ops on the compacted K:
    2 * computed output cells * K tiles * 128  (tcgen05: only the 256-blocks touching the upper triangle are computed)
    2 * rows_pad^2 * ceil(ncols / 4) * 4        (dp4a, rows_pad <= 32)
summed over the matrices.  bench.py's roofline still counts 4096 columns per 6|6 Gram; these are the ops actually issued.

    python scripts/gram_compaction_timing.py [--sites 1000000] [--reps 3] [--out FILE]

Prints one JSON object with the GPU's name and power limit beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

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


def computed_cells(layout, rows_pad):
    if layout == eng.SPB_S0_K4MAJOR or rows_pad == 128:
        return rows_pad * rows_pad
    B = rows_pad // 256
    return B * (B + 1) // 2 * 256 * 256


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n = 12
    codes = torch.from_numpy(BI.simulate_codes(n, 0.05, "JC", args.sites, 2)).cuda()
    tab = eng.count_patterns(eng.pack(codes))
    idx = BI.all_splits_idx(n)
    scorer = eng.CountScorer(tab)
    spans = {}

    def hook(run, nb):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        spans.setdefault(hook.cls, []).append((e0, e1, nb))

    scorer.score_many(idx)  # warm-up: buffers, modules
    torch.cuda.synchronize()
    scorer.gram_hook = hook
    classes = {}
    for s, (ia, ib) in enumerate(idx):
        classes.setdefault(min(len(ia), len(ib)), []).append(s)
    gram_ms = {a: [] for a in classes}
    for _ in range(args.reps):
        spans.clear()
        for a, members in sorted(classes.items()):
            hook.cls = a
            sub = [idx[s] for s in members]
            scorer.score_many(sub)
        torch.cuda.synchronize()
        for a in classes:
            gram_ms[a].append(sum(e0.elapsed_time(e1) for e0, e1, _ in spans[a]))
    scorer.gram_hook = None
    out = {"gpu": gpu_info(), "sites": args.sites, "patterns": tab.num, "n_hi": scorer.n_hi, "classes": {}}
    for a, members in sorted(classes.items()):
        R, Cc = 4 ** a, 4 ** (n - a)
        layout, rows_pad, pitch = scorer.geometry(R, Cc)
        rec, _ = scorer._encoded_group(idx, a, members)
        ncols_all, rank_ms = [], 0.0
        for b0 in range(0, len(members), scorer.GNB):
            nb = min(scorer.GNB, len(members) - b0)
            arr = (sp._lib.SpbSplit * nb).from_buffer(rec, b0 * rec.itemsize)
            scorer._col_ranks(arr, nb)  # warm
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, _, ncols = scorer._col_ranks(arr, nb)
            e1.record()
            torch.cuda.synchronize()
            rank_ms += e0.elapsed_time(e1)
            ncols_all.append(ncols[:nb].cpu().numpy().astype(np.int64))
        nc = np.concatenate(ncols_all)
        if layout == eng.SPB_S0_K4MAJOR:
            kexec = (nc + 3) // 4 * 4
        else:
            kexec = np.maximum(1, (nc + 127) // 128) * 128
        ops = 2.0 * computed_cells(layout, rows_pad) * float(kexec.sum())
        ms = float(np.median(gram_ms[a]))
        out["classes"][f"{a}|{n - a}"] = {
            "splits": len(members), "rows_pad": rows_pad, "K_full": pitch, "S0_pitch": scorer._col_pitch(layout, pitch),
            "ncols_min": int(nc.min()), "ncols_mean": float(nc.mean()), "ncols_max": int(nc.max()),
            "K_share": float(kexec.mean() / pitch),
            "route": "int32" if scorer._use_i32(layout, rows_pad, pitch) and R > eng.JACOBI_MAX_K else "fp64",
            "gram_ms": ms, "gram_ms_reps": [round(x, 4) for x in gram_ms[a]], "rank_pass_ms": rank_ms,
            "executed_ops": ops, "executed_TOPS": ops / (ms * 1e-3) / 1e12 if ms > 0 else None,
        }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
