"""Timing of quartet split scores (batch.quartet_scores; engine.quartet_scores, csrc/quartets.cu) on seeded inputs of
bench_inputs (balanced tree, JC, branch length 0.05): every quartet of 20, 32 and 64 taxa x 10^6 sites, each method.

Per case and method, device times from CUDA events (median of `--repeats` runs after a warm-up run of the same shape):
  pack      the uint8 code matrix (already on the device) -> bit planes (engine.pack)
  tables    spb_quartet_tables over all groups (flattening, mutual information) or the pair tables (subflattening)
  score     spb_quartet_flattening_scores / spb_quartet_mi_scores / the subflattening scorer, with the column mapping
  call_ms   the whole batch.quartet_scores call from host codes (host clock, ends in a device synchronise)
The counting kernel's work, Q x 256 AND + POPC per 32-site word, is computed from the shapes and divided by the tables time.
The host time of the default quartet list (engine.all_quartets) is timed on its own.

Baseline: the drop-in loop a user would write today, per quartet Alignment(mapping, taxa).sub_alignment([a, b, c, d]),
then flattening(split, sub, FlatFormat.reduced) and split_score for its three splits, with `mapping` the pattern counts of
the whole alignment (built and uploaded once, not timed).  It is timed on a SAMPLE of `--sample` random quartets and reported as that
sample's time; the maximum difference of its scores from the flattening column of quartet_scores is reported with it.

    python scripts/quartet_timing.py [--out profiles/r12_quartet_timing.json] [--repeats 3] [--sample 20]

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
from splitp_b200.enums import FlatFormat, Method  # noqa: E402
from splitp_b200.parsers.fasta import get_pattern_counts  # noqa: E402
from tests import quartet_reference as QR  # noqa: E402  (true quartet topologies of the balanced tree)

eng = sp.engine
SITES = 1_000_000


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


def phases(d_codes, q, method):
    """Device times of one engine.quartet_scores run from codes on the device: {pack, tables, score} in ms."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    timer = eng.PhaseTimer()
    a.record()
    aln = eng.pack(d_codes, want_sm=False)
    b.record()
    out = eng.quartet_scores(aln, q, method, timer)
    torch.cuda.synchronize()
    tot = timer.totals()
    return {"pack": a.elapsed_time(b), "tables": tot["tables"][0], "score": tot["score"][0]}, out


def drop_in_sample(codes, taxa, quartets):
    """The per-quartet drop-in loop over `quartets` (labels): (ms, scores [len, 3])."""
    mapping, _ = get_pattern_counts(BI.codes_to_sequences(codes, taxa))
    aln = sp.Alignment(mapping, taxa)
    eng.table_from_mapping(aln)  # the one-time upload of the mapping; each sub_alignment call still validates it
    out = np.zeros((len(quartets), 3))

    def run():
        for i, (a, b, c, d) in enumerate(quartets):
            sub = aln.sub_alignment([a, b, c, d])
            for j, split in enumerate([((a, b), (c, d)), ((a, c), (b, d)), ((a, d), (b, c))]):
                out[i, j] = float(sp.split_score(sp.flattening(split, sub, FlatFormat.reduced)))
        return out
    ms, _ = wall(run)
    return ms, out


def case(n, repeats, sample):
    codes = BI.simulate_codes(n, 0.05, "JC", SITES, n)
    taxa = BI.taxa_of(BI.balanced_parents(n)[1])
    t0 = time.perf_counter()
    q = eng.all_quartets(n)
    list_ms = (time.perf_counter() - t0) * 1e3
    Q, words = int(q.shape[0]), (SITES + 31) // 32
    ops = Q * 256 * words
    d_codes = torch.from_numpy(codes).cuda()
    res = {"taxa": n, "sites": SITES, "quartets": Q, "quartet_list_host_ms": list_ms, "table_and_popc_ops": ops}
    full = {}
    for m in (Method.flattening, Method.mutual_information, Method.subflattening):
        phases(d_codes, q, m)  # warm-up of the same shapes
        runs = [phases(d_codes, q, m)[0] for _ in range(repeats)]
        med = {k: float(np.median([r[k] for r in runs])) for k in runs[0]}
        call_ms = [wall(lambda: batch.quartet_scores(codes, None, m))[0] for _ in range(repeats)]
        full[m.name] = batch.quartet_scores(codes, None, m)
        entry = {"phase_ms": med, "phase_ms_all": runs, "call_ms": float(np.median(call_ms)), "call_ms_all": call_ms}
        if m != Method.subflattening:
            entry["table_ops_per_s"] = ops / (med["tables"] * 1e-3)
        res[m.name] = entry
        print(json.dumps({"taxa": n, m.name: entry}), flush=True)
    truth = QR.true_pairing(QR.leaf_distances(n), q)
    res["true_topology_fraction"] = {k: float((v.argmin(axis=1) == truth).mean()) for k, v in full.items()}
    rng = np.random.default_rng(n)
    pick = rng.choice(Q, sample, replace=False)
    labels = [tuple(taxa[i] for i in row) for row in q[pick].tolist()]
    drop_in_sample(codes[:, :1000], taxa, labels[:1])  # warm-up
    ms, scores = drop_in_sample(codes, taxa, labels)
    ref = full["flattening"][pick]
    res["drop_in_sample"] = {"quartets_timed": sample, "ms": ms, "ms_per_quartet": ms / sample,
                             "max_rel_diff_to_quartet_scores": float(np.max(np.abs(scores - ref) / np.maximum(np.abs(ref), 1e-300)))}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_quartet_timing.json"))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sample", type=int, default=20)
    ap.add_argument("--taxa", type=int, nargs="+", default=[20, 32, 64])
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "cases": [case(n, args.repeats, args.sample) for n in args.taxa], "gpu_after": gpu_info()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
