"""A/B timing of pair_kernel (spb_pair_tables) between two builds of the library, in one session, runs alternating:

    python scripts/pair_kernel_ab.py --base DIR_OF_OTHER_BUILD [--out profiles/r8_pair_kernel_ab.json] [--rounds 3]

For each build (the tree this script is in, and --base: another checkout with its library built) and each taxon count
20 / 32 / 40 / 64 (pair_kernel<PPT> with PPT = 1 / 2 / 4 / 8), the kernel time of one spb_pair_tables pass over random
codes on the device, planes of about 320 MB (larger than the 126 MB L2): CUDA events over 20 launches after one warm-up,
launches only.  Then bench.py --workload c3 and c5 (subflattening end to end: c3 runs pair_kernel<1>, c5 pair_kernel<2>)
from each tree.  Prints one JSON object with the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KERNEL = r"""
import json, sys, torch
sys.path.insert(0, sys.argv[1])
import splitp_b200 as sp
eng = sp.engine
out = {}
for n in (20, 32, 40, 64):
    N = (1_280_000_000 // n) // 32 * 32
    aln = eng.pack(torch.randint(0, 4, (n, N), dtype=torch.uint8, device="cuda"), want_sm=False)
    raw = eng._zeros(int(eng.lib.spb_pair_raw_words(n)), torch.int64)
    run = lambda: eng.call("spb_pair_tables", eng._p(aln.planes), eng._p(aln.valid), n, aln.plane_words, 0, aln.plane_words,
                           eng._p(raw), eng._st())
    run()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        run()
    b.record()
    b.synchronize()
    out[n] = {"sites": N, "ms": a.elapsed_time(b) / 20}
    del aln, raw
    torch.cuda.empty_cache()
print(json.dumps(out))
"""


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[:1]


def bench(tree, workload):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "5", "--warmup", "2", "--workload", workload,
                        "--extras", "none"], cwd=tree, capture_output=True, text=True)
    line = [x for x in r.stdout.strip().splitlines() if x.startswith("{")][-1]
    return json.loads(line)["value"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True)
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    trees = {"base": os.path.abspath(args.base), "this": ROOT}
    res = {"gpu": gpu_info(), "kernel_ms": {k: [] for k in trees}, "c3_split_scores_per_s": {k: [] for k in trees},
           "c5_split_scores_per_s": {k: [] for k in trees}}
    for _ in range(args.rounds):
        for name, tree in trees.items():
            r = subprocess.run([sys.executable, "-c", KERNEL, tree], capture_output=True, text=True, check=True)
            res["kernel_ms"][name].append(json.loads(r.stdout.strip().splitlines()[-1]))
    for _ in range(2):
        for name, tree in trees.items():
            res["c3_split_scores_per_s"][name].append(bench(tree, "c3"))
            res["c5_split_scores_per_s"][name].append(bench(tree, "c5"))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
