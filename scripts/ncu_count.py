"""One pattern-count launch (12 taxa x 10^8 sites, direct table) bracketed by cudaProfilerStart/Stop, for
`ncu --profile-from-start off`; prints the CUDA-event time of the same launch."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import splitp_b200 as sp
eng = sp.engine
n, N = 12, int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
tree = sp.trees.balanced_tree(n, 0.05)
codes = sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=12)
aln = eng.pack(codes, want_planes=False)
del codes
table = torch.zeros(4 ** n, dtype=torch.int32, device="cuda")
usable = torch.zeros(1, dtype=torch.int64, device="cuda")


def run():
    eng.call("spb_count_direct", eng._p(aln.sm), eng._p(aln.valid), n, 0, N, eng._p(table), None, eng._p(usable), eng._st())


run()
torch.cuda.synchronize()
table.zero_()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.profiler.start()
a.record()
run()
b.record()
torch.cuda.synchronize()
torch.cuda.profiler.stop()
cnt = table.to(torch.int64)
consts = [int(cnt[c * 0x555555].item()) for c in range(4)]
print(f"N={N} ms={a.elapsed_time(b):.4f} distinct={int((cnt > 0).sum())} "
      f"constant-pattern share={sum(consts) / N:.4f} sum={int(cnt.sum())}")
