"""Micro-benchmark of the G0 Q product kernels of the eigen-solver (spb_symv_i32: 0 = column-owning FMA kernel, 1 = DMMA
kernel) on the same int32 Gram batch, checked against torch fp64, timed with CUDA events.
Usage: python scripts/symv_bench.py [k] [batch]"""
import ctypes
import json
import sys

import torch

sys.path.insert(0, ".")
from splitp_b200 import _lib  # noqa: E402

lib = _lib.lib
k = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
nb = int(sys.argv[2]) if len(sys.argv) > 2 else 48
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(1)
G = torch.randint(0, 1 << 27, (nb, k, k), dtype=torch.int32, device=dev, generator=g)
Q = torch.randn((nb, 8, k), dtype=torch.float64, device=dev, generator=g)
AQ = torch.empty_like(Q)
Qt = torch.empty(int(lib.spb_symv_i32_ws(k, nb)), dtype=torch.float64, device=dev)
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
ref = torch.stack([Q[b] @ G[b].double() for b in range(min(nb, 4))])
scale = ref.abs().max().item()
out = {"k": k, "batch": nb, "mbytes_per_matrix": k * k * 4 / 1e6, "variants": {}}
for variant in range(2):
    AQ.zero_()
    rc = lib.spb_symv_i32(G.data_ptr(), k, k, nb, Q.data_ptr(), AQ.data_ptr(), Qt.data_ptr(), variant, st)
    assert rc == 0, (variant, lib.spb_last_error())
    torch.cuda.synchronize()
    err = (AQ[: ref.shape[0]] - ref).abs().max().item() / scale
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        lib.spb_symv_i32(G.data_ptr(), k, k, nb, Q.data_ptr(), AQ.data_ptr(), Qt.data_ptr(), variant, st)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    us = min(ts) * 1e3 / nb
    out["variants"][variant] = {"us_per_matrix": round(us, 2), "gbs": round(k * k * 4 / us / 1e3, 1), "rel_err": err}
    print(f"variant {variant}: {us:7.2f} us per {k}^2 product  {k * k * 4 / us / 1e3:7.1f} GB/s  rel err {err:.2e}", flush=True)
print(json.dumps(out))
