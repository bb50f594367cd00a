#!/usr/bin/env python
"""Benchmark of the SplitP hot path on B200 (contract: the task statement; metric: BASELINE.json).

    python bench.py --gpus N --steps K --warmup W [--workload c2|c3|c4|c5] [--extras c3,c5,c4|none] [--impl reference]
                    [--dump-outputs DIR]

Headline workload c2 (BASELINE.json configs[1]): balanced 12-taxon Jukes-Cantor tree, branch length 0.05, 1,000,000
sites (seeded synthetic alignment from bench_inputs.py, identical in both arms), ALL 2,035 splits scored from dense count
flattenings (4^a x 4^b, 4096 x 4096 for the 462 6|6 splits) through the exact-integer tensor-core Gram + eigen-solver.
One step = one pass of the whole path: pack -> pattern count -> (count allreduce) -> per split flatten + Gram +
high-part correction + score -> (score all-gather).

The same JSON line carries a `workloads` object with the other BASELINE configs, each measured the same way (same number of
timed steps): c3 (configs[2], the north-star target: 20-taxon GTR tree, 10M sites, subflattening scores of all 524,267 splits),
c5 (configs[4]: 10^5 random splits of a 32-taxon tree) and c4 (configs[3] scaled to 10M sites: 64 taxa, 128-bit pattern
compression + thin reduced-flattening scores).

`--dump-outputs DIR` writes the scores that each GPU workload's last timed step returned, DIR/<workload>_scores.npy (float64,
split-list order), and names the file under `dumped` in that workload's result (null when the workload failed).  Every input
is generated from a fixed seed, so two builds of the project can be compared output for output.

N > 1 (torchrun): splits are sharded for scoring; sites are sharded for counting (exchange of the compacted pattern lists /
integer allreduce of the pair statistics) unless counting the whole alignment on every rank is cheaper than that exchange
(c2: 0.16 ms against 1.5 ms on 8 ranks; `config.parallelism` says which); total work is fixed => "scaling": "strong".
All lines carry `phase_ms`.

`--impl reference` times the UNMODIFIED reference (pip-installed into the git-ignored baseline/_ref, see DESIGN.md) on
the host cores: get_pattern_counts over all sites + flattening(reduced) + split_score for a stratified sample of
splits; the oracle port is timed beside it.  That process imports neither torch nor splitp_b200.
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to its children; the CPU arm must use the box's host cores whatever launched
    # it, and BLAS reads these variables when numpy is first imported -- so they are set before that import
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_host_cores())

import argparse  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

import bench_inputs as BI  # noqa: E402

WORKLOADS = {
    "c2": dict(n=12, sites=1_000_000, bl=0.05, model="JC", seed=2, method="flattening",
               desc="BASELINE configs[1]: balanced 12-taxon JC tree bl=0.05, 1M sites, all 2035 splits, dense count "
                    "flattenings (6|6 = 4096x4096), exact u8 tensor-core Gram + eigen score"),
    "c3": dict(n=20, sites=10_000_000, bl=0.05, model="GTR", seed=3, method="subflattening",
               desc="BASELINE configs[2]: balanced 20-taxon GTR tree bl=0.05, 10M sites, subflattening scores of all "
                    "524267 splits"),
    "c4": dict(n=64, sites=10_000_000, bl=0.05, model="JC", seed=4, method="thin", pair_splits=True,
               desc="BASELINE configs[3] (scaled: 10M sites by default, --sites 100000000 for the full size): balanced 64-taxon JC "
                    "tree bl=0.05, 128-bit pattern compression + reduced flattening scores of 2|62 splits"),
    "c5": dict(n=32, sites=1_000_000, bl=0.05, model="JC", seed=5, method="subflattening", random_splits=100_000,
               desc="BASELINE configs[4]: 10^5 random splits (side sizes 2..16, numpy default_rng(5)) of a balanced 32-taxon JC "
                    "tree bl=0.05, 1M sites, subflattening scores"),
}
EXTRA_SPLIT_CAP = {"c4": 256}  # splits scored when c4 runs as an extra workload (stated in its config)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--extras", default=None, help="comma list of extra workloads reported under `workloads` "
                    "(default: c3,c5,c4 when the headline is c2; 'none' to skip)")
    ap.add_argument("--sites", type=int, default=None, help="override the number of sites of the headline workload")
    ap.add_argument("--max-splits", type=int, default=None, help="score only the first M splits (debug runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores of every GPU workload's last timed step to DIR/<workload>_scores.npy (float64, one "
                         "per split in split-list order; under 4.2 MB per workload), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    return args


def split_list(wl, max_splits=None):
    """Position form of the workload's split list (all_splits order, bench_inputs.all_splits_idx)."""
    if wl.get("pair_splits"):
        out = BI.all_splits_idx(wl["n"], size=2)
    elif wl.get("random_splits"):
        out = BI.random_splits_idx(wl["n"], wl["random_splits"], seed=5)
    else:
        out = BI.all_splits_idx(wl["n"])
    return out[:max_splits] if max_splits else out


def sites_replicated(wl, world):
    """Mirror of splitp_b200.batch.replicate_sites (kept here so that the reference arm does not import the package)."""
    return wl["method"] == "flattening" and world > 1 and float(wl["n"]) * float(wl["sites"]) <= 2.0e8


def config_of(name, wl, n_splits, world):
    """The `config` object: identical keys and values in both arms."""
    par = f"splits sharded x{world} (contiguous runs of the size-class-ordered list, cut at equal modelled cost), sites " \
          f"replicated (counting them all is cheaper than the exchange)" if sites_replicated(wl, world) \
        else f"sites+splits sharded x{world}"
    return {"workload": wl["desc"], "name": name, "taxa": wl["n"], "sites": wl["sites"], "splits": n_splits,
            "model": wl["model"], "branch_length": wl["bl"], "seed": wl["seed"],
            "l2": "flushed between timed steps (256 MB fill)", "parallelism": par}


# ------------------------------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed loops: an in-process NVML (nvidia_ml_py) thread polling
    the two cheap per-field queries every 100 ms, initialised before the warm-up.  Measured on the c2 step
    (scripts/step_jitter.py): this leaves the steps within +3 ms, whereas a looping `nvidia-smi` child, a poll from the
    launching thread, or cudaMemGetInfo inside the step each produced sporadic 100-170 ms steps.
    Falls back to a looping nvidia-smi child when NVML is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.nvml, self.handle, self.max_mhz = None, None, None
        self.sm, self.reasons, self.active = [], set(), False
        self.quit = threading.Event()

    def _poll(self):
        n = self.nvml
        masks = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        while not self.quit.wait(0.1):
            if not self.active:
                continue
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:  # noqa: BLE001
                continue
            if self.active:
                self.sm.append(mhz)
                self.reasons.update(k for k, m in masks.items() if r & m)

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            # torch device `index` of this process -> NVML handle via the PCI bus id (CUDA_VISIBLE_DEVICES-proof)
            bus = getattr(torch.cuda.get_device_properties(self.index), "pci_bus_id", None)
            if isinstance(bus, int):
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.handle = h
                        break
            if self.handle is None:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)  # the first query initialises (about 20 ms)
            self.nvml = pynvml
            threading.Thread(target=self._poll, daemon=True).start()
            return
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] NVML sampling unavailable ({type(exc).__name__}: {exc}); falling back to nvidia-smi", file=sys.stderr)
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "250",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            if self.active:
                self.rows.append([x.strip() for x in line.split(",")])

    def reset(self):
        """Start of a timed loop: forget earlier samples and record from now on."""
        self.sm, self.reasons, self.rows = [], set(), []
        self.active = True

    def sample(self):
        """One extra sample from the calling thread (used when a timed loop is shorter than the polling period)."""
        if self.nvml is not None and not self.sm:
            try:
                self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)))
            except Exception:  # noqa: BLE001
                pass

    def close(self):
        self.quit.set()
        if self.proc is not None:
            self.proc.terminate()
            self.proc = None

    def stop(self):
        """End of a timed loop: summary of the samples taken since reset()."""
        self.active = False
        if self.nvml is not None:
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml thread, 100 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi -lms 250"}


# ------------------------------------------------------------------------------------------------
# CPU side: the unmodified reference (baseline/_ref) and the oracle port, on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------
def load_reference():
    """The pip-installed, unmodified js51/SplitP from the git-ignored baseline/_ref (None when it did not travel)."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "splitp")):
        print("[bench] baseline/_ref not installed (build() with SPLITP_REFERENCE set installs it): the CPU baseline is the "
              "oracle port", file=sys.stderr)
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import splitp
        import splitp.parsers.fasta  # noqa: F401
        return splitp if os.path.realpath(splitp.__file__).startswith(os.path.realpath(ref_dir)) else None
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] reference import failed: {type(exc).__name__}: {exc}", file=sys.stderr)
        return None


def blas_threads():
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=_host_cores())
        return max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:  # noqa: BLE001
        return None


def stratified_sample(idx_all, per_size=1):
    """One (or per_size) split(s) per short-side size, taken from the middle of each size class."""
    by_size = {}
    for s, (ia, ib) in enumerate(idx_all):
        by_size.setdefault(min(len(ia), len(ib)), []).append(s)
    picks = {}
    for a, members in sorted(by_size.items()):
        step = max(1, len(members) // (per_size + 1))
        picks[a] = [members[min(len(members) - 1, (j + 1) * step)] for j in range(per_size)]
    return by_size, picks


def cpu_flattening_sample(name, wl, codes, idx_all, use_reference=True, sizes=None, budget_s=60.0):
    """Times the CPU path of a `flattening`-method workload on the host cores.

    Stage 1 (measured on ALL sites): pattern counting -- the reference's get_pattern_counts (fasta.py:48-63) +
    pattern_counts_to_probs, and the oracle port.  Stage 2 (measured on a stratified sample: one split per short-side
    size): flattening(split, probs, FlatFormat.reduced) + split_score (constructions.py:31-55, phylogenetics.py:280-300).
    The whole-job rate is the size-weighted estimate S / (t_count + sum_a n_a t_a); measured and extrapolated parts are
    reported separately.  Returns (cpu_baseline dict, {split index: reference score})."""
    from oracle import splitp_oracle as O
    n = wl["n"]
    taxa = BI.taxa_of(BI.balanced_parents(n)[1])
    by_size, picks = stratified_sample(idx_all)
    if sizes is not None:
        picks = {a: p for a, p in picks.items() if a in sizes}
    ref = load_reference() if use_reference else None
    out = {"unit": "split-scores/s", "cores": _host_cores(), "blas_threads": blas_threads()}
    scores = {}
    # ---- oracle port (numpy + LAPACK) ----
    t0 = time.perf_counter()
    keys, counts, usable = O.get_pattern_counts_arrays(codes)
    t_count_port = time.perf_counter() - t0
    vals = counts / float(usable)
    port_t, port_scores = {}, {}
    for a, members in picks.items():
        ia, ib = idx_all[members[0]]
        t1 = time.perf_counter()
        port_scores[members[0]] = float(O.split_score(O.flattening_reduced(keys, vals, n, ia, ib)))
        port_t[a] = time.perf_counter() - t1
    port_total = t_count_port + sum(len(by_size[a]) * port_t[a] for a in port_t)
    covered = sum(len(by_size[a]) for a in port_t)
    out["port"] = {"value": covered / port_total, "t_count_s": t_count_port, "t_split_s": {str(a): port_t[a] for a in port_t},
                   "sites_per_s": codes.shape[1] / t_count_port}
    if ref is None:
        out.update({"kind": "port", "value": out["port"]["value"], "sites_per_s": out["port"]["sites_per_s"],
                    "sample": f"oracle port (baseline/_ref absent): pattern count of all {codes.shape[1]} sites + one split per side size "
                              f"{sorted(port_t)} (reduced flattening + LAPACK gesdd score); value = S / (t_count + sum_a n_a t_a)"})
        return out, port_scores
    # ---- the unmodified reference ----
    seqs = BI.codes_to_sequences(codes, taxa)
    t0 = time.perf_counter()
    pc, seq_len = ref.parsers.fasta.get_pattern_counts(seqs)
    probs = ref.parsers.fasta.pattern_counts_to_probs(pc, seq_len)
    t_count = time.perf_counter() - t0
    assert seq_len == usable and len(pc) == len(keys), "reference and oracle disagree on the pattern table"
    ref_t, spent = {}, t_count
    for a, members in picks.items():
        if spent > budget_s and ref_t:
            break
        ia, ib = idx_all[members[0]]
        split = (tuple(taxa[i] for i in ia), tuple(taxa[i] for i in ib))
        t1 = time.perf_counter()
        F = ref.flattening(split, probs, ref.FlatFormat.reduced)
        tf = time.perf_counter() - t1
        sc = ref.split_score(F)
        ref_t[a] = (tf, time.perf_counter() - t1 - tf)
        spent += sum(ref_t[a])
        scores[members[0]] = float(sc)
    covered = sum(len(by_size[a]) for a in ref_t)
    total = t_count + sum(len(by_size[a]) * sum(ref_t[a]) for a in ref_t)
    if len(ref_t) < len(picks):  # budget exhausted: the largest size classes are priced with the port's time (stated)
        for a in picks:
            if a not in ref_t:
                total += len(by_size[a]) * port_t[a]
                covered += len(by_size[a])
    out.update({
        "kind": "reference", "value": covered / total, "sites_per_s": codes.shape[1] / t_count,
        "measured": {"t_count_s": t_count, "flattening_s": {str(a): ref_t[a][0] for a in ref_t},
                     "split_score_s": {str(a): ref_t[a][1] for a in ref_t}, "splits_timed": len(ref_t),
                     "rate_on_sample": len(ref_t) / max(spent, 1e-9)},
        "extrapolation": "value = S / (t_count + sum_a n_a (t_flattening_a + t_score_a)), n_a = number of splits with short side a: "
                         + ", ".join(f"{a}:{len(by_size[a])}" for a in sorted(by_size)),
        "sample": f"unmodified js51/SplitP v0.3.2 from baseline/_ref on {_host_cores()} host cores: parsers.fasta.get_pattern_counts + "
                  f"pattern_counts_to_probs over all {codes.shape[1]} sites ({t_count:.2f} s, single-threaded Python), then "
                  f"flattening(split, probs, FlatFormat.reduced) + split_score (LAPACK gesdd, all cores) for one split per short-side "
                  f"size {sorted(ref_t)}" + ("" if len(ref_t) == len(picks) else f" (sizes {sorted(set(picks) - set(ref_t))} priced with the "
                                             "oracle port's time: budget)"),
        "port_vs_reference_max_rel": max((abs(port_scores[s] - scores[s]) / abs(scores[s]) for s in scores if scores[s]), default=None),
    })
    return out, scores


def cpu_port_sample(name, wl, codes, idx_all, budget_s=15.0):
    """Oracle-port timing for the subflattening / thin workloads (the reference's own subflattening is O(rows cols P n)
    Python operations per split -- hours at 20 taxa, SURVEY.md 3.4 -- so only the port can be timed at these sizes)."""
    from oracle import splitp_oracle as O
    n = wl["n"]
    S = len(idx_all)
    cores = _host_cores()
    if wl["method"] == "thin":
        sub = codes[:, : min(codes.shape[1], 200_000)]
        t0 = time.perf_counter()
        d, usable = O.get_pattern_counts_wide(sub)
        t_count = time.perf_counter() - t0
        done, t2 = 0, time.perf_counter()
        while done < S and time.perf_counter() - t2 < budget_s:
            ia, ib = idx_all[(done * 7919) % S]
            side = ia if len(ia) <= len(ib) else ib
            O.split_score(O.flattening_reduced_from_dict(d, side, [t for t in range(n) if t not in side]))
            done += 1
        t_split = (time.perf_counter() - t2) / max(done, 1)
        scale = codes.shape[1] / sub.shape[1]
        return {"value": S / (scale * (t_count + S * t_split)), "unit": "split-scores/s", "cores": cores, "kind": "port",
                "blas_threads": blas_threads(), "sites_per_s": sub.shape[1] / t_count,
                "sample": f"oracle port on the first {sub.shape[1]} of {codes.shape[1]} sites: byte-row pattern count ({t_count:.2f} s) + "
                          f"{done} 2|62 splits ({t_split:.3f} s each: dict-based reduced flattening + LAPACK score); both stages are "
                          f"linear in the number of distinct patterns (= sites at 64 taxa), so value = S / (scale * (t_count + S * t_split)) "
                          f"with scale = {scale:.0f}"}
    t1 = time.perf_counter()
    tables, usable = O.pair_tables_from_codes(codes)
    t_pairs = time.perf_counter() - t1
    done, t2 = 0, time.perf_counter()
    while done < S and time.perf_counter() - t2 < budget_s:
        ia, ib = idx_all[(done * 7919) % S]
        O.split_score(O.subflattening_from_tables(tables, 1.0, ia, ib))
        done += 1
    t_split = (time.perf_counter() - t2) / max(done, 1)
    return {"value": S / (t_pairs + S * t_split), "unit": "split-scores/s", "cores": cores, "kind": "port",
            "blas_threads": blas_threads(), "sites_per_s": codes.shape[1] / t_pairs,
            "sample": f"oracle port: numpy pair tables from the {codes.shape[1]}-site code matrix ({t_pairs:.2f} s) + {done} splits "
                      f"({t_split * 1e3:.3f} ms each: subflattening from tables + LAPACK score); value = S / (t_pairs + S * t_split)"}


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write there too (NCCL prints "NCCL version ..." when the
    environment sets NCCL_DEBUG), so file descriptor 1 points at stderr for the whole run and emit() restores it."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(line, flush=True)


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, on the GPU arm's config.
    Imports neither torch nor splitp_b200 (checked by tests/test_host_cpu.py)."""
    name = args.workload
    wl = dict(WORKLOADS[name])
    if args.sites:
        wl["sites"] = args.sites
    idx_all = split_list(wl, args.max_splits)
    sites = wl["sites"] if wl["method"] == "flattening" else min(wl["sites"], 1_000_000)
    codes = BI.simulate_codes(wl["n"], wl["bl"], wl["model"], sites, wl["seed"])
    vals, cb = [], None
    steps = args.steps
    for _ in range(args.warmup):  # warm-up: page in LAPACK / the reference, smallest size class only
        if wl["method"] == "flattening":
            cpu_flattening_sample(name, wl, codes[:, : min(sites, 100_000)], idx_all, sizes={2})
        else:
            cpu_port_sample(name, wl, codes[:, : min(sites, 100_000)], idx_all, budget_s=1.0)
    t0 = time.perf_counter()
    for _ in range(steps):
        if wl["method"] == "flattening":
            cb, _ = cpu_flattening_sample(name, wl, codes, idx_all)
        else:
            cb = cpu_port_sample(name, wl, codes, idx_all, budget_s=10.0)
            if sites != wl["sites"]:
                cb["sample"] += f"; pair tables timed on {sites} of {wl['sites']} sites"
        vals.append(cb["value"])
    dt = (time.perf_counter() - t0) / steps
    v = float(np.mean(vals))
    cb["value"] = v
    cb["values_per_step"] = vals
    emit(json.dumps({"impl": "reference", "metric": "split_scores_per_sec", "value": v, "unit": "split-scores/s",
                     "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                     "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                     "config": config_of(name, wl, len(idx_all), args.gpus), "cpu_baseline": cb,
                     "threads": {"host_cores": _host_cores(), "blas_threads": cb.get("blas_threads"),
                                 "OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS")},
                     "e2e": {"value": v, "unit": "split-scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     **({"modules": sorted(m for m in ("torch", "splitp_b200", "splitp", "oracle") if m in sys.modules)}
                        if os.environ.get("SPB_BENCH_REPORT_MODULES") else {})}))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def measure_int8_peak(torch, seconds=1.0):
    """cuBLASLt IGEMM (torch._int_mm) 8192^3 on this GPU: the measured int8 tensor peak (scripts/int8_peak.py)."""
    try:
        n = 8192
        a = torch.randint(-127, 127, (n, n), dtype=torch.int8, device="cuda")
        b = torch.randint(-127, 127, (n, n), dtype=torch.int8, device="cuda").t().contiguous().t()
        ops = 2.0 * n ** 3
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = max(best, ops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, t0 = 0, time.perf_counter()
        e0.record()
        while time.perf_counter() - t0 < seconds:
            for _ in range(20):
                torch._int_mm(a, b)
            reps += 20
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        del a, b
        return {"burst": best, "sustained": ops * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12,
                "how": f"torch._int_mm (cuBLASLt IGEMM s8 x s8 -> s32) 8192^3: best of 6 / back to back for {seconds:.0f} s"}
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] int8 peak measurement failed: {type(exc).__name__}: {exc}", file=sys.stderr)
        return None


def gpu_workload(name, wl, args, ctx, steps, warmup, max_splits=None, cpu_baseline=True):
    """Measures one workload on the GPU arm; returns the result object (rank 0) or None (other ranks)."""
    torch, dist, sp, spd, eng, batch = ctx["torch"], ctx["dist"], ctx["sp"], ctx["spd"], ctx["eng"], ctx["batch"]
    rank, local, world, dev = ctx["rank"], ctx["local"], ctx["world"], ctx["dev"]
    n, N = wl["n"], wl["sites"]
    idx_all = split_list(wl, max_splits)
    S = len(idx_all)
    method = wl["method"]

    # ---- inputs: the same seeded alignment on every rank; this rank keeps its contiguous site shard ----
    if method == "flattening":
        codes_np = BI.simulate_codes(n, wl["bl"], wl["model"], N, wl["seed"])  # numpy generator shared with the CPU arm
        codes_full = torch.from_numpy(codes_np).to(dev)
    else:
        tree = sp.trees.balanced_tree(n, wl["bl"])
        model = sp.simulation.GTR.JukesCantor(0.5) if wl["model"] == "JC" else sp.simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6))
        codes_full = sp.simulation.simulate_codes(tree, model, N, wl["seed"])
        codes_np = None
    replicated = sites_replicated(wl, world)
    assert replicated == (method == "flattening" and batch.replicate_sites(n, N, world))
    sb, se = (0, N) if replicated else spd.shard_range(N, rank, world, 32)
    codes_dev = codes_full[:, sb:se].contiguous()
    if method == "subflattening":  # e2e input: the 2-bit host format (4 bases per byte instead of 1)
        planes, valid = batch.pack_planes_host(codes_dev.cpu().numpy())
        host_in = batch.HostPlanes(planes, valid, n, se - sb, pin=True)
        h2d_bytes = host_in.nbytes
    else:
        host_in = codes_dev.cpu().pin_memory()
        h2d_bytes = int(host_in.numel())
    if method != "flattening":
        del codes_full
    flush = ctx["flush"]
    # The timed steps record only the spans the roofline objects are computed from (the dominant kernel's launches, the count /
    # pair stage); the full per-phase breakdown (~130 event pairs per c2 step, 0.8 ms of host and device time) comes from separate
    # instrumented passes after the timed region.
    timer = eng.PhaseTimer(only={f"gram_i32_r{4 ** (n // 2)}", "count", "pairs"})

    if method == "thin":
        sides = [min((ia, ib), key=len) for ia, ib in spd.shard_strided(idx_all, rank, world)]

        def run(inp, t=None):
            with eng._span(t, "h2d+pack"):
                wide, valid_w, n_, N_ = eng.pack_wide(inp if inp.is_cuda else inp.to(dev, non_blocking=True))
            with eng._span(t, "count"):
                table = spd.count_patterns_wide_sharded(wide, valid_w, n_, N_, rank, world, local=True)
            with eng._span(t, "thin_gram+score", len(sides)):
                out = eng.thin_split_scores(table, sides)
            with eng._span(t, "gather"):
                return spd.gather_strided(out, S, rank, world)
        call_name = "engine.pack_wide + distributed.count_patterns_wide_sharded + engine.thin_split_scores"
    else:
        scorer = batch.SplitScorer(idx_all, None, sp.Method.flattening if method == "flattening" else sp.Method.subflattening,
                                   rank, world, sites="replicated" if replicated else "shard",
                                   refit_steps=(2,) if max(warmup, 1) >= 3 else ())  # one partition re-cut, after warm-up step 2,
                                                                                     # warmed up by step 3; never inside the timed region

        def run(inp, t=None):
            scorer.timer = t
            return scorer.device_scores(inp)
        call_name = "splitp_b200.batch.SplitScorer (= batch.score_splits with its buffers kept): host alignment -> scores"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ctx["sampler"]
    for _ in range(max(warmup, 1)):
        scores = run(codes_dev)
    barrier()

    # ---- timed: device-resident inputs ----
    sampler.reset()
    launches0 = int(eng.lib.spb_launch_count())
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for _ in range(steps):
        flush.fill_(1)  # L2 flush between timed iterations (outside the per-step event pair)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        scores = run(codes_dev, timer)
        b.record()
        evs.append((a, b))
    sampler.sample()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = int(eng.lib.spb_launch_count()) - launches0
    sc = scores.cpu().numpy()  # the last timed step's scores, taken before the passes below run the path again
    clocks = sampler.stop()
    step_ms = [a.elapsed_time(b) for a, b in evs]
    t = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / steps
    value = S / (ms_per_step * 1e-3)
    phases = {k: v for k, v in timer.totals().items()}
    # ---- instrumented passes (not part of `value`): every span, for `phase_ms` ----
    full = eng.PhaseTimer()
    evs_f = []
    for _ in range(steps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(codes_dev, full)
        b.record()
        evs_f.append((a, b))
    barrier()
    step_ms_f = [a.elapsed_time(b) for a, b in evs_f]
    phases_f = full.totals()
    phase_ms = {k: round(v[0] / steps, 4) for k, v in phases_f.items()}
    phase_ms["step_total"] = round(sum(step_ms_f) / steps, 4)
    phase_ms["note"] = "from separate fully instrumented passes after the timed region (their step_total includes the event overhead)"
    rank_busy_ms = None
    if world > 1:  # per-rank time before the score gather (= before waiting for the slowest rank): the balance of the split partition
        busy = torch.tensor([(sum(step_ms_f) - phases_f.get("gather", (0.0, 0))[0]) / steps], dtype=torch.float64, device=dev)
        allb = [torch.zeros_like(busy) for _ in range(world)]
        dist.all_gather(allb, busy)
        rank_busy_ms = [round(float(x.item()), 3) for x in allb]

    # ---- e2e: host buffers through the public batched call, H2D + D2H inside the timed region ----
    for _ in range(2):
        run(host_in).cpu()
    barrier()
    sampler.reset()
    evs2 = []
    for _ in range(steps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        host_scores = run(host_in).cpu()
        b.record()
        evs2.append((a, b))
    sampler.sample()
    barrier()
    clocks2 = sampler.stop()
    e2e_steps = [a.elapsed_time(b) for a, b in evs2]
    t2 = torch.tensor([sum(e2e_steps)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_ms = float(t2.item()) / steps
    e2e = {"value": S / (e2e_ms * 1e-3), "unit": "split-scores/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": h2d_bytes * world, "d2h_bytes_per_step": S * 8,
           "ms_steps_rank0": [round(x, 3) for x in e2e_steps], "clocks": clocks2, "call": call_name,
           "input": "2-bit bit planes + validity mask (batch.pack_planes_host), pinned" if method == "subflattening"
                    else "uint8 code matrix [taxa, sites], pinned"}

    # ---- roofline of the dominant kernel, from the CUDA-event spans of the timed steps ----
    peaks = ctx["peaks"]
    hbm = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s"
    roof = None
    R = 4 ** (n // 2)
    gram_key = f"gram_i32_r{R}"  # span of the int32 tensor-core Gram launches of the balanced splits (engine.CountScorer)
    if method == "flattening" and gram_key in phases:
        ms_tot, launches_timed, mats = phases[gram_key]
        ms = ms_tot / max(mats, 1)
        ops_alg = 2.0 * R ** 3                       # SURVEY 8(d): 2 R^2 C per balanced split (GEMM convention)
        blocks = R // 256
        exec_frac = (blocks * (blocks + 1) / 2) / (blocks * blocks)  # 256 x 256 blocks touching the upper triangle
        ops_exec = ops_alg * exec_frac
        i8 = ctx.get("int8_peak")
        bf16 = peaks.get("bf16_tflops") or 1590.0
        peak = i8["burst"] if i8 else 2 * bf16
        traffic, traffic_note = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_gram_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_note = tj.get("dram_bytes_per_matrix"), tj.get("note")
        roof = {"kernel": f"gram_u8 tcgen05 kernel (kind::i8), {R}x{R}x{R} per balanced split, int32 epilogue", "bound": "tensor",
                "achieved": ops_exec / (ms * 1e-3) / 1e12, "peak": peak, "unit": "TOP/s",
                "frac": ops_exec / (ms * 1e-3) / 1e12 / peak,
                "peak_source": (i8["how"] + " (burst; measured in this run)") if i8 else "2 x MEASURED_PEAKS.json bf16 burst (int8 GEMM measurement failed)",
                "peak_sustained": i8["sustained"] if i8 else None,
                "frac_of_sustained": (ops_exec / (ms * 1e-3) / 1e12 / i8["sustained"]) if i8 else None,
                "ops_counted": "EXECUTED MMAs only: the kernel computes the 256x256 blocks touching the upper triangle "
                               f"({exec_frac:.4f} of the full product) and mirrors the rest",
                "achieved_algorithmic": ops_alg / (ms * 1e-3) / 1e12, "algorithmic_ops_per_matrix": ops_alg,
                "ms_per_matrix": ms, "launches_timed": launches_timed, "matrices_timed": mats,
                "matrices_per_launch": mats / max(launches_timed, 1),
                "share_of_step": ms_tot / max(sum(step_ms), 1e-9),
                "concurrent_streams": int(os.environ.get("SPB_SCORE_STREAMS", "1")),
                "traffic": traffic, "traffic_note": traffic_note or "dram bytes per matrix from the ncu --set full capture: see profiles/"}
    elif method == "thin" and "count" in phases:
        ms = phases["count"][0] / max(phases["count"][1], 1)
        nbytes = (se - sb) * 16.0 + (se - sb) / 8.0  # one 128-bit key per site (= N n / 4 at 64 taxa) + validity mask
        roof = {"kernel": "count_wide_kernel (+ table setup, compaction and merge when sharded)", "bound": "hbm",
                "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / hbm,
                "traffic": None, "peak_source": hbm_src, "launch_ms": ms,
                "note": "random 16-byte CAS + 4-byte atomic per distinct pattern: DRAM-transaction bound, not streaming bound"}
    elif method == "subflattening" and "pairs" in phases:
        ms = phases["pairs"][0] / max(phases["pairs"][1], 1)
        nbytes = (se - sb) * n / 4.0 + (se - sb) / 8.0  # SURVEY 8(d): N n / 4 (+ N / 8 validity mask)
        roof = {"kernel": "pair_kernel (bit-plane AND + POPC pair statistics)", "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9,
                "peak": hbm, "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "traffic": None, "peak_source": hbm_src,
                "launch_ms": ms, "share_of_step": phases["pairs"][0] / max(sum(step_ms), 1e-9),
                "note": "pair_kernel is the only HBM-streaming kernel of this workload; the step is dominated by the batched "
                        "score kernel (instruction-issue bound, no HBM roofline): its throughput is `value`"}
    count_roof = None
    if method == "flattening" and "count" in phases:
        ms = phases["count"][0] / max(phases["count"][1], 1)
        nbytes = (se - sb) * n / 4.0 + (se - sb) / 8.0
        count_roof = {"kernel": "count stage: count_class_kernel + compaction" + (" + list exchange" if world > 1 and not replicated else ""),
                      "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                      "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "stage_ms": ms,
                      "note": "stage time includes the 64 MB table memset + compaction; kernel-only figures: profiles/r2_count_*"}

    if rank != 0:
        return None
    if rank_busy_ms is not None:
        phase_ms["rank_busy_ms"] = rank_busy_ms
    partition = None
    if method == "flattening" and world > 1 and getattr(scorer, "_cls", None) is not None:
        partition = {"kind": "contiguous runs of the size-class-ordered split list, cut at equal modelled cost; costs re-fitted once "
                             "from the per-rank device times of warm-up step 2 (distributed.refit_costs)",
                     "class_cost_us": {str(a): round(v, 2) for a, v in sorted(scorer._per.items())},
                     "splits_per_rank": [{str(a): c for a, c in sorted(h.items())} for h in scorer._held],
                     "refit_rank_times_us": [round(x, 1) for x in scorer.rank_times_us] if scorer.rank_times_us else None}
    out = {"metric": "split_scores_per_sec", "value": value, "unit": "split-scores/s", "n_gpus": world, "steps": steps,
           "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": {"flattening": "u8", "thin": "u128"}.get(method, "f64"), "data": "synthetic",
           "config": config_of(name, wl, S, world),
           "sites_per_sec": (N / (phases["count"][0] / phases["count"][1] * 1e-3)) if "count" in phases else N / (ms_per_step * 1e-3),
           "wall_s_timed_region": t_wall, "ms_steps_rank0": [round(x, 3) for x in step_ms], "phase_ms": phase_ms,
           "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof}
    if count_roof:
        out["roofline_count"] = count_roof
    if args.dump_outputs:
        np.save(os.path.join(args.dump_outputs, f"{name}_scores.npy"), sc.astype(np.float64, copy=False))
        out["dumped"] = f"{name}_scores.npy"
    checks = {"finite": bool(np.isfinite(sc).all()), "host_equals_device": bool(np.array_equal(sc, host_scores.numpy()))}
    if partition is not None:
        out["partition"] = partition
    if cpu_baseline and world == 1 and not args.no_cpu_baseline:
        if method == "flattening":
            cb, ref_scores = cpu_flattening_sample(name, wl, codes_np, idx_all, budget_s=25.0)
            errs = {s: abs(sc[s] - r) / abs(r) for s, r in ref_scores.items() if r}
            tol = {s: max(1e-9, 64 * np.finfo(float).eps / (r * r)) for s, r in ref_scores.items() if r}
            checks["max_rel_err_vs_oracle"] = max(errs.values()) if errs else None
            checks["oracle_kind"] = cb["kind"]
            checks["splits_checked"] = len(errs)
            checks["within_tolerance"] = bool(all(errs[s] <= tol[s] for s in errs))
        else:
            cb = cpu_port_sample(name, wl, codes_dev.cpu().numpy()[:, :1_000_000], idx_all, budget_s=10.0)
        out["cpu_baseline"] = cb
    elif world > 1:
        out["cpu_baseline"] = None
    out["checks"] = checks
    return out


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    import splitp_b200 as sp
    from splitp_b200 import batch
    from splitp_b200 import distributed as spd
    eng = sp.engine
    rank, local, world = spd.init_from_env()
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
    dev = eng.device()
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    sampler = ClockSampler(local)
    sampler.start()  # NVML initialisation happens here, before any warm-up, so that it cannot disturb a timed step
    ctx = {"torch": torch, "dist": dist, "sp": sp, "spd": spd, "eng": eng, "batch": batch, "rank": rank, "local": local,
           "world": world, "dev": dev, "peaks": peaks, "sampler": sampler,
           "flush": torch.empty(256 << 20, dtype=torch.uint8, device=dev)}  # > 126 MB L2
    name = args.workload
    wl = dict(WORKLOADS[name])
    if args.sites:
        wl["sites"] = args.sites
    if wl["method"] == "flattening":
        ctx["int8_peak"] = measure_int8_peak(torch)
    out = gpu_workload(name, wl, args, ctx, args.steps, max(args.warmup, 3), args.max_splits)
    extras = args.extras
    if extras is None:
        extras = "c3,c5,c4" if (name == "c2" and not args.sites and not args.max_splits) else "none"
    results = {}
    for ex in [e for e in extras.split(",") if e and e != "none"]:
        wl_x = dict(WORKLOADS[ex])
        t0 = time.perf_counter()
        try:
            r = gpu_workload(ex, wl_x, args, ctx, steps=args.steps, warmup=3, max_splits=EXTRA_SPLIT_CAP.get(ex),
                             cpu_baseline=(ex != "c4"))
        except Exception as exc:  # noqa: BLE001  (an extra workload must never take the headline line down with it)
            r = {"error": f"{type(exc).__name__}: {exc}"} if rank == 0 else None
            if r is not None and args.dump_outputs:
                r["dumped"] = None  # no DIR/<name>_scores.npy for a workload that failed
        torch.cuda.empty_cache()
        if rank == 0 and r is not None:
            r["bench_wall_s"] = round(time.perf_counter() - t0, 2)
            results[ex] = r
    sampler.close()
    if rank == 0:
        if results:
            out["workloads"] = results
        emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
