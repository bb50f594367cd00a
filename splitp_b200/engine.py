"""Device-side engine behind the drop-in functions.

Everything here drives the C-ABI library (`include/splitp_b200.h`) with torch tensors used purely
as device buffers (`tensor.data_ptr()`), on the current torch CUDA stream.  There is no CPU
fallback: without a CUDA device or without the built library every entry point raises.

Objects
  DeviceAlignment  2-bit packed alignment (site-major bit stream + taxon-major bit planes + validity)
  PatternTable     compressed site patterns: keys (base-4 number of the pattern, taxon 0 most
                   significant, as `__index_of`, splitp/constructions.py:166-171) with integer
                   counts (from an alignment) or float64 values (from a {pattern: value} mapping)
  PairTables       4x4 joint tables of every taxon pair and their Hadamard-type transform: all a
                   subflattening needs (SURVEY.md section 0)
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import threading
import warnings

import numpy as np
import torch

from . import _lib
from ._lib import SPB_S0_K4MAJOR, SPB_S0_ROWMAJOR, SPB_S0_TILED, SPB_U8_NO_MEMSET, SPB_VAL_F64, SPB_VAL_U32, call, lib, make_split

STATES = "ACGT"
_UPPER_LUT = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(STATES):
    _UPPER_LUT[ord(_c)] = _i
DIRECT_MAX_TAXA = 12   # direct-indexed count table up to 4^12 cells (64 MB); hash table above
JACOBI_MAX_K = 128
SUBFLATTEN_TABLES_MAX_TAXA = 43  # triple-table subflattening scorer: k = 3 floor(n / 2) + 1 <= 64
SCORE_INFO = 10        # doubles per matrix in the block-Krylov status record (SPB_SCORE_INFO)


# --------------------------------------------------------------------------------------------
# plumbing
# --------------------------------------------------------------------------------------------
def device():
    if not torch.cuda.is_available():
        raise RuntimeError("splitp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _zeros(shape, dtype):
    return torch.zeros(shape, dtype=dtype, device=device())


def _empty(shape, dtype):
    return torch.empty(shape, dtype=dtype, device=device())


class PhaseTimer:
    """Per-phase device time from CUDA events on the launch stream (bench.py `phase_ms`).  Inactive unless an instance
    is handed to the scorers; recording an event pair costs a few microseconds of host time."""

    def __init__(self, only=None):
        """only: names of the spans to record (None = all).  A step of the 12-taxon workload has ~130 spans; recording all of
        them costs 0.8 ms of a 47 ms step, so a benchmark times its steps with the ONE span it needs and takes the full
        breakdown from separate passes."""
        self.events, self.extra = [], []
        self.only = None if only is None else frozenset(only)

    @contextlib.contextmanager
    def span(self, name, units=1):
        if self.only is not None and name not in self.only:
            yield
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        try:
            yield
        finally:
            b.record()
            self.events.append((name, a, b, units))

    def add(self, name, ms, units=1):
        """A span measured elsewhere (the C library's own CUDA events)."""
        self.extra.append((name, float(ms), units))

    def totals(self):
        """{phase: (ms, spans, units)}; call after a synchronize."""
        out = {}
        for name, a, b, units in self.events:
            ms, n, u = out.get(name, (0.0, 0, 0))
            out[name] = (ms + a.elapsed_time(b), n + 1, u + units)
        for name, ms_x, units in self.extra:
            ms, n, u = out.get(name, (0.0, 0, 0))
            out[name] = (ms + ms_x, n + 1, u + units)
        return out

    def clear(self):
        self.events, self.extra = [], []


_NULL_SPAN = contextlib.nullcontext()


def _span(timer, name, units=1):
    return timer.span(name, units) if timer is not None else _NULL_SPAN


def split_positions(split, taxa):
    """Taxon labels of both sides -> positions in `taxa` (order kept: it is the digit significance)."""
    indexer = {t: i for i, t in enumerate(taxa)}
    return [indexer[s] for s in split[0]], [indexer[s] for s in split[1]]


def covers_all(n, idx_a, idx_b):
    return len(idx_a) + len(idx_b) == n and set(idx_a) | set(idx_b) == set(range(n))


# --------------------------------------------------------------------------------------------
# alignment packing (SURVEY section 8 row f1; validity rule of splitp/parsers/fasta.py:54-57)
# --------------------------------------------------------------------------------------------
class DeviceAlignment:
    def __init__(self, n, N, sm, planes, valid, taxa=None):
        self.n, self.N, self.sm, self.planes, self.valid = n, N, sm, planes, valid
        self.taxa = tuple(taxa) if taxa is not None else None
        self.plane_words = int(lib.spb_plane_words(N))


def pack(chars, is_ascii=False, taxa=None, want_sm=True, want_planes=True):
    """chars: uint8 [n, N] (torch tensor on the device, or anything np.asarray accepts on the host).
    is_ascii: bytes are characters (ACGTacgt valid) rather than codes 0..3."""
    if not isinstance(chars, torch.Tensor):
        host = torch.from_numpy(np.ascontiguousarray(np.asarray(chars, dtype=np.uint8)))
        chars = host.to(device(), non_blocking=False)
    if chars.dtype != torch.uint8 or chars.dim() != 2:
        raise ValueError("pack: expected a uint8 [n_taxa, n_sites] array")
    chars = chars.contiguous()
    n, N = int(chars.shape[0]), int(chars.shape[1])
    Wp = int(lib.spb_plane_words(N))
    sm = _empty(int(lib.spb_sm_words(n, N)), torch.int32) if (want_sm and n <= 32) else None
    planes = _empty((n, 2, Wp), torch.int32) if want_planes else None
    valid = _zeros(Wp, torch.int32)
    if N > 0:
        call("spb_pack", _p(chars), n, N, N, int(bool(is_ascii)), _p(sm), _p(planes), _p(valid), _st())
    return DeviceAlignment(n, N, sm, planes, valid, taxa)


# --------------------------------------------------------------------------------------------
# pattern tables
# --------------------------------------------------------------------------------------------
class PatternTable:
    def __init__(self, n, keys, counts=None, values=None, divisor=0.0, first=None, taxa=None):
        self.n, self.keys, self.counts, self.values = n, keys, counts, values
        self.divisor = float(divisor)  # counts / divisor = probabilities (fasta.py:66-70); 0 = leave counts
        self.first, self.taxa = first, (tuple(taxa) if taxa is not None else None)
        self.integral = False  # values came from Python ints: dict round trips give ints back (alignment.py:26-30 adds ints)

    @property
    def num(self):
        return int(self.keys.shape[0])

    def val_args(self, as_counts=False):
        """(pointer, kind, divisor) triple of the flattening entry points."""
        if self.counts is not None:
            return _p(self.counts), SPB_VAL_U32, 0.0 if as_counts else self.divisor
        return _p(self.values), SPB_VAL_F64, 0.0

    def values_f64(self):
        if self.values is not None:
            return self.values
        v = self.counts.to(torch.float64)
        if self.divisor <= 0:
            return v
        # tensor / tensor: one correctly rounded IEEE division per pattern, as fasta.py:66-70 (dividing by a python
        # scalar would be turned into a multiplication by the reciprocal, which is 1 ulp off for some counts)
        return torch.div(v, torch.full_like(v, self.divisor))


def count_patterns(aln, site_begin=0, site_end=None, want_first=False, force_hash=False, sort=True, reduce_fn=None, gather_fn=None):
    """Kernel 1: {pattern: count} of the usable sites in [site_begin, site_end)
    (splitp/parsers/fasta.py:48-63).  Keys come back ascending (= lexicographic A<C<G<T order of
    splitp/simulation.py:50-54); `first` holds the first site of each pattern (dict insertion order).
    Multi-GPU hooks for the direct table (n <= 12): reduce_fn(tensor, op) allreduces the whole table before compaction
    (needed with want_first); gather_fn(keys, counts) -> (all keys, all counts) exchanges the COMPACTED per-rank lists instead
    (a few hundred KB instead of 64 MB at 12 taxa) and the lists are merged into a fresh table."""
    n = aln.n
    if aln.sm is None:
        raise NotImplementedError("pattern counting uses uint64 keys: at most 31 taxa (site-major stream <= 32)")
    if n > 31:
        raise NotImplementedError("pattern counting uses uint64 keys: at most 31 taxa")
    site_end = aln.N if site_end is None else site_end
    nsites = max(0, site_end - site_begin)
    if aln.N == 0 and reduce_fn is None:  # nothing to count (and no buffers to hand to the kernels)
        return PatternTable(n, _empty(0, torch.int64), counts=_empty(0, torch.int32), divisor=0.0,
                            first=_empty(0, torch.int32) if want_first else None, taxa=aln.taxa)
    usable = _zeros(1, torch.int64)
    num = _zeros(1, torch.int64)
    if n <= DIRECT_MAX_TAXA and not force_hash:
        cells = 4 ** n
        table = _zeros(cells, torch.int32)
        first = torch.full((cells,), -1, dtype=torch.int32, device=device()) if want_first else None
        call("spb_count_direct", _p(aln.sm), _p(aln.valid), n, site_begin, site_end, _p(table), _p(first), _p(usable), _st())
        if reduce_fn is not None:
            reduce_fn(table, "sum")
            reduce_fn(usable, "sum")
            if first is not None:
                reduce_fn(first, "min_u32")
        cap = min(cells, max(nsites, 1)) if reduce_fn is None else cells
        tmp = _empty(int(lib.spb_compact_tmp_words(cells)), torch.int32)
        keys, counts = _empty(cap, torch.int64), _empty(cap, torch.int32)
        fo = _empty(cap, torch.int32) if want_first else None
        call("spb_compact_direct", _p(table), _p(first), cells, _p(keys), _p(counts), _p(fo), cap, _p(num), _p(tmp), _st())
        P = int(num.item())
        keys, counts = keys[:P], counts[:P]
        fo = fo[:P] if fo is not None else None
        if gather_fn is not None:
            if want_first or reduce_fn is not None:
                raise ValueError("count_patterns: gather_fn excludes reduce_fn / want_first")
            all_keys, all_counts = gather_fn(keys, counts)
            table.zero_()
            total = int(all_keys.shape[0])
            call("spb_direct_merge", _p(all_keys.contiguous()), _p(all_counts.contiguous()), total, cells, _p(table), _st())
            cap = min(cells, max(total, 1))
            keys, counts = _empty(cap, torch.int64), _empty(cap, torch.int32)
            call("spb_compact_direct", _p(table), None, cells, _p(keys), _p(counts), None, cap, _p(num), _p(tmp), _st())
            P = int(num.item())
            keys, counts = keys[:P], counts[:P]
            usable = counts.to(torch.int64).sum().reshape(1)  # every usable site of every rank is in exactly one pattern
    else:
        cap = 1024
        while cap < 2 * min(4 ** n, max(nsites, 1)):
            cap *= 2
        hk = torch.full((cap,), -1, dtype=torch.int64, device=device())
        hc = _zeros(cap, torch.int32)
        hf = torch.full((cap,), -1, dtype=torch.int32, device=device()) if want_first else None
        ovf = _zeros(1, torch.int32)
        call("spb_count_hash", _p(aln.sm), _p(aln.valid), n, site_begin, site_end, _p(hk), _p(hc), _p(hf), cap, _p(usable),
             _p(ovf), _st())
        outcap = min(cap, max(nsites, 1))
        tmp = _empty(int(lib.spb_compact_tmp_words(cap)), torch.int32)
        keys, counts = _empty(outcap, torch.int64), _empty(outcap, torch.int32)
        fo = _empty(outcap, torch.int32) if want_first else None
        call("spb_compact_hash", _p(hk), _p(hc), _p(hf), cap, _p(keys), _p(counts), _p(fo), outcap, _p(num), _p(tmp), _st())
        if int(ovf.item()):
            raise MemoryError("splitp_b200: pattern hash table overflow")
        P = int(num.item())
        keys, counts = keys[:P], counts[:P]
        fo = fo[:P] if fo is not None else None
        if reduce_fn is not None:
            raise NotImplementedError("hashed tables are merged by distributed.count_patterns_sharded, not by an allreduce")
        if sort and P > 1:
            keys, perm = torch.sort(keys)  # keys < 2^62: signed order = unsigned order
            counts = counts[perm]
            fo = fo[perm] if fo is not None else None
    return PatternTable(n, keys, counts=counts, divisor=float(int(usable.item())), first=fo, taxa=aln.taxa)


def merge_tables(n, keys, counts, first=None, sort=True):
    """Sums the counts of equal keys of a concatenated (key, count) list: the merge step of the sharded
    hashed counting (one spb_hash_merge pass into a fresh open-addressing table, then compaction)."""
    total = int(keys.shape[0])
    cap = 1024
    while cap < 2 * max(total, 1):
        cap *= 2
    hk = torch.full((cap,), -1, dtype=torch.int64, device=device())
    hc = _zeros(cap, torch.int32)
    hf = torch.full((cap,), -1, dtype=torch.int32, device=device()) if first is not None else None
    ovf, num = _zeros(1, torch.int32), _zeros(1, torch.int64)
    call("spb_hash_merge", _p(keys.contiguous()), _p(counts.contiguous()), _p(first), total, _p(hk), _p(hc), _p(hf), cap, _p(ovf), _st())
    outcap = max(total, 1)
    tmp = _empty(int(lib.spb_compact_tmp_words(cap)), torch.int32)
    ok, oc = _empty(outcap, torch.int64), _empty(outcap, torch.int32)
    of = _empty(outcap, torch.int32) if first is not None else None
    call("spb_compact_hash", _p(hk), _p(hc), _p(hf), cap, _p(ok), _p(oc), _p(of), outcap, _p(num), _p(tmp), _st())
    if int(ovf.item()):
        raise MemoryError("splitp_b200: pattern hash table overflow")
    P = int(num.item())
    ok, oc = ok[:P], oc[:P]
    of = of[:P] if of is not None else None
    if sort and P > 1:
        ok, perm = torch.sort(ok)
        oc = oc[perm]
        of = of[perm] if of is not None else None
    return PatternTable(n, ok, counts=oc, first=of)


NARROW_MAX_TAXA = 31  # uint64 pattern keys
WIDE_MAX_TAXA = 64    # 128-bit pattern keys {lo, hi}


def _base4(codes):
    """uint8 codes [P, m], m <= 32 -> uint64 base-4 numbers, first column most significant."""
    m = codes.shape[1]
    weights = np.uint64(4) ** np.arange(m - 1, -1, -1, dtype=np.uint64)
    return (codes.astype(np.uint64) * weights).sum(axis=1, dtype=np.uint64)


def encode_patterns(patterns):
    """list of equal-length ACGT strings -> (keys, n): uint64 [P] up to 31 taxa, uint64 [P, 2] = {lo, hi} for 32..64 taxa
    (the 128-bit key of csrc/wide.cu: lo holds the last 32 digits).  Any other character raises KeyError exactly like
    `__index_of` (constructions.py:166-171) does."""
    P = len(patterns)
    if P == 0:
        return np.zeros(0, dtype=np.uint64), 0
    n = len(patterns[0])
    joined = "".join(patterns)
    if len(joined) != P * n:
        raise KeyError("patterns of unequal length")
    if n > WIDE_MAX_TAXA:
        raise NotImplementedError(f"pattern keys are at most 128 bits: at most {WIDE_MAX_TAXA} taxa (got {n})")
    raw = np.frombuffer(joined.encode("latin-1", errors="replace"), dtype=np.uint8).reshape(P, n)
    codes = _UPPER_LUT[raw]
    bad = np.argwhere(codes > 3)
    if len(bad):
        raise KeyError(chr(raw[bad[0][0], bad[0][1]]))
    if n <= NARROW_MAX_TAXA:
        return _base4(codes), n
    keys = np.empty((P, 2), dtype=np.uint64)
    keys[:, 0] = _base4(codes[:, n - 32:])
    keys[:, 1] = _base4(codes[:, :n - 32])
    return keys, n


def decode_keys(keys, n):
    """uint64 keys [P] (or 128-bit keys [P, 2] = {lo, hi}) -> list of pattern strings."""
    keys = np.asarray(keys, dtype=np.uint64)
    if len(keys) == 0:
        return []
    shifts = (2 * np.arange(n - 1, -1, -1)).astype(np.uint64)
    if keys.ndim == 2:  # digit j sits in lo (keys[:, 0]) for the last 32 positions, in hi above
        word = np.where(shifts >= 64, 1, 0)
        codes = ((keys[:, word] >> (shifts % np.uint64(64))[None, :]) & np.uint64(3)).astype(np.uint8)
    else:
        codes = ((keys[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)
    chars = np.frombuffer(STATES.encode(), dtype=np.uint8)[codes]
    flat = chars.tobytes().decode("ascii")
    return [flat[i * n:(i + 1) * n] for i in range(len(keys))]


class WidePatternTable:
    """A {pattern: value} mapping of 32..64 taxa on the device: keys int64 [P, 2] = {lo, hi} (the 128-bit key of
    csrc/wide.cu and `WideTable.compact`), values float64 [P], both in mapping order."""

    counts = None
    divisor = 0.0

    def __init__(self, n, keys, values, taxa=None):
        self.n, self.keys, self.values = n, keys, values
        self.taxa = tuple(taxa) if taxa is not None else None
        self.integral = False  # as PatternTable.integral

    @property
    def num(self):
        return int(self.keys.shape[0])

    def values_f64(self):
        return self.values


def _narrow_only(table, what):
    """The kernels behind `what` read uint64 pattern keys."""
    if isinstance(table, WidePatternTable):
        raise NotImplementedError(f"{what} is limited to {NARROW_MAX_TAXA} taxa (uint64 pattern keys); this table has {table.n}")


_TABLE_CACHE = {}


def table_from_mapping(mapping):
    """{pattern: value} mapping (plain dict or Alignment) -> PatternTable (up to 31 taxa) or WidePatternTable (32..64 taxa)
    with float64 values, in the mapping's iteration order.  A one-entry-per-object cache avoids re-uploading an unchanged
    mapping (validated against the joined keys and the values, so a mutated mapping is re-encoded)."""
    if isinstance(mapping, (PatternTable, WidePatternTable)):
        return mapping
    pats = list(mapping.keys())
    raw = list(mapping.values())
    try:  # ints / floats / numpy scalars convert at C speed (this validation runs on EVERY drop-in call: README loop, config 1)
        vals = np.fromiter(raw, dtype=np.float64, count=len(pats))
    except (TypeError, ValueError):
        vals = np.fromiter((float(v) for v in raw), dtype=np.float64, count=len(pats))
    integral = bool(raw) and all(type(v) is int and abs(v) < (1 << 53) for v in raw)
    joined = "".join(pats)
    hit = _TABLE_CACHE.get(id(mapping))
    if hit is not None and hit[0] == joined and hit[1].shape == vals.shape and np.array_equal(hit[1], vals, equal_nan=True):
        table = hit[2]
    else:
        keys, n = encode_patterns(pats)
        dev = device()
        keys_d, vals_d = torch.from_numpy(keys.view(np.int64)).to(dev), torch.from_numpy(vals).to(dev)
        table = WidePatternTable(n, keys_d, vals_d) if keys.ndim == 2 else PatternTable(n, keys_d, values=vals_d)
        if len(_TABLE_CACHE) > 16:
            _TABLE_CACHE.clear()
        _TABLE_CACHE[id(mapping)] = (joined, vals, table)
    table.integral = integral
    table.taxa = tuple(mapping.taxa) if hasattr(mapping, "taxa") else None
    return table


def table_to_dict(table, as_counts=False):
    keys = table.keys.cpu().numpy().view(np.uint64)
    pats = decode_keys(keys, table.n)
    if table.counts is not None:
        cnt = table.counts.cpu().numpy().view(np.uint32)
        if as_counts or table.divisor <= 0:
            return {p: int(c) for p, c in zip(pats, cnt)}
        return {p: int(c) / table.divisor for p, c in zip(pats, cnt)}  # one IEEE division, fasta.py:66-70
    vals = table.values.cpu().numpy()
    if table.integral:  # sums of ints below 2^53 are exact in float64: hand ints back like the reference's dict arithmetic
        return {p: int(v) for p, v in zip(pats, vals)}
    return dict(zip(pats, vals.tolist()))


# --------------------------------------------------------------------------------------------
# flattenings (kernel 2)
# --------------------------------------------------------------------------------------------
def project_keys(table, idx):
    """Digits of the taxon positions `idx` (in that order, first most significant) of every key of a WidePatternTable:
    int64 [P] for up to 31 positions, 128-bit keys int64 [P, 2] = {lo, hi} for more."""
    m = len(idx)
    out = _empty((table.num, 2) if m > NARROW_MAX_TAXA else table.num, torch.int64)
    call("spb_project_wide", _p(table.keys), table.num, table.n, bytes(idx), m, _p(out), _st())
    return out


def flatten_coo(table, idx_a, idx_b):
    """(rows, cols) int64 of every pattern: the triplets behind FlatFormat.sparse (constructions.py:86-102)."""
    if isinstance(table, WidePatternTable):
        if max(len(idx_a), len(idx_b)) > NARROW_MAX_TAXA:
            raise NotImplementedError(f"flattening: a side of {max(len(idx_a), len(idx_b))} taxa has 4^side row or column indices, "
                                      f"which do not fit in 64 bits (sides are limited to {NARROW_MAX_TAXA} taxa)")
        return project_keys(table, idx_a), project_keys(table, idx_b)
    sp = make_split(table.n, idx_a, idx_b)
    rows, cols = _empty(table.num, torch.int64), _empty(table.num, torch.int64)
    call("spb_flatten_coo", _p(table.keys), table.num, C.byref(sp), _p(rows), _p(cols), _st())
    return rows, cols


def flatten_dense(table, idx_a, idx_b, as_counts=False):
    a, b = len(idx_a), len(idx_b)
    if isinstance(table, WidePatternTable):  # rows / columns from the projection kernel, placed as in _flatten_reduced_large
        rows, cols = flatten_coo(table, idx_a, idx_b)
        out = _zeros((4 ** a, 4 ** b), torch.float64)
        _place(out, rows, cols, table.values, covers_all(table.n, idx_a, idx_b))
        return out
    sp = make_split(table.n, idx_a, idx_b)
    out = _empty((4 ** a, 4 ** b), torch.float64)
    win = None if covers_all(table.n, idx_a, idx_b) else _empty(4 ** (a + b), torch.int32)
    vp, kind, div = table.val_args(as_counts)
    call("spb_flatten_dense_w", _p(table.keys), vp, kind, div, table.num, C.byref(sp), _p(out), _p(win), _st())
    return out


def reduced_plan(table, idx_a, idx_b):
    _narrow_only(table, "the reduced-flattening plan")
    a, b = len(idx_a), len(idx_b)
    sp = make_split(table.n, idx_a, idx_b)
    rank_r, rank_c = _empty(4 ** a + 1, torch.int32), _empty(4 ** b + 1, torch.int32)
    tmp = _empty(int(lib.spb_compact_tmp_words(max(4 ** a, 4 ** b) + 1)), torch.int32)
    shape = (C.c_int64 * 2)()
    call("spb_flatten_reduced_plan", _p(table.keys), table.num, C.byref(sp), _p(rank_r), _p(rank_c), _p(tmp), shape, _st())
    return sp, rank_r, rank_c, int(shape[0]), int(shape[1])


def flatten_reduced(table, idx_a, idx_b, as_counts=False):
    """constructions.py:31-55: all-zero rows / columns dropped, rows and columns in ascending index order."""
    if max(len(idx_a), len(idx_b)) > 13 or isinstance(table, WidePatternTable):
        return _flatten_reduced_large(table, idx_a, idx_b, as_counts)
    sp, rank_r, rank_c, R, Cc = reduced_plan(table, idx_a, idx_b)
    out = _empty((R, Cc), torch.float64)
    if R == 0 or Cc == 0:
        return out
    win = None if covers_all(table.n, idx_a, idx_b) else _empty(R * Cc, torch.int32)
    vp, kind, div = table.val_args(as_counts)
    call("spb_flatten_reduced_fill_w", _p(table.keys), vp, kind, div, table.num, C.byref(sp), _p(rank_r), _p(rank_c), R, Cc,
         _p(out), _p(win), _st())
    return out


def _flatten_reduced_large(table, idx_a, idx_b, as_counts):
    # sides above 13 taxa (and tables with 128-bit keys): the used-index flag arrays (4^side cells) no longer fit, so the
    # ranks come from a sort-unique of the per-pattern indices (torch.unique: library sort, documented in DESIGN.md)
    if max(len(idx_a), len(idx_b)) > 31 and not isinstance(table, WidePatternTable):
        raise NotImplementedError("reduced flattening: sides are limited to 31 taxa (int64 indices)")
    rows, cols = flatten_coo(table, idx_a, idx_b)
    ur, ri = torch.unique(rows, return_inverse=True)
    uc, ci = torch.unique(cols, return_inverse=True)
    out = _zeros((len(ur), len(uc)), torch.float64)
    vals = table.counts.to(torch.float64) if (as_counts and table.counts is not None) else table.values_f64()
    _place(out, ri, ci, vals, covers_all(table.n, idx_a, idx_b))
    return out


def _place(out, ri, ci, vals, covering):
    """out[ri, ci] = vals; where the split leaves taxa out several patterns share a cell and the last one in table order
    wins it (the reference's assignment, constructions.py:43,101)."""
    if not covering:
        cols = out.shape[1]
        cell = ri * cols + ci
        order = torch.arange(cell.shape[0], device=cell.device)
        last = torch.zeros(out.shape[0] * cols, dtype=torch.int64, device=cell.device).scatter_reduce_(0, cell, order, "amax")
        keep = last[cell] == order
        ri, ci, vals = ri[keep], ci[keep], vals[keep]
    out[ri, ci] = vals


# --------------------------------------------------------------------------------------------
# scores (kernels 4 and 5)
# --------------------------------------------------------------------------------------------
def gram_f64(A):
    """G = A A^T, A float64 [batch, R, C] (or [R, C]) -> [batch, R, R]."""
    if A.dim() == 2:
        A = A.unsqueeze(0)
    A = A.contiguous()
    batch, R, Cc = (int(x) for x in A.shape)
    G = _empty((batch, R, R), torch.float64)
    ws_elems = int(lib.spb_gram_f64_ws(R, Cc, batch))
    ws = _empty(ws_elems, torch.float64) if ws_elems else None
    call("spb_gram_f64", _p(A), R, Cc, batch, _p(G), _p(ws), _st())
    return G


_KRYLOV_WS = {}


def _krylov_ws(k, batch):
    """Workspace of the block-Krylov solver, one per CUDA stream (size classes scored concurrently must not share it)."""
    need = int(lib.spb_score_gram_large_ws(k, batch))
    key = int(torch.cuda.current_stream().cuda_stream)
    ws = _KRYLOV_WS.get(key)
    if ws is None or ws.numel() < need or ws.device != device():
        ws = _KRYLOV_WS[key] = _empty(need, torch.float64)
    return ws


def score_gram(G, k=None, want_info=False):
    """Scores from symmetric PSD Gram matrices G [batch, ld, ld] using the leading k x k block.
    k <= 4 -> 0.0 (at most 4 singular values: 1 - top4/total vanishes, phylogenetics.py:293-300)."""
    if G.dim() == 2:
        G = G.unsqueeze(0)
    G = G.contiguous()
    batch, ld = int(G.shape[0]), int(G.shape[1])
    k = ld if k is None else int(k)
    scores = _empty(batch, torch.float64)
    info = None
    if k <= 4:
        scores.zero_()
        return (scores, None) if want_info else scores
    if k <= JACOBI_MAX_K:
        info = _empty((batch, k), torch.float64) if want_info else None
        call("spb_score_gram_small", _p(G), k, ld, batch, _p(scores), _p(info), _st())
    else:
        info = _solve_large(batch, scores,
                            lambda sel, sc, inf, ws, budget: call("spb_score_gram_large_n", _p(G if sel is None else G.index_select(0, sel)),
                                                                  k, ld, int(sc.shape[0]), _p(sc), _p(inf), _p(ws), budget, _st()), k)
        _warn_unconverged()
    return (scores, info) if want_info else scores


FIRST_CYCLES = 2   # cycles the WHOLE batch runs through (two blocks each); matrices still open after them are solved as their own batch
MIN_COMPACT = 16   # batches below this are not worth a second call


def _solve_large(batch, scores, run, k):
    """Block-Krylov scores of a batch with straggler compaction.  The solver keeps every matrix of a batch in the cycle until the
    last one is accepted, and its cycles grow (2, 2, 4, 4, 12, ... blocks of 8 vectors = that many G Q products per matrix): with
    up to 512 matrices per batch one slow matrix would cost hundreds of products.  So the whole batch gets FIRST_CYCLES cycles;
    whatever reports converged = 0 after them is gathered into a batch of its own and solved with the full budget.
    run(sel, scores, info, ws, budget): one solver call on the matrices `sel` (None = all).  Returns the info array [batch, 10]."""
    info = _empty((batch, SCORE_INFO), torch.float64)
    if batch < MIN_COMPACT:
        run(None, scores, info, _krylov_ws(k, batch), 40)
        return info
    run(None, scores, info, _krylov_ws(k, batch), FIRST_CYCLES)
    if int(lib.spb_score_last_unconverged()) == 0:
        return info
    sel = torch.nonzero(info[:, 8] == 0.0).flatten()
    m = int(sel.shape[0])
    sc2, inf2 = _empty(m, torch.float64), _empty((m, SCORE_INFO), torch.float64)
    run(sel, sc2, inf2, _krylov_ws(k, m), 40)
    scores.index_copy_(0, sel, sc2)
    info.index_copy_(0, sel, inf2)
    return info


def _warn_unconverged():
    """The block-Krylov solver keeps the last score of a matrix that exhausted its cycle budget; say so."""
    bad = int(lib.spb_score_last_unconverged())
    if bad:
        warnings.warn(f"splitp_b200: {bad} Gram matrices did not reach the 1e-11 acceptance bound of the block-Krylov "
                      "eigen-solver; their scores are the last iterates", RuntimeWarning, stacklevel=3)


def score_matrix(A):
    """split_score of a float64 device matrix [R, C] (or a batch [B, R, C]): Gram on the short side."""
    if A.dim() == 2:
        A = A.unsqueeze(0)
    if A.shape[1] > A.shape[2]:
        A = A.transpose(1, 2)
    if min(A.shape[1], A.shape[2]) == 0:
        return torch.full((A.shape[0],), float("nan"), dtype=torch.float64, device=A.device)
    return score_gram(gram_f64(A.contiguous()))


class CountScorer:
    """Exact-integer scoring of count flattenings: u8 low-byte matrix -> Gram on the tensor cores
    (tcgen05 kind::i8) or dp4a for <= 64 rows -> sparse high-part correction -> eigen-solver.
    Buffers are allocated once and reused across splits; up to SPB_MAX_BATCH splits share one launch of
    every stage (the scatter / correction kernels are a few microseconds each, so batching them is what
    keeps the GPU busy)."""

    NB = _lib.SPB_MAX_BATCH   # splits per scatter / clear launch (kernel-parameter limit); 16 in round 1: 266 launches per c2 step
    GNB = 64                  # matrices per Gram / correction launch: 20 tiles x 16 matrices leave the 148 persistent CTAs
                              # with 2 or 3 tiles each (72 % efficiency at 5|7 of 12 taxa), 64 matrices level that out

    def __init__(self, table, hi_cap=None):
        if table.counts is None:
            raise ValueError("CountScorer needs a PatternTable with integer counts")
        self._table = None
        self.hi_cap = int(hi_cap) if hi_cap is not None else 0
        # Size classes can be scored on up to NSTREAMS CUDA streams at once (one host thread per stream; buffers that a class
        # writes per launch exist once per stream slot).  Measured on B200 (12 taxa, 10^6 sites): 67.0 ms with two streams
        # against 66.5 ms with one, at N = 1 and N = 2 alike -- the big kernels already fill the SMs -- so the default is 1.
        self.nstreams = max(1, int(os.environ.get("SPB_SCORE_STREAMS", "1")))
        self._tl = threading.local()
        self._hi = {}
        self._side = None
        self.table = table
        self._s0 = {}
        self._G = {}
        self._Gi = {}
        self._ws = {}
        self._batch_bytes = None
        self._hi_ws = {}
        self._plans = {}       # (id(split list), taxa, class) -> encoded splits + output positions, see _encoded_group
        self.strip_from_table = os.environ.get("SPB_STRIP_KERNEL", "table") != "scan"  # A/B switch: column scans of S0 (round 1)
        self.int32_gram = True  # large dense splits keep G as int32 + correction strip (half the eigen-stage traffic)
        self.gram_hook = None  # optional wrapper (fn, nb) around the Gram launch
        self.timer = None      # optional PhaseTimer: scatter / gram / correction / eigen spans (bench.py phase_ms)

    @property
    def table(self):
        return self._table

    @table.setter
    def table(self, table):
        """The number of counts >= 256 is a property of the table (every split scatters the same patterns), so the
        high-part buffers are sized once per table: no per-split overflow tracking is needed."""
        self._table = table
        self.n_hi = int((table.counts.to(torch.int64) & 0xFFFFFFFF).ge(256).sum().item()) if table.num else 0
        if not self._hi or self.n_hi > self.hi_cap:
            self.hi_cap = max(self.hi_cap, 1024, 2 * self.n_hi)
            self._hi = {slot: (_empty((self.GNB, self.hi_cap, 2), torch.int32), _empty((self.GNB, self.hi_cap), torch.int32),
                               _zeros(self.GNB, torch.int32)) for slot in range(self.nstreams)}

    @property
    def _slot(self):
        return getattr(self._tl, "slot", 0)

    @property
    def hi_rc(self):
        return self._hi[self._slot][0]

    @property
    def hi_val(self):
        return self._hi[self._slot][1]

    @property
    def hi_num(self):
        return self._hi[self._slot][2]

    @staticmethod
    def geometry(rows, cols):
        """(layout, rows_pad, pitch) for a rows x cols count matrix with rows <= cols."""
        if rows <= 32:  # dp4a; above that the (zero-padded) 128-row tensor-core tile is faster than dp4a on 64 rows
            return SPB_S0_K4MAJOR, max((rows + 3) // 4 * 4, 4), (cols + 15) // 16 * 16
        rp = 128 if rows <= 128 else (rows + 255) // 256 * 256
        return SPB_S0_TILED, rp, (cols + 127) // 128 * 128

    def _gnb(self, rows_pad, pitch):
        """Matrices per Gram launch: GNB, fewer when one u8 matrix is large (the S0 batch stays within 4 GB)."""
        return int(max(16, min(self.GNB, (4 << 30) // (rows_pad * pitch))))

    def _buffers(self, layout, rows_pad, pitch, batch=1):
        key = (layout, rows_pad, pitch)
        if key not in self._s0:
            self._s0[key] = _zeros((self._gnb(rows_pad, pitch), rows_pad * pitch), torch.uint8)
        g = self._G.get(rows_pad)
        if g is None or g.shape[0] < batch:
            g = self._G[rows_pad] = _empty((batch, rows_pad, rows_pad), torch.float64)
        if key not in self._ws:
            n = int(lib.spb_gram_u8_ws(rows_pad, pitch, layout, 1))
            self._ws[key] = _empty(self._gnb(rows_pad, pitch) * rows_pad * rows_pad, torch.int64) if n else None
        return self._s0[key], g, self._ws[key]

    I32_MIN_ROWS = int(os.environ.get("SPB_I32_MIN_ROWS", "1024"))  # 1024: the 5|7 class of 12 taxa as well (round 1: 2048)
    I32_MAX_HI = 4096  # strip rows: the correction strip costs n_hi * rows_pad * 8 bytes per matrix and O(n_hi^2) work

    def _use_i32(self, layout, rows_pad, pitch):
        """int32 Gram + correction strip only while the strip stays small (a table with many counts >= 256, e.g.
        12 taxa from 10^8 sites, goes through the fp64 Gram, which has no such limit)."""
        return (self.int32_gram and layout == SPB_S0_TILED and rows_pad >= self.I32_MIN_ROWS and rows_pad % 256 == 0
                and pitch <= 32768 and self.n_hi <= self.I32_MAX_HI)

    def _buffers_i32(self, rows_pad, batch):
        """int32 Gram batch + correction strip (rows sized by the number of high counts of the table)."""
        cs_rows = max(self.n_hi, 1)
        b = self._Gi.get(rows_pad)
        if b is None or b["G"].shape[0] < batch or b["Cs"].shape[1] < cs_rows:
            b = self._Gi[rows_pad] = {
                "G": _empty((batch, rows_pad, rows_pad), torch.int32),
                "Cs": _empty((batch, cs_rows, rows_pad), torch.float64),
                "pos": _empty((batch, rows_pad), torch.int32),
                "hr": _empty((batch, cs_rows), torch.int32),
                "hm": _empty(batch, torch.int32),
            }
        return b

    def _strip_ws(self, pitch):
        """int32 scratch of spb_gram_hi_strip_batch_table for this thread's stream slot."""
        key = (getattr(self._tl, "slot", 0), int(pitch))
        ws = self._hi_ws.get(key)
        need = int(_lib.lib.spb_gram_hi_strip_table_ws(self.GNB, int(pitch), self.hi_cap))
        if ws is None or ws.numel() < need:
            ws = self._hi_ws[key] = _empty(need, torch.int32)
        return ws

    def _scatter(self, arr, nb, s0, layout, rows_pad, pitch, clear=False):
        """Scatter (or un-scatter) nb <= GNB splits into s0[0:nb], SPB_MAX_BATCH splits per launch."""
        t = self.table
        s0_stride, sz = rows_pad * pitch, C.sizeof(_lib.SpbSplit)
        for j in range(0, nb, self.NB):
            m = min(self.NB, nb - j)
            sub = (_lib.SpbSplit * m).from_buffer(arr, j * sz)
            if clear:
                call("spb_flatten_u8_clear_batch", _p(t.keys), t.num, sub, m, _p(s0[j:]), s0_stride, rows_pad, pitch, layout, _st())
            else:
                call("spb_flatten_u8_batch", _p(t.keys), _p(t.counts), t.num, sub, m, _p(s0[j:]), s0_stride, rows_pad, pitch, layout,
                     SPB_U8_NO_MEMSET, _p(self.hi_rc[j:]), _p(self.hi_val[j:]), _p(self.hi_num[j:]), self.hi_cap, _st())

    def _gram_batch_i32(self, splits, s0, buf, b0, layout, rows_pad, pitch):
        """As _gram_batch, into the int32 Gram + strip buffers at batch offset b0."""
        nb = len(splits)
        arr = splits if isinstance(splits, C.Array) else (_lib.SpbSplit * nb)(*splits)
        s0_stride, g_stride = rows_pad * pitch, rows_pad * rows_pad
        cs_rows = int(buf["Cs"].shape[1])
        G, Cs, pos, hr, hm = buf["G"][b0:], buf["Cs"][b0:], buf["pos"][b0:], buf["hr"][b0:], buf["hm"][b0:]
        t = self.timer
        try:
            with _span(t, "scatter", nb):
                self._scatter(arr, nb, s0, layout, rows_pad, pitch)
            run = lambda: call("spb_gram_u8_batch_i32", _p(s0), s0_stride, nb, rows_pad, pitch, _p(G), g_stride, _st())  # noqa: E731
            with _span(t, f"gram_i32_r{rows_pad}", nb):  # int32 tensor-core Gram, one span name per row count (bench.py roofline)
                run() if self.gram_hook is None else self.gram_hook(run, nb)
            with _span(t, "correction", nb):
                if self.strip_from_table and nb <= self.NB:
                    tb = self.table  # cross terms by a join of the pattern list with the high list (no column scans of S0)
                    call("spb_gram_hi_strip_batch_table", _p(tb.keys), _p(tb.counts), tb.num, arr, nb, rows_pad, pitch, _p(self.hi_rc),
                         _p(self.hi_val), _p(self.hi_num), self.hi_cap, _p(Cs), cs_rows, _p(pos), _p(hr), _p(hm),
                         _p(self._strip_ws(pitch)), _st())
                else:
                    call("spb_gram_hi_strip_batch", _p(s0), s0_stride, nb, rows_pad, pitch, layout, _p(self.hi_rc), _p(self.hi_val),
                         _p(self.hi_num), self.hi_cap, _p(Cs), cs_rows, _p(pos), _p(hr), _p(hm), _st())
            with _span(t, "scatter", 0):
                self._scatter(arr, nb, s0, layout, rows_pad, pitch, clear=True)
        except BaseException:
            self._drop_s0()  # the cached S0 buffers are assumed all-zero between uses: never keep a dirty one
            raise

    def _score_i32(self, buf, batch, k, want_info=False):
        rows_pad = int(buf["G"].shape[1])
        cs_rows = int(buf["Cs"].shape[1])
        scores = _empty(batch, torch.float64)

        def run(sel, sc, inf, ws, budget):
            if sel is None:
                G, Cs, pos, hr, hm = (buf[key] for key in ("G", "Cs", "pos", "hr", "hm"))
            else:  # the stragglers as a batch of their own (copies of their 32-bit Gram and strip: a few matrices)
                G, Cs, pos, hr, hm = (buf[key][:batch].index_select(0, sel) for key in ("G", "Cs", "pos", "hr", "hm"))
            call("spb_score_gram_large_i32_n", _p(G), k, rows_pad, int(sc.shape[0]), _p(Cs), cs_rows, _p(pos), _p(hr), _p(hm), _p(sc),
                 _p(inf), _p(ws), budget, _st())

        info = _solve_large(batch, scores, run, k)
        _warn_unconverged()
        return (scores, info) if want_info else scores

    def _drop_s0(self):
        self._s0.clear()

    def _plan(self, idx_a, idx_b, reduced):
        """Orient the split so that the Gram is taken on the short side; returns the launch geometry."""
        t = self.table
        if not covers_all(t.n, idx_a, idx_b):
            raise ValueError("CountScorer: the split must cover all taxa")
        rank_r = rank_c = None
        if reduced:
            sp, rank_r, rank_c, R, Cc = reduced_plan(t, idx_a, idx_b)
            if R > Cc:  # Gram on the short side: swap the roles of the two sides
                idx_a, idx_b, rank_r, rank_c, R, Cc = idx_b, idx_a, rank_c, rank_r, Cc, R
                sp = make_split(t.n, idx_a, idx_b)
        else:
            if len(idx_a) > len(idx_b):
                idx_a, idx_b = idx_b, idx_a
            sp = make_split(t.n, idx_a, idx_b)
            R, Cc = 4 ** len(idx_a), 4 ** len(idx_b)
        return sp, rank_r, rank_c, R, Cc

    def _gram_into(self, plan, s0, G, ws, layout, rows_pad, pitch):
        """One split (supports the reduced-format rank arrays): flatten -> Gram -> correction -> un-scatter."""
        t = self.table
        sp, rank_r, rank_c, R, Cc = plan
        try:
            call("spb_flatten_u8", _p(t.keys), _p(t.counts), t.num, C.byref(sp), _p(rank_r), _p(rank_c), _p(s0), rows_pad, pitch,
                 layout, SPB_U8_NO_MEMSET, _p(self.hi_rc), _p(self.hi_val), _p(self.hi_num), self.hi_cap, _st())
            run = lambda: call("spb_gram_u8", _p(s0), rows_pad, pitch, layout, _p(G), _p(ws), _st())  # noqa: E731
            run() if self.gram_hook is None else self.gram_hook(run, 1)
            call("spb_gram_hi_correction", _p(s0), rows_pad, pitch, layout, _p(self.hi_rc), _p(self.hi_val), _p(self.hi_num),
                 self.hi_cap, _p(G), _st())
            call("spb_flatten_u8_clear", _p(t.keys), t.num, C.byref(sp), _p(rank_r), _p(rank_c), _p(s0), rows_pad, pitch, layout,
                 _st())
        except BaseException:
            self._drop_s0()
            raise

    def _gram_batch(self, splits, s0, G, ws, layout, rows_pad, pitch):
        """nb <= GNB dense splits of equal shape: scatter, ONE Gram launch, ONE correction launch, un-scatter.
        G: [nb, rows_pad, rows_pad] view."""
        nb = len(splits)
        arr = splits if isinstance(splits, C.Array) else (_lib.SpbSplit * nb)(*splits)
        s0_stride, g_stride = rows_pad * pitch, rows_pad * rows_pad
        t = self.timer
        try:
            with _span(t, "scatter", nb):
                self._scatter(arr, nb, s0, layout, rows_pad, pitch)
            run = lambda: call("spb_gram_u8_batch", _p(s0), s0_stride, nb, rows_pad, pitch, layout, _p(G), g_stride, _p(ws), _st())  # noqa: E731
            with _span(t, "gram", nb):
                run() if self.gram_hook is None else self.gram_hook(run, nb)
            with _span(t, "correction", nb):
                call("spb_gram_hi_correction_batch", _p(s0), s0_stride, nb, rows_pad, pitch, layout, _p(self.hi_rc), _p(self.hi_val),
                     _p(self.hi_num), self.hi_cap, _p(G), g_stride, _st())
            with _span(t, "scatter", 0):
                self._scatter(arr, nb, s0, layout, rows_pad, pitch, clear=True)
        except BaseException:
            self._drop_s0()
            raise

    def gram(self, idx_a, idx_b, reduced=False):
        """Exact F F^T (short side) of the count flattening of one split.  Returns (G [rows_pad, rows_pad], k)."""
        plan = self._plan(idx_a, idx_b, reduced)
        R, Cc = plan[3], plan[4]
        layout, rows_pad, pitch = self.geometry(R, Cc)
        s0, G, ws = self._buffers(layout, rows_pad, pitch)
        self._gram_into(plan, s0[0], G[0], ws, layout, rows_pad, pitch)
        return G[0], R

    def score(self, idx_a, idx_b, reduced=False):
        G, k = self.gram(idx_a, idx_b, reduced)
        if k == 0:
            return torch.full((1,), float("nan"), dtype=torch.float64, device=G.device)
        return score_gram(G, k)

    def score_many(self, splits_idx, reduced=False, max_batch=512, max_batch_bytes=None, big_hook=None):
        """Scores of many splits.  Dense count flattenings of equal shape are batched: their Gram matrices are
        built up to 64 at a time into G[b] and ONE batched eigen-solver call scores up to `max_batch` of them
        (the Jacobi / Krylov kernels are latency-bound per matrix, so batching is what keeps all SMs busy)."""
        out = _empty(len(splits_idx), torch.float64)
        if reduced:
            for s, (ia, ib) in enumerate(splits_idx):
                out[s:s + 1] = self.score(ia, ib, True)
            return out
        if max_batch_bytes is None:
            # Gram batch buffer: at most 48 GB and at most a third of what was free when this scorer first scored (16 GB / 256
            # matrices until round 2: the 462 6|6 matrices of 12 taxa then went through the eigen-solver in 3 chunks, each with its
            # own ~0.5 ms chain of latency-bound kernels and a host synchronisation; one chunk of 462 needs 31 GB of int32 Gram).
            # Queried ONCE: cudaMemGetInfo was measured to take 4-50 ms per call on a busy context.
            if self._batch_bytes is None:
                self._batch_bytes = min(48 << 30, torch.cuda.mem_get_info()[0] // 3)
            max_batch_bytes = self._batch_bytes
        n = self.table.n
        gkey = (id(splits_idx), n, "groups")
        hit = self._plans.get(gkey)
        if hit is not None and hit[0] is splits_idx and hit[1] == len(splits_idx):
            tasks = hit[2]
        else:
            groups = {}
            for s, (ia, ib) in enumerate(splits_idx):
                groups.setdefault(min(len(ia), len(ib)), []).append(s)
            tasks = sorted(groups.items(), key=lambda g: -(4.0 ** (2 * g[0])) * 4.0 ** (n - g[0]) * len(g[1]))  # Gram work, descending
            self._plans[gkey] = (splits_idx, len(splits_idx), tasks)
        if self.nstreams == 1 or len(tasks) == 1:
            for a, members in tasks:
                self._score_group(splits_idx, a, members, out, max_batch, max_batch_bytes)
            return out
        # two host threads, two streams: greedy split of the classes by Gram work (largest class alone on the caller's stream)
        load, mine, theirs = [0.0, 0.0], [], []
        for a, members in tasks:
            cost = (4.0 ** (2 * a)) * 4.0 ** (n - a) * len(members)
            slot = 0 if load[0] <= load[1] else 1
            load[slot] += cost
            (mine if slot == 0 else theirs).append((a, members))
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream(device=out.device)
        side, dev_index, failure = self._side, out.device.index, []
        side.wait_stream(main)  # the table and `out` were produced on the caller's stream

        def worker():
            try:
                torch.cuda.set_device(dev_index)
                self._tl.slot = 1
                with torch.cuda.stream(side):
                    for a, members in theirs:
                        self._score_group(splits_idx, a, members, out, max_batch, max_batch_bytes)
            except BaseException as exc:  # noqa: BLE001  (re-raised on the calling thread)
                failure.append(exc)

        th = threading.Thread(target=worker, name="splitp_b200-score-stream-1")
        th.start()
        try:
            for a, members in mine:
                self._score_group(splits_idx, a, members, out, max_batch, max_batch_bytes)
        finally:
            th.join()
            main.wait_stream(side)
        if failure:
            raise failure[0]
        return out

    def _encoded_group(self, splits_idx, a, members):
        """Encoded splits of one size class (short side first = rows of the Gram side) and the device index list that scatters its
        scores into the output.  Cached per (split list, class): a serving loop scores the SAME splits of every new alignment,
        and rebuilding 2,035 records plus one synchronous index upload per class per step left the GPU idle between the classes
        (0.9 ms of an 8.9 ms step on 8 GPUs)."""
        n = self.table.n
        key = (id(splits_idx), n, a)
        hit = self._plans.get(key)
        if hit is not None and hit[0] is splits_idx and hit[1] == members:
            return hit[2], hit[3]
        everyone = np.arange(n)
        short, long_ = [], []
        for s in members:
            ia, ib = splits_idx[s]
            if len(ia) > len(ib):
                ia, ib = ib, ia
            short.append(ia)
            long_.append(ib)
        try:
            both = np.concatenate([np.asarray(short, dtype=np.int64).reshape(len(members), -1),
                                   np.asarray(long_, dtype=np.int64).reshape(len(members), -1)], axis=1)
        except ValueError:
            both = None
        if both is None or both.shape[1] != n or not (np.sort(both, axis=1) == everyone).all():
            raise ValueError("CountScorer: the split must cover all taxa")
        _, rec = _lib.make_splits(n, short, long_)
        where = None
        if members != list(range(members[0], members[0] + len(members))):
            where = torch.tensor(members, dtype=torch.int64, device=device())
        if len(self._plans) > 64:
            self._plans.clear()
        self._plans[key] = (splits_idx, list(members), rec, where)
        return rec, where

    def _score_group(self, splits_idx, a, members, out, max_batch, max_batch_bytes):
        """All splits whose shorter side has `a` taxa (equal shapes): batched scatter / Gram / correction / eigen-solver."""
        n = self.table.n
        rec, where = self._encoded_group(splits_idx, a, members)
        R, Cc = 4 ** a, 4 ** (n - a)
        layout, rows_pad, pitch = self.geometry(R, Cc)
        i32 = self._use_i32(layout, rows_pad, pitch) and R > JACOBI_MAX_K
        per_matrix = rows_pad * rows_pad * 8 if not i32 else rows_pad * rows_pad * 4 + max(self.n_hi, 1) * rows_pad * 8
        B = int(max(1, min(len(members), max_batch, max_batch_bytes // per_matrix)))
        B = -(-len(members) // -(-len(members) // B))  # equal chunks: no small tail batch through the eigen-solver
        if i32:
            s0 = self._buffers(layout, rows_pad, pitch, 1)[0]
            buf = self._buffers_i32(rows_pad, B)
        else:
            s0, G, ws = self._buffers(layout, rows_pad, pitch, B)
        for c0 in range(0, len(members), B):
            chunk = members[c0:c0 + B]
            gnb = self._gnb(rows_pad, pitch)
            for b0 in range(0, len(chunk), gnb):
                nsub = min(gnb, len(chunk) - b0)
                plans = (_lib.SpbSplit * nsub).from_buffer(rec, (c0 + b0) * rec.itemsize)
                if i32:
                    self._gram_batch_i32(plans, s0, buf, b0, layout, rows_pad, pitch)
                else:
                    self._gram_batch(plans, s0, G[b0:b0 + nsub], ws, layout, rows_pad, pitch)
            with _span(self.timer, "eigen", len(chunk)):
                sc = self._score_i32(buf, len(chunk), R) if i32 else score_gram(G[:len(chunk)], R)
            if where is None:
                out[chunk[0]:chunk[0] + len(chunk)] = sc
            else:
                out.index_copy_(0, where[c0:c0 + len(chunk)], sc)

    def check_hi(self):
        """Kept for API stability: the capacity is guaranteed by construction (see the `table` setter)."""
        if self.n_hi > self.hi_cap:
            raise MemoryError(f"splitp_b200: {self.n_hi} counts >= 256 exceed the high-part capacity {self.hi_cap}")


def score_splits_counts(table, splits_idx, reduced=False):
    """Scores of many splits [(idx_a, idx_b), ...] of a count table, exact-integer Gram path."""
    scorer = CountScorer(table)
    out = scorer.score_many(splits_idx, reduced)
    scorer.check_hi()
    return out


# --------------------------------------------------------------------------------------------
# subflattenings (kernel 3)
# --------------------------------------------------------------------------------------------
class PairTables:
    def __init__(self, n, N_tab, T, total):
        self.n, self.N, self.T, self.total = n, N_tab, T, total
        self.triples = None  # triple tables of the round-2 scorer (built on first use by subflatten_scores)


def pair_raw(aln, word_begin=0, word_end=None):
    """Raw pair statistics of a range of 32-site words (sum-reducible across GPUs)."""
    if aln.planes is None:
        raise ValueError("pair tables need the taxon-major bit planes (pack(want_planes=True))")
    word_end = (aln.N + 31) // 32 if word_end is None else word_end
    raw = _zeros(int(lib.spb_pair_raw_words(aln.n)), torch.int64)
    call("spb_pair_tables", _p(aln.planes), _p(aln.valid), aln.n, aln.plane_words, word_begin, word_end, _p(raw), _st())
    return raw


def pair_finalize(raw, n, divisor=0.0):
    N_tab, T, total = _empty((n, n, 4, 4), torch.float64), _empty((n, n, 4, 4), torch.float64), _empty(1, torch.float64)
    call("spb_pair_finalize", _p(raw), n, float(divisor), _p(N_tab), _p(T), _p(total), _st())
    return PairTables(n, N_tab, T, total)


def pair_tables_from_alignment(aln, as_counts=False):
    raw = pair_raw(aln)
    usable = 0.0 if as_counts else float(int(raw[-1].item()))
    return pair_finalize(raw, aln.n, usable)


def pair_tables_from_table(table, as_counts=False):
    n = table.n
    vals = table.counts.to(torch.float64) if (as_counts and table.counts is not None) else table.values_f64()
    if isinstance(table, WidePatternTable):  # deterministic fp64 tensor-core product (csrc/wide.cu)
        N_tab = _empty((n, n, 4, 4), torch.float64)
        ws = _empty(max(int(lib.spb_pair_tables_wide_ws(table.num, n)), 1), torch.float64)
        call("spb_pair_tables_wide", _p(table.keys), _p(vals.contiguous()), table.num, n, _p(N_tab), _p(ws), _st())
    else:
        N_tab = _zeros((n, n, 4, 4), torch.float64)
        call("spb_pair_tables_weighted", _p(table.keys), _p(vals.contiguous()), table.num, n, _p(N_tab), _st())
    T, total = _empty((n, n, 4, 4), torch.float64), _empty(1, torch.float64)
    call("spb_pair_transform", _p(N_tab), n, _p(T), _p(total), _st())
    return PairTables(n, N_tab, T, total)


def subflatten(pt, idx_a, idx_b):
    sp = make_split(pt.n, idx_a, idx_b)
    out = _empty((3 * len(idx_a) + 1, 3 * len(idx_b) + 1), torch.float64)
    call("spb_subflatten", _p(pt.T), _p(pt.total), pt.n, C.byref(sp), _p(out), _st())
    return out


def masks_from_splits(splits_idx):
    ma = np.zeros(len(splits_idx), dtype=np.uint64)
    mb = np.zeros(len(splits_idx), dtype=np.uint64)
    for s, (ia, ib) in enumerate(splits_idx):
        ma[s] = sum(1 << t for t in ia)
        mb[s] = sum(1 << t for t in ib)
    return ma, mb


def subflatten_scores(pt, masks_a, masks_b=None):
    """Batched subflattening scores.  masks: uint64 bit masks over taxon positions (torch int64 tensors on
    the device, or numpy uint64 arrays).  Side taxa are taken in ascending position order."""
    def up(m):
        if m is None or isinstance(m, torch.Tensor):
            return m
        return torch.from_numpy(np.ascontiguousarray(m).view(np.int64)).to(device())
    ma, mb = up(masks_a), up(masks_b)
    out = _empty(int(ma.shape[0]), torch.float64)
    if pt.n <= SUBFLATTEN_TABLES_MAX_TAXA and os.environ.get("SPB_SUBFLATTEN_KERNEL", "tables") == "tables":
        ready = pt.triples is not None
        if not ready:
            pt.triples = _empty(int(lib.spb_subflatten_tables_doubles(pt.n)), torch.float64)
        call("spb_subflatten_score_tables", _p(pt.T), _p(pt.total), pt.n, _p(ma), _p(mb), int(ma.shape[0]), _p(out), _p(pt.triples),
             int(ready), _st())
    else:  # sides above 21 taxa (or SPB_SUBFLATTEN_KERNEL=staged for A/B runs): the kernels that stage the subflattening
        call("spb_subflatten_score", _p(pt.T), _p(pt.total), pt.n, _p(ma), _p(mb), int(ma.shape[0]), _p(out), _st())
    return out


# --------------------------------------------------------------------------------------------
# Alignment.sub_alignment support (splitp/alignment.py:10-31)
# --------------------------------------------------------------------------------------------
def marginalise(table, idx):
    """Pattern table over the taxa positions `idx` (ascending): values of collapsing patterns are added.  Keys come back
    ascending.  A WidePatternTable gives a PatternTable when at most 31 taxa are kept, else a WidePatternTable."""
    idx = sorted(idx)
    if isinstance(table, WidePatternTable) and len(idx) > NARROW_MAX_TAXA:
        # 128-bit sub-keys: stable two-pass sort (as WideTable.compact), then one sum per run of equal keys
        keys = project_keys(table, idx)
        order = _wide_order(keys)
        keys, vals = keys[order], table.values[order]
        new = torch.ones(keys.shape[0], dtype=torch.bool, device=keys.device)
        new[1:] = (keys[1:] != keys[:-1]).any(dim=1)
        seg = torch.cumsum(new, 0) - 1
        keys = keys[new].contiguous()
        acc = torch.zeros(keys.shape[0], dtype=torch.float64, device=keys.device).index_add_(0, seg, vals)
        out = WidePatternTable(len(idx), keys, acc)
        out.integral = table.integral
        return out
    rows = project_keys(table, idx) if isinstance(table, WidePatternTable) else flatten_coo(table, idx, [])[0]
    if table.counts is not None and len(idx) <= DIRECT_MAX_TAXA:
        # integer counts, at most 12 taxa: add into the direct-indexed table and compact it (the library's own kernels; the
        # compaction returns the keys in ascending order, as torch.unique did)
        m, cells, total = len(idx), 4 ** len(idx), int(rows.shape[0])
        if int(table.counts.to(torch.int64).sum().item()) >= 2 ** 31:
            raise OverflowError("marginalise: pattern counts above 2^31 - 1 do not fit the 32-bit count table")
        direct = _zeros(cells, torch.int32)
        call("spb_direct_merge", _p(rows.contiguous()), _p(table.counts.contiguous()), total, cells, _p(direct), _st())
        cap = min(cells, max(total, 1))
        keys, counts, num = _empty(cap, torch.int64), _empty(cap, torch.int32), _zeros(1, torch.int64)
        tmp = _empty(int(lib.spb_compact_tmp_words(cells)), torch.int32)
        call("spb_compact_direct", _p(direct), None, cells, _p(keys), _p(counts), None, cap, _p(num), _p(tmp), _st())
        P = int(num.item())
        return PatternTable(m, keys[:P], counts=counts[:P], divisor=table.divisor)
    uniq, inv = torch.unique(rows, return_inverse=True)  # larger sub-alignments / probability tables: library sort (DESIGN.md section 7)
    if table.counts is not None:
        acc = torch.zeros(len(uniq), dtype=torch.int64, device=rows.device).index_add_(0, inv, table.counts.to(torch.int64))
        return PatternTable(len(idx), uniq, counts=acc.to(torch.int32), divisor=table.divisor)
    acc = torch.zeros(len(uniq), dtype=torch.float64, device=rows.device).index_add_(0, inv, table.values)
    out = PatternTable(len(idx), uniq, values=acc)
    out.integral = table.integral
    return out


# --------------------------------------------------------------------------------------------
# marginals, rank-1 approximation and rank-1 divergence of a flattening (SURVEY section 8 row f4;
# splitp/phylogenetics.py:331-373, banned states: splitp/constructions.py:94-101)
# --------------------------------------------------------------------------------------------
MI_DIRECT_CELLS = 1 << 22  # a side of up to 11 taxa keeps its sums in a direct-indexed array, longer sides in a hash table


class SideSums:
    """Sums of the raw table values per row (or column) index of a flattening: `sums[index]` when `keys` is None,
    else an open-addressing table (`keys[slot]` = index or -1, `sums[slot]`)."""

    def __init__(self, side_len, distinct_bound):
        cells = 4 ** side_len
        cap = 1024
        while cap < 2 * max(distinct_bound, 1):
            cap *= 2
        if cells <= MI_DIRECT_CELLS or (side_len <= 15 and cells <= cap):
            self.keys, self.cap = None, cells
        else:
            self.keys, self.cap = torch.full((cap,), -1, dtype=torch.int64, device=device()), cap
        self.sums = _zeros(self.cap, torch.float64)

    def args(self):
        return _p(self.sums), _p(self.keys), self.cap


def table_marginals(table, idx_a, idx_b, ban_row=-1, ban_col=-1):
    """(row sums, column sums) of the flattening of a split that places every taxon on one side, as SideSums of the RAW
    table values (counts stay integers).  ban_row / ban_col: state code 0..3 whose repeated occurrence in the row /
    column pattern zeroes the entry (constructions.py:94-99), -1 = none."""
    _narrow_only(table, "table marginals")
    sp = make_split(table.n, idx_a, idx_b)
    rs, cs = SideSums(len(idx_a), table.num), SideSums(len(idx_b), table.num)
    ovf = _zeros(1, torch.int32)
    vp, kind, _ = table.val_args(True)
    call("spb_table_marginals", _p(table.keys), vp, kind, table.num, C.byref(sp), int(ban_row), int(ban_col),
         *rs.args(), *cs.args(), _p(ovf), _st())
    if (rs.keys is not None or cs.keys is not None) and int(ovf.item()):
        raise MemoryError("splitp_b200: side-sum hash table overflow")
    return rs, cs


def _partials():
    return _empty(int(lib.spb_mi_partials()), torch.float64)


def rank1_divergence_table(table, idx_a, idx_b):
    """sum over patterns of v log(v / (r c)) without materialising the flattening (phylogenetics.py:364-373);
    float64 tensor [1].  NotImplementedError (from the library) for a split that does not cover all taxa."""
    _narrow_only(table, "the rank-1 divergence")
    rs, cs = table_marginals(table, idx_a, idx_b)
    sp = make_split(table.n, idx_a, idx_b)
    vp, kind, div = table.val_args()
    out = _empty(1, torch.float64)
    call("spb_mi_table", _p(table.keys), vp, kind, div, table.num, C.byref(sp), *rs.args(), *cs.args(), _p(_partials()),
         _p(out), _st())
    return out


def marginals_dense(F):
    """(row sums, column sums) of a device matrix."""
    F = F.contiguous()
    rows, cols = F.shape
    rowsum, colsum = _empty(rows, torch.float64), _empty(cols, torch.float64)
    call("spb_marginals_dense", _p(F), rows, cols, F.stride(0) if rows else cols, _p(rowsum), _p(colsum), _st())
    return rowsum, colsum


def rank1_divergence_dense(F):
    F = F.contiguous()
    rows, cols = F.shape
    rowsum, colsum = marginals_dense(F)
    out = _empty(1, torch.float64)
    call("spb_mi_dense", _p(F), rows, cols, F.stride(0) if rows else cols, _p(rowsum), _p(colsum), _p(_partials()), _p(out), _st())
    return out


def rank1_divergence(table, idx_a, idx_b):
    """Rank-1 divergence of the flattening of (idx_a | idx_b): from the table when the split covers all taxa, else
    from the reduced flattening (dropping all-zero rows / columns does not change the sum)."""
    if covers_all(table.n, idx_a, idx_b):
        return rank1_divergence_table(table, idx_a, idx_b)
    return rank1_divergence_dense(flatten_reduced(table, idx_a, idx_b))


def outer(x, y, out=None, accumulate=False):
    """out[i, j] (+)= x[i] * y[j] on the device."""
    x, y = x.contiguous(), y.contiguous()
    if out is None:
        out = _empty((x.shape[0], y.shape[0]), torch.float64)
        accumulate = False
    call("spb_outer_f64", _p(x), x.shape[0], _p(y), y.shape[0], _p(out), int(bool(accumulate)), _st())
    return out


def flatten_coo_banned(table, idx_a, idx_b, ban_row=-1, ban_col=-1):
    """(rows, cols, banned) of every pattern; banned[i] = 1 where the banned-state rule assigns 0."""
    _narrow_only(table, "flattening with banned patterns")
    sp = make_split(table.n, idx_a, idx_b)
    rows, cols = _empty(table.num, torch.int64), _empty(table.num, torch.int64)
    banned = _empty(table.num, torch.uint8)
    call("spb_flatten_coo_banned", _p(table.keys), table.num, C.byref(sp), int(ban_row), int(ban_col), _p(rows), _p(cols),
         _p(banned), _st())
    return rows, cols, banned


# --------------------------------------------------------------------------------------------
# wide keys: up to 64 taxa (BASELINE config 4)
# --------------------------------------------------------------------------------------------
class WideTable:
    """Hashed pattern table with 128-bit keys (two uint64 words {lo, hi} per key).  `hkeys` / `hcounts` are the
    open-addressing table itself (kept because the thin-split Gram looks patterns up in it), `special` the count
    of the all-ones key (the all-T pattern at exactly 64 taxa doubles as the EMPTY marker), `hfirst` (optional,
    cap + 1 cells) the first site of every pattern."""

    def __init__(self, n, hkeys, hcounts, cap, special, usable, taxa=None, hfirst=None):
        self.n, self.hkeys, self.hcounts, self.cap, self.special = n, hkeys, hcounts, cap, special
        self.hfirst = hfirst
        self.divisor = float(usable)
        self.taxa = tuple(taxa) if taxa is not None else None

    def compact(self, sort=True, want_first=False):
        """(keys int64 [P, 2] = {lo, hi}, counts int32 [P][, first int32 [P]]); sorted ascending as unsigned 128-bit
        numbers (= lexicographic A<C<G<T pattern order) when sort=True."""
        if want_first and self.hfirst is None:
            raise ValueError("this table was built without first-site tracking")
        num = _zeros(1, torch.int64)
        used = max(int((self.hcounts != 0).sum().item()), 1)
        keys, counts = _empty((used, 2), torch.int64), _empty(used, torch.int32)
        first = _empty(used, torch.int32) if want_first else None
        call("spb_compact_hash_wide", _p(self.hkeys), _p(self.hcounts), _p(self.hfirst) if want_first else None, self.cap, _p(keys),
             _p(counts), _p(first), used, _p(num), _st())
        P = int(num.item())
        keys, counts = keys[:P], counts[:P]
        first = first[:P] if want_first else None
        sp = int(self.special.item())
        if sp:  # the all-ones pattern lives outside the table
            keys = torch.cat([keys, torch.full((1, 2), -1, dtype=torch.int64, device=keys.device)])
            counts = torch.cat([counts, torch.tensor([sp], dtype=torch.int32, device=keys.device)])
            if want_first:
                first = torch.cat([first, self.hfirst[self.cap:self.cap + 1]])
        if sort and keys.shape[0] > 1:
            order = _wide_order(keys)
            keys, counts = keys[order], counts[order]
            first = first[order] if want_first else None
        return (keys, counts, first) if want_first else (keys, counts)

    def _patterns(self, keys):
        k = keys.cpu().numpy().view(np.uint64)
        out = []
        for lo, hi in k:
            v = (int(hi) << 64) | int(lo)
            out.append("".join(STATES[(v >> (2 * (self.n - 1 - j))) & 3] for j in range(self.n)))
        return out

    def to_dict(self, as_counts=True, order="sorted"):
        """{pattern: count (or count / usable)}; order = "sorted" (lexicographic, simulation.py:50-54) or "first"
        (first occurrence along the alignment, the dict order of fasta.py:48-63)."""
        if order == "first":
            keys, counts, first = self.compact(sort=False, want_first=True)
            perm = torch.argsort(first.to(torch.int64) & 0xFFFFFFFF)
            keys, counts = keys[perm], counts[perm]
        else:
            keys, counts = self.compact()
        c = counts.cpu().numpy().view(np.uint32)
        return {p: (int(x) if as_counts or self.divisor <= 0 else int(x) / self.divisor) for p, x in zip(self._patterns(keys), c)}


def _wide_order(keys):
    """Permutation that sorts 128-bit keys int64 [P, 2] = {lo, hi} ascending as unsigned numbers: stable sort by lo, then
    by hi (torch.sort: library sort, DESIGN.md section 7)."""
    flip = torch.tensor(-(1 << 63), dtype=torch.int64, device=keys.device)  # unsigned order through signed sorts
    o1 = torch.sort(keys[:, 0] ^ flip, stable=True).indices
    o2 = torch.sort((keys[:, 1] ^ flip)[o1], stable=True).indices
    return o1[o2]


def pack_wide(chars, is_ascii=False):
    """chars uint8 [n, N] (device tensor or host array) -> (wide int64 [N, 2], valid int32 [Wp], n, N)."""
    if not isinstance(chars, torch.Tensor):
        chars = torch.from_numpy(np.ascontiguousarray(np.asarray(chars, dtype=np.uint8))).to(device())
    chars = chars.contiguous()
    n, N = int(chars.shape[0]), int(chars.shape[1])
    wide = _empty((max(N, 1), 2), torch.int64)
    valid = _zeros(int(lib.spb_plane_words(N)), torch.int32)
    if N:
        call("spb_pack_wide", _p(chars), n, N, N, int(bool(is_ascii)), _p(wide), _p(valid), _st())
    return wide, valid, n, N


def _new_wide_table(entries):
    cap = 1024
    while cap < 2 * max(int(entries), 1):
        cap *= 2
    hk = torch.full((cap, 2), -1, dtype=torch.int64, device=device())
    return hk, _zeros(cap, torch.int32), cap


def count_patterns_wide(wide, valid, n, N, site_begin=0, site_end=None, taxa=None, want_first=False):
    """Pattern compression with 128-bit keys (n <= 64): one pass, open-addressing table."""
    site_end = N if site_end is None else site_end
    hk, hc, cap = _new_wide_table(site_end - site_begin)
    hf = torch.full((cap + 1,), -1, dtype=torch.int32, device=device()) if want_first else None
    special, usable, ovf = _zeros(1, torch.int64), _zeros(1, torch.int64), _zeros(1, torch.int32)
    if site_end > site_begin:
        call("spb_count_hash_wide", _p(wide), _p(valid), site_begin, site_end, _p(hk), _p(hc), _p(hf), cap, _p(special), _p(usable),
             _p(ovf), _st())
    if int(ovf.item()):
        raise MemoryError("splitp_b200: pattern hash table overflow")
    return WideTable(n, hk, hc, cap, special, int(usable.item()), taxa, hf)


def merge_wide_tables(n, keys, counts, usable, taxa=None):
    """One table from a concatenated (key, count) list (the multi-GPU merge of hashed wide tables)."""
    hk, hc, cap = _new_wide_table(keys.shape[0])
    special, ovf = _zeros(1, torch.int64), _zeros(1, torch.int32)
    if keys.shape[0]:
        call("spb_hash_merge_wide", _p(keys.contiguous()), _p(counts.contiguous()), None, int(keys.shape[0]), _p(hk), _p(hc), None, cap,
             _p(special), _p(ovf), _st())
    if int(ovf.item()):
        raise MemoryError("splitp_b200: pattern hash table overflow")
    return WideTable(n, hk, hc, cap, special, usable, taxa)


def thin_split_scores(table, thin_sides, filtered=True):
    """Scores of the splits {side} | {all other taxa} for sides of 1, 2 or 3 taxon positions: exact Gram of the REDUCED
    flattening (4^a rows, one column per distinct pattern of the other taxa) from hash lookups, then the small-matrix
    scorer.  Sides of one taxon give a 4-row matrix, hence score 0 like the reference.  filtered: a per-split column
    bitmap lets patterns without a partner in their column skip the lookups (same result)."""
    out = _empty(len(thin_sides), torch.float64)
    cells = 4 ** (2 * max([len(list(s)) for s in thin_sides] + [2]))
    G = _empty((len(thin_sides), cells), torch.float64)
    words = int(lib.spb_thin_filter_words(table.cap)) if filtered else 0
    filt = _empty(2 * words, torch.int32) if filtered else None
    by_a = {1: [], 2: [], 3: []}
    for s, side in enumerate(thin_sides):
        side = list(side)
        if len(side) not in (1, 2, 3):
            raise NotImplementedError("thin_split_scores: the thin side must have 1, 2 or 3 taxa")
        call("spb_thin_gram_wide_filtered", _p(table.hkeys), _p(table.hcounts), table.cap, _p(table.special), table.n, bytes(side),
             len(side), _p(filt), words, _p(G[s]), _st())
        by_a[len(side)].append(s)
    for a, members in by_a.items():
        if not members:
            continue
        idx = torch.tensor(members, dtype=torch.int64, device=out.device)
        R = 4 ** a
        # the Gram of entry s occupies the leading R*R doubles of G[s] with row stride R: repack to [R, R] matrices
        Gs = G[idx][:, :R * R].reshape(len(members), R, R).contiguous()
        out.index_copy_(0, idx, score_gram(Gs, R))
    return out
