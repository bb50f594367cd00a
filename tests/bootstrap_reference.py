"""Host model of the bootstrap resampling rule of csrc/bootstrap.cu (tests/test_bootstrap_cpu.py, tests/test_gpu_bootstrap.py).

Draw s of replicate b over a table with counts c (N = sum c, table order):
    u = fmix(seed + gamma (b 2^40 + s + 1))   SplitMix64 output, all mod 2^64
    j = floor(u N / 2^64)
    pattern p with prefix[p] <= j < prefix[p + 1], prefix = exclusive cumulative counts
`draws` is the vectorised form (numpy uint64 wraps mod 2^64; the high word of u N is assembled from 32-bit halves);
`draw_scalar` restates it with Python integers.
"""
import numpy as np

GAMMA = 0x9E3779B97F4A7C15
MASK64 = (1 << 64) - 1
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def fmix(z):
    z = np.asarray(z, dtype=np.uint64)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def mulhi(a, b):
    """High 64 bits of the 128-bit products a * b (uint64 arrays)."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    a_lo, a_hi, b_lo, b_hi = a & _LO, a >> _32, b & _LO, b >> _32
    ll, hl, lh, hh = a_lo * b_lo, a_hi * b_lo, a_lo * b_hi, a_hi * b_hi
    cross = (ll >> _32) + (hl & _LO) + lh  # < 2^64: (2^32 - 1)^2 + 2 (2^32 - 1)
    return hh + (hl >> _32) + (cross >> _32)


def uniforms(seed, b, s):
    """u of draws s (array) of replicate b."""
    with np.errstate(over="ignore"):
        ctr = np.uint64((b << 40) & MASK64) + np.asarray(s, dtype=np.uint64) + np.uint64(1)
        return fmix(np.uint64(seed) + np.uint64(GAMMA) * ctr)


def sites(seed, b, N, s=None):
    """Site indices j of draws s (default 0 .. N - 1) of replicate b."""
    s = np.arange(N, dtype=np.uint64) if s is None else np.asarray(s, dtype=np.uint64)
    return mulhi(uniforms(seed, b, s), np.uint64(N))


def prefix_of(counts):
    c = np.asarray(counts, dtype=np.int64)
    return np.cumsum(c) - c


def draws(counts, seed, b):
    """Pattern index of every draw of replicate b, in draw order."""
    N = int(np.sum(np.asarray(counts, dtype=np.int64)))
    j = sites(seed, b, N).astype(np.int64)
    return np.searchsorted(prefix_of(counts), j, side="right") - 1


def replicate(counts, seed, b):
    """Counts of replicate b (int64 [P])."""
    return np.bincount(draws(counts, seed, b), minlength=len(counts))


def replicates(counts, seed, first, count):
    return np.stack([replicate(counts, seed, b) for b in range(first, first + count)])


def draw_scalar(counts, seed, b, s):
    """Pattern index of draw s of replicate b with Python integers."""
    z = (seed + GAMMA * (b * 2 ** 40 + s + 1)) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    u = z ^ (z >> 31)
    N = sum(int(c) for c in counts)
    j = (u * N) >> 64
    acc = 0
    for p, c in enumerate(counts):
        acc += int(c)
        if j < acc:
            return p
    raise AssertionError("j >= N")


def atomics_after_aggregation(pattern_of_draw):
    """Atomics the counting kernel issues for one replicate: one per distinct pattern of every aligned group of 32 draws."""
    d = np.asarray(pattern_of_draw, dtype=np.int64)
    pad = (-len(d)) % 32
    g = np.concatenate([d, np.full(pad, -1)]).reshape(-1, 32)
    g = np.sort(g, axis=1)
    distinct = 1 + (g[:, 1:] != g[:, :-1]).sum(axis=1)
    return int(distinct.sum() - (g[:, 0] == -1).sum())
