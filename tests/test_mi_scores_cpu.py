"""Host-side parts of the batched rank-1 divergence (engine.rank1_divergence_scores): side digit masks for uint64 and 128-bit
keys, batch cutting by workspace bytes, and the inputs the public entry points refuse before any device work."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def eng():
    from splitp_b200 import engine
    return engine


def _key_words(eng, patterns):
    keys, n = eng.encode_patterns(patterns)
    keys = np.asarray(keys, dtype=np.uint64)
    return (keys[:, 0], keys[:, 1]) if keys.ndim == 2 else (keys, np.zeros_like(keys))


@pytest.mark.parametrize("n", [5, 31, 32, 47, 64])
def test_side_mask_matches_zeroed_digits(eng, n):
    """key AND side_mask(side) is the key of the pattern with every other taxon set to A (digit 0), for both key layouts."""
    rng = np.random.default_rng(n)
    pats = ["".join(rng.choice(list("ACGT"), size=n)) for _ in range(50)] + ["T" * n]
    lo, hi = _key_words(eng, pats)
    for _ in range(6):
        side = sorted(rng.choice(n, size=int(rng.integers(1, n)), replace=False).tolist())
        mlo, mhi = eng.side_mask(n, side)
        zeroed = ["".join(ch if t in side else "A" for t, ch in enumerate(p)) for p in pats]
        zlo, zhi = _key_words(eng, zeroed)
        assert np.array_equal(lo & np.uint64(mlo), zlo) and np.array_equal(hi & np.uint64(mhi), zhi)
        full = np.uint64(2**64 - 1)
        assert not (((lo & np.uint64(mlo)) == full) & ((hi & np.uint64(mhi)) == full)).any()  # never the EMPTY marker
    if n <= 31:
        assert eng.side_mask(n, range(n))[1] == 0


def test_side_cap(eng):
    lib = eng.lib
    assert lib.spb_mi_side_cap(60_203, 1) == 8            # 4 distinct side keys
    assert lib.spb_mi_side_cap(60_203, 6) == 8192         # 4^6 distinct
    assert lib.spb_mi_side_cap(60_203, 11) == 131_072     # bounded by the pattern count
    assert lib.spb_mi_side_cap(1_000_000, 63) == 1 << 21
    for P in (1, 7, 1000, 65_536):
        for a in (1, 3, 12, 40):
            cap = lib.spb_mi_side_cap(P, a)
            assert cap & (cap - 1) == 0 and cap >= 2 * min(P, 4 ** a)


def test_batches_cut_by_bytes(eng, monkeypatch):
    lib = eng.lib
    P, W = 60_203, 1
    slots = [lib.spb_mi_side_cap(P, a) + lib.spb_mi_side_cap(P, 12 - a) for a in (1, 2, 3, 4, 5, 6) for _ in range(40)]
    cap = 64 << 20
    batches = eng.mi_batches(slots, P, W, cap=cap)
    assert batches[0][0] == 0 and batches[-1][1] == len(slots)
    assert all(b0 < b1 for b0, b1 in batches) and all(a[1] == b[0] for a, b in zip(batches, batches[1:]))
    for b0, b1 in batches:
        assert 8 * lib.spb_mi_scores_ws(P, W, sum(slots[b0:b1]), b1 - b0) <= cap
    for (b0, b1), (c0, _) in zip(batches, batches[1:]):  # each batch is cut only when the next split would not fit
        assert 8 * lib.spb_mi_scores_ws(P, W, sum(slots[b0:c0 + 1]), c0 + 1 - b0) > cap
    # a single split larger than the cap still gets its own batch
    assert eng.mi_batches([1 << 30, 8], P, W, cap=1024) == [(0, 1), (1, 2)]
    monkeypatch.setattr(eng, "MI_BATCH_BYTES", cap)
    assert eng.mi_batches(slots, P, W) == batches


def test_distance_still_refused():
    from splitp_b200 import batch
    from splitp_b200.enums import Method
    with pytest.raises(NotImplementedError):
        batch.SplitScorer([([0], [1, 2, 3])], method=Method.distance)
    batch.SplitScorer([([0], [1, 2, 3])], method=Method.mutual_information)  # accepted


def test_non_covering_split_raises(eng):
    table = eng.PatternTable(4, torch.zeros(0, dtype=torch.int64), values=torch.zeros(0, dtype=torch.float64))
    for bad in (([0, 1], [2]), ([0, 1], [1, 2, 3]), ([0, 1, 2, 3, 4], [])):
        with pytest.raises(ValueError):
            eng.rank1_divergence_scores(table, [([0], [1, 2, 3]), bad])
