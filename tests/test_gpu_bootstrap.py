"""GPU tests of the bootstrap (csrc/bootstrap.cu, engine.bootstrap_counts / bootstrap_tables, batch.bootstrap_scores):
replicate counts bit for bit against the host model of tests/bootstrap_reference.py, compaction against a host filter, and
the scores of every replicate against `score_splits` on the alignment that repeats each pattern as often as the replicate
drew it.  Run with `-m gpu`.

Expected agreement with the expanded replicate (the same pattern table in the same order reaches the same scorer):
flattening and mutual information scores are equal; subflattening scores come from pair tables of the replicate's counts
instead of the alignment's bit planes and agree within max(1e-9, 64 eps / score^2) relative.
"""
import numpy as np
import pytest

import bench_inputs as BI
from tests import bootstrap_reference as BR

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0x5EED


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401  (bootstrap_scores, score_splits)
    return splitp_b200


@pytest.fixture(scope="module")
def inputs():
    """name -> code matrix [n, N]."""
    return {
        "c2": BI.simulate_codes(12, 0.05, "JC", 1_000_000, 2),       # bench workload c2's input
        "t20_big": BI.simulate_codes(20, 0.1, "JC", 400_000, 3),     # P > 131,072: past the shared-memory index at 16 entries a line
        "t20": BI.simulate_codes(20, 0.05, "JC", 100_000, 3),
        "t40": BI.simulate_codes(40, 0.1, "JC", 20_000, 4),
        "t64": BI.simulate_codes(64, 0.1, "JC", 20_000, 5),
    }


def parent(sp, codes):
    """(table as bootstrap_scores counts it, keys numpy, counts numpy) of a code matrix."""
    eng = sp.engine
    n = codes.shape[0]
    if n <= eng.NARROW_MAX_TAXA:
        table = eng.count_patterns(eng.pack(codes))
        keys, counts = table.keys, table.counts
    else:
        table = eng.count_patterns_wide(*eng.pack_wide(codes))
        keys, counts = table.compact()
    return table, keys.cpu().numpy().view(np.uint64), counts.cpu().numpy().view(np.uint32).astype(np.int64)


def key_codes(keys, n):
    """uint64 keys [P] (or {lo, hi} [P, 2]) -> uint8 codes [P, n], taxon 0 most significant."""
    sh = 2 * (n - 1 - np.arange(n))
    if keys.ndim == 1:
        return ((keys[:, None] >> sh.astype(np.uint64)) & np.uint64(3)).astype(np.uint8)
    lo = (keys[:, 0:1] >> np.minimum(sh, 62).astype(np.uint64)) & np.uint64(3)
    hi = (keys[:, 1:2] >> np.maximum(sh - 64, 0).astype(np.uint64)) & np.uint64(3)
    return np.where(sh >= 64, hi, lo).astype(np.uint8)


def expanded(keys, counts_b, n):
    """The alignment [n, N] that holds pattern p counts_b[p] times."""
    return np.ascontiguousarray(np.repeat(key_codes(keys, n), counts_b, axis=0).T)


@pytest.mark.parametrize("name", ["c2", "t20_big", "t64"])
def test_counts_equal_model(sp, inputs, name):
    table, _, counts = parent(sp, inputs[name])
    if name == "t20_big":
        assert len(counts) > 8192 * 16
    got = sp.engine.bootstrap_counts(table, 0, 3, SEED).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, BR.replicates(counts, SEED, 0, 3))


def test_counts_of_a_later_chunk(sp, inputs):
    table, _, counts = parent(sp, inputs["c2"])
    eng = sp.engine
    late = eng.bootstrap_counts(table, 5, 2, 7).cpu().numpy().view(np.uint32)
    assert np.array_equal(late, BR.replicates(counts, 7, 5, 2))
    assert np.array_equal(late, eng.bootstrap_counts(table, 0, 7, 7).cpu().numpy().view(np.uint32)[5:])


@pytest.mark.parametrize("patterns", [1, 2])
def test_counts_of_tiny_tables(sp, patterns):
    codes = np.zeros((6, 1000), dtype=np.uint8)
    codes[2, :300] = 3 if patterns == 2 else 0
    table, _, counts = parent(sp, codes)
    assert len(counts) == patterns
    got = sp.engine.bootstrap_counts(table, 0, 9, 1).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, BR.replicates(counts, 1, 0, 9))
    assert (got.sum(axis=1) == 1000).all()


@pytest.mark.parametrize("name", ["t20_big", "t64"])
def test_compaction_equals_host_filter(sp, inputs, name):
    n = inputs[name].shape[0]
    table, keys, counts = parent(sp, inputs[name])
    N = int(counts.sum())
    model = BR.replicates(counts, SEED, 0, 3)
    for b, tb in enumerate(sp.engine.bootstrap_tables(table, 3, SEED)):
        nz = model[b] != 0
        assert tb.n == n and tb.divisor == N
        assert np.array_equal(tb.keys.cpu().numpy().view(np.uint64), keys[nz])
        assert np.array_equal(tb.counts.cpu().numpy().view(np.uint32), model[b][nz])
        if n > sp.engine.NARROW_MAX_TAXA:
            assert isinstance(tb, sp.engine.WidePatternTable)
            assert np.array_equal(tb.values.cpu().numpy(), model[b][nz] / N)
        else:
            assert isinstance(tb, sp.engine.PatternTable)


CASES = [  # (method, input, split count or None = all)
    ("flattening", "c2", None), ("flattening", "t20", 12), ("flattening", "t40", 12),
    ("subflattening", "c2", None), ("subflattening", "t20", 300), ("subflattening", "t40", 100),
    ("mutual_information", "c2", None), ("mutual_information", "t40", 100),
]


@pytest.mark.parametrize("method,name,count", CASES)
def test_scores_equal_expanded_replicates(sp, inputs, method, name, count):
    codes = inputs[name]
    n = codes.shape[0]
    splits = BI.all_splits_idx(n) if count is None else BI.random_splits_idx(n, count, seed=n)
    m = getattr(sp.Method, method)
    got = sp.batch.bootstrap_scores(codes, splits, m, replicates=3, seed=SEED)
    assert got.shape == (3, len(splits)) and got.dtype == np.float64
    table, keys, _ = parent(sp, codes)
    rows = sp.engine.bootstrap_counts(table, 0, 3, SEED).cpu().numpy().view(np.uint32)
    for b in range(3):
        ref = sp.batch.score_splits(expanded(keys, rows[b], n), splits, m)
        if method == "subflattening":
            tol = np.maximum(1e-9, 64 * np.finfo(float).eps / ref ** 2)
            assert (np.abs(got[b] - ref) <= tol * np.abs(ref)).all(), np.max(np.abs(got[b] - ref) / np.abs(ref))
        else:
            assert np.array_equal(got[b], ref), np.max(np.abs(got[b] - ref))


def test_reproducible_and_chunk_independent(sp, inputs, monkeypatch):
    codes = inputs["c2"][:, :100_000]
    splits = BI.all_splits_idx(12)[::17]
    bs = sp.batch.bootstrap_scores
    for m in (sp.Method.flattening, sp.Method.mutual_information):
        a = bs(codes, splits, m, replicates=5, seed=3)
        assert np.array_equal(a, bs(codes, splits, m, replicates=5, seed=3))
        assert not np.array_equal(a, bs(codes, splits, m, replicates=5, seed=4))
        with monkeypatch.context() as mp:
            mp.setattr(sp.engine, "BOOTSTRAP_BATCH_BYTES", 1)  # one replicate per pass
            assert np.array_equal(a, bs(codes, splits, m, replicates=5, seed=3))
        assert np.array_equal(a[:2], bs(codes, splits, m, replicates=2, seed=3))
    wide = inputs["t40"]
    splits = BI.random_splits_idx(40, 20, seed=1)
    a = bs(wide, splits, sp.Method.mutual_information, replicates=3, seed=2 ** 64 - 1)
    assert np.array_equal(a, bs(wide, splits, sp.Method.mutual_information, replicates=3, seed=2 ** 64 - 1))


def test_labels_and_edge_cases(sp, inputs):
    codes = inputs["c2"][:, :20_000]
    taxa = [f"t{i}" for i in range(12)]
    splits = BI.all_splits_idx(12)[:40]
    labelled = [([taxa[i] for i in a], [taxa[i] for i in b]) for a, b in splits]
    aln = {t: "".join("ACGT"[c] for c in row) for t, row in zip(taxa, codes)}
    mi = sp.Method.mutual_information
    ref = sp.batch.bootstrap_scores(codes, splits, mi, replicates=2, seed=9)
    assert np.array_equal(sp.batch.bootstrap_scores(aln, labelled, mi, replicates=2, seed=9), ref)
    assert np.array_equal(sp.batch.bootstrap_scores(codes, labelled, mi, replicates=2, seed=9, taxa=taxa), ref)
    assert sp.batch.bootstrap_scores(codes, [], mi, replicates=4).shape == (4, 0)
    for n in (12, 40):
        gaps = np.zeros((n, 500), dtype=np.uint8)
        gaps[0] = 255  # no usable site
        with pytest.raises(ValueError, match="usable site"):
            sp.batch.bootstrap_scores(gaps, [(list(range(n // 2)), list(range(n // 2, n)))], mi, replicates=2)
