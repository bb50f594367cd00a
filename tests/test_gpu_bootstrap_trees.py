"""GPU tests of bootstrap trees (csrc/agglomerate.cu, the multi-table subflattening kernels of csrc/pairs.cu,
engine.erickson_lockstep / subflatten_scores_multi / bootstrap_tree_masks, batch.bootstrap_trees).  Run with `-m gpu`.

The lockstep agglomeration is checked against the restatement of erickson_SVD's loop in tests/erickson_reference.py: with
a fake integer-valued score (many exact ties) the chosen sequences must be equal, and with the real scores every pick must
be the first minimum of its step.
"""
import numpy as np
import pytest

import bench_inputs as BI
from tests import erickson_reference as ER

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0x7EE5


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401
    return splitp_b200


def counted(sp, codes):
    """The table bootstrap_scores / bootstrap_trees count for a code matrix."""
    eng = sp.engine
    if codes.shape[0] <= eng.NARROW_MAX_TAXA:
        return eng.count_patterns(eng.pack(codes))
    return eng.count_patterns_wide(*eng.pack_wide(codes))


def names_for(n, seed):
    """Leaf names in a shuffled sort order: the smallest name is not in row 0."""
    perm = np.random.default_rng(seed).permutation(n)
    return [f"x{int(p):02d}" for p in perm]


def hashed_scores(ma, mb, per_table):
    a = ma.cpu().numpy().view(np.uint64)
    b = mb.cpu().numpy().view(np.uint64)
    r = (np.arange(len(a), dtype=np.uint64) // np.uint64(per_table))
    with np.errstate(over="ignore"):
        h = (a * np.uint64(0x9E3779B97F4A7C15)) ^ (b * np.uint64(0xC2B2AE3D27D4EB4F)) ^ (r * np.uint64(0x94D049BB133111EB))
    v = ((h >> np.uint64(40)) % np.uint64(5)).astype(np.float64)
    return torch.from_numpy(v).to(ma.device)


@pytest.mark.parametrize("n,reps", [(2, 5), (3, 40), (4, 40), (5, 40), (12, 24), (33, 6), (64, 3)])
def test_lockstep_equals_restatement_with_ties(sp, n, reps):
    taxa = names_for(n, n)
    first = min(range(n), key=lambda i: taxa[i])
    masks, scores = sp.engine.erickson_lockstep(n, reps, first, hashed_scores)
    assert masks.shape == (reps, max(n - 2, 0)) and scores.shape == masks.shape
    masks = masks.cpu().numpy().view(np.uint64)
    scores = scores.cpu().numpy()
    index = {t: i for i, t in enumerate(taxa)}
    for r in range(reps):
        def score_many(splits):
            return [ER.hashed_score(ER.mask_of(a, index), ER.mask_of(b, index), r) for a, b in splits]

        chosen, trace = ER.agglomerate(taxa, score_many)
        assert [ER.split_of_mask(int(m), taxa) for m in masks[r]] == chosen, r
        assert [min(t.values()) for t in trace] == scores[r].tolist()


def random_masks(n, count, rng):
    ma = np.zeros(count, np.uint64)
    for s in range(count):
        a = int(rng.integers(1, n))
        side = rng.choice(n, size=a, replace=False)
        ma[s] = sum(1 << int(t) for t in side)
    full = np.uint64((1 << n) - 1) if n < 64 else np.uint64(2 ** 64 - 1)
    return ma, full & ~ma


@pytest.mark.parametrize("n", [12, 20, 33, 43, 44, 64])
def test_multi_table_scorer_equals_single_table(sp, n):
    eng = sp.engine
    codes = BI.simulate_codes(n + n % 2, 0.1, "JC", 5_000, n)[:n]  # balanced trees have an even number of leaves
    tables = list(eng.bootstrap_tables(counted(sp, codes), 3, SEED))
    per = 97
    rng = np.random.default_rng(n)
    stack = eng.SubflattenTables(n, len(tables))
    ma_all, mb_all, ref = [], [], []
    for i, tb in enumerate(tables):
        stack.add(i, tb)
        ma, mb = random_masks(n, per, rng)
        ma_all.append(ma)
        mb_all.append(mb)
        ref.append(eng.subflatten_scores(eng.pair_tables_from_table(tb, as_counts=True), ma, mb).cpu().numpy())
    dev = eng.device()
    ma = torch.from_numpy(np.concatenate(ma_all).view(np.int64)).to(dev)
    mb = torch.from_numpy(np.concatenate(mb_all).view(np.int64)).to(dev)
    got = eng.subflatten_scores_multi(stack, ma, mb, per).cpu().numpy()
    ref = np.concatenate(ref)
    assert not np.isnan(ref).any()
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))


@pytest.mark.parametrize("n,sites", [(8, 20_000), (20, 20_000), (40, 10_000), (64, 5_000)])
def test_scores_tie_to_bootstrap_scores(sp, n, sites):
    eng = sp.engine
    codes = BI.simulate_codes(n, 0.1, "JC", sites, n + 1)
    taxa = names_for(n, n + 1)
    first = min(range(n), key=lambda i: taxa[i])
    reps = 2
    table = counted(sp, codes)
    masks, scores = eng.bootstrap_tree_masks(table, reps, SEED, first)
    assert masks.shape == (reps + 1, n - 2)
    assert not np.isnan(scores).any()  # the step kernel orders NaN as +inf; scores of a table with sites are never NaN
    index = {t: i for i, t in enumerate(taxa)}
    full = (1 << n) - 1
    for b, tb in enumerate(eng.bootstrap_tables(table, reps, SEED)):
        row = b + 1
        # every chosen split, canonical orientation, in position form: its bootstrap_scores score, bit for bit
        canon = []
        for m in masks[row]:
            m = int(m)
            a = m if m >> first & 1 else full & ~m
            canon.append(([i for i in range(n) if a >> i & 1], [i for i in range(n) if not a >> i & 1]))
        bs = sp.batch.bootstrap_scores(codes, canon, sp.Method.subflattening, replicates=reps, seed=SEED)[b]
        assert np.array_equal(bs.view(np.uint64), scores[row].view(np.uint64))
        # every pick is the first minimum of its step under the replicate's scores
        pt = eng.pair_tables_from_table(tb, as_counts=True)

        def score_many(splits):
            ma = np.array([ER.mask_of(s[0], index) for s in splits], dtype=np.uint64)
            mb = np.array([ER.mask_of(s[1], index) for s in splits], dtype=np.uint64)
            return eng.subflatten_scores(pt, ma, mb).cpu().numpy().tolist()

        chosen, trace = ER.agglomerate(taxa, score_many)
        assert [ER.split_of_mask(int(m), taxa) for m in masks[row]] == chosen
        assert [min(t.values()) for t in trace] == scores[row].tolist()


def informative(tree):
    return {frozenset(s) for s in tree if min(len(s[0]), len(s[1])) >= 2}


def mapping_of(keys, counts, n):
    """{pattern string: count / N} of a table's keys and counts."""
    from tests.test_gpu_bootstrap import key_codes
    codes = key_codes(keys, n)
    N = counts.sum()
    lut = np.array(list("ACGT"))
    return {"".join(lut[c]): int(k) / N for c, k in zip(codes, counts)}


@pytest.mark.parametrize("n", [12, 40])
def test_trees_agree_with_erickson_svd(sp, n):
    from splitp_b200.alignment import Alignment
    from splitp_b200.phylogenetics import erickson_SVD
    eng = sp.engine
    codes = BI.simulate_codes(n, 0.05, "JC", 50_000, 7 * n)
    taxa = names_for(n, 3 * n)
    aln = BI.codes_to_sequences(codes, taxa)
    res = sp.batch.bootstrap_trees(aln, replicates=3, seed=SEED)
    table = counted(sp, codes)
    cases = [(res.tree, table)] + [(res.replicate_trees[b], tb) for b, tb in enumerate(eng.bootstrap_tables(table, 3, SEED))]
    for tree, tb in cases:
        if isinstance(tb, eng.WideTable):
            keys, counts = tb.compact()
        else:
            keys, counts = tb.keys, tb.counts
        keys = keys.cpu().numpy().view(np.uint64)
        counts = counts.cpu().numpy().view(np.uint32).astype(np.int64)
        trace = []
        host = erickson_SVD(Alignment(mapping_of(keys, counts, n), taxa), taxa=taxa, method=sp.Method.subflattening, trace=trace)
        assert informative(tree) == informative(host)
        for got, want, step in zip(tree, host, trace):
            vals = sorted(step["scores"].values())
            if len(vals) > 1 and vals[1] - vals[0] > 1e-6 * abs(vals[1]):
                assert got == want
            elif got != want:
                break  # a near-tie decided the other way: the clusters differ from here on


def true_splits(n):
    parent, names = BI.balanced_parents(n)
    taxa = BI.taxa_of(names)
    leaves = {node: {name} for node, name in names.items()}
    for node in range(len(parent) - 1, 0, -1):
        leaves.setdefault(parent[node], set()).update(leaves.setdefault(node, set()))
    out = set()
    for node in range(1, len(parent)):
        side = leaves[node]
        if 2 <= len(side) <= n - 2:
            a = tuple(sorted(side))
            b = tuple(sorted(set(taxa) - side))
            out.add(tuple(sorted((a, b))))
    return taxa, sorted(out)


def test_support_of_a_well_resolved_tree(sp):
    n = 20
    codes = BI.simulate_codes(n, 0.05, "JC", 100_000, 11)
    taxa, truth = true_splits(n)
    res = sp.batch.bootstrap_trees(codes, replicates=20, seed=SEED, splits=truth)
    assert (res.support == 1.0).all(), res.support
    assert informative(res.tree) == {frozenset(s) for s in truth}
    # support of the tree's own splits recomputed on the host from replicate_trees
    own = sp.batch.bootstrap_trees(codes, replicates=20, seed=SEED)
    assert own.tree == res.tree and own.replicate_trees == res.replicate_trees
    reps = [{frozenset(s) for s in t} for t in own.replicate_trees]
    want = [sum(frozenset(s) in r for r in reps) / len(reps) for s in own.tree]
    assert own.support.dtype == np.float64 and own.support.tolist() == want


def test_reproducible_and_group_independent(sp, monkeypatch):
    codes = BI.simulate_codes(16, 0.1, "JC", 20_000, 5)
    bt = sp.batch.bootstrap_trees
    a = bt(codes, replicates=10, seed=3)
    b = bt(codes, replicates=10, seed=3)
    assert a.tree == b.tree and a.replicate_trees == b.replicate_trees and np.array_equal(a.support, b.support)
    with monkeypatch.context() as mp:
        mp.setattr(sp.engine, "BOOTSTRAP_TREES_BATCH_BYTES", 1)  # one table per lockstep group
        c = bt(codes, replicates=10, seed=3)
    assert c.tree == a.tree and c.replicate_trees == a.replicate_trees and np.array_equal(c.support, a.support)
    d = bt(codes, replicates=5, seed=3)
    assert d.tree == a.tree and d.replicate_trees == a.replicate_trees[:5]
    assert len(a.tree) == 14 and len(a.replicate_trees) == 10


def test_edge_cases(sp):
    codes = BI.simulate_codes(4, 0.1, "JC", 2_000, 1)[:2]
    res = sp.batch.bootstrap_trees(codes, replicates=3, taxa=["q", "p"])
    assert res.tree == [] and res.replicate_trees == [[], [], []] and res.support.shape == (0,)
    res = sp.batch.bootstrap_trees(codes, replicates=3, taxa=["q", "p"], splits=[(["p"], ["q"])])
    assert res.support.tolist() == [0.0]
    gaps = np.zeros((6, 500), dtype=np.uint8)
    gaps[0] = 255  # no usable site
    with pytest.raises(ValueError, match="usable site"):
        sp.batch.bootstrap_trees(gaps, replicates=2)
