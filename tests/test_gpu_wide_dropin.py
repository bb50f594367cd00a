"""GPU tests of the drop-in functions on {pattern: value} mappings of 32..64 taxa (128-bit pattern keys): pair tables
(csrc/wide.cu spb_pair_tables_wide), subflattening + split_score, flattening (spb_project_wide), Alignment.sub_alignment
and erickson_SVD(Method.subflattening), against the oracle and dict-based restatements.  Run with `-m gpu`.

Tolerances:
  * pair tables from counts, flattenings, sub-alignments of counts: BIT-EXACT.
  * pair tables from probabilities: rtol = atol = 1e-14 (summation order differs from the oracle's).
  * subflattening entries from probabilities: rtol = 1e-12, atol = 1e-13 (entries are signed sums that can cancel to 0).
  * scores: rel <= max(1e-9, 64 * eps / score^2), as in test_gpu_parity.py.
  * sub-alignment sums of probabilities: rel 1e-13.
"""
import collections
import itertools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
SIZES = {33: ("random", 6000), 40: ("simulated", 4000), 64: ("simulated", 8000)}


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    return splitp_b200


def random_codes(n, N, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 4, size=(n, 48))  # a few frequent patterns plus noise: counts from 1 to hundreds
    codes = base[:, rng.integers(0, 48, size=N)]
    mut = rng.random((n, N)) < 0.02
    codes = np.where(mut, rng.integers(0, 4, size=(n, N)), codes).astype(np.uint8)
    codes[rng.random((n, N)) < 0.0005] = 255  # a few unusable sites
    return codes


def names(n):
    from splitp_b200.trees import _leaf_name
    return [_leaf_name(i, n) for i in range(n)]


class Case:
    def __init__(self, sp, n):
        kind, N = SIZES[n]
        self.tree = None
        if kind == "random":
            self.codes, self.taxa = random_codes(n, N, seed=n), names(n)
        else:
            self.tree = sp.trees.balanced_tree(n, 0.1)
            self.codes = sp.simulation.simulate_codes(self.tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=n).cpu().numpy()
            self.taxa = list(self.tree.taxa)
        from splitp_b200.parsers import fasta
        seqs = collections.OrderedDict((t, "".join("ACGTN"[min(int(c), 4)] for c in row)) for t, row in zip(self.taxa, self.codes))
        self.counts, self.usable = fasta.get_pattern_counts(seqs)
        self.probs = {p: c / self.usable for p, c in self.counts.items()}  # pattern_counts_to_probs (fasta.py:66-70)
        self.n = n


@pytest.fixture(scope="module")
def cases(sp):
    return {n: Case(sp, n) for n in SIZES}


def assert_score(got, ref):
    got, ref = float(got), float(ref)
    tol = max(1e-9, 64 * EPS / max(ref * ref, 1e-300))
    assert abs(got - ref) <= tol * abs(ref), (got, ref)


def index_of(pat, idx):
    v = 0
    for t in idx:
        v = v * 4 + "ACGT".index(pat[t])
    return v


def dense_from_dict(mapping, idx_a, idx_b):
    out = np.zeros((4 ** len(idx_a), 4 ** len(idx_b)))
    for pat, val in mapping.items():
        out[index_of(pat, idx_a), index_of(pat, idx_b)] = val  # the last pattern wins a cell (constructions.py:101)
    return out


def cells_from_dict(mapping, idx_a, idx_b):
    cells = {}
    for pat, val in mapping.items():
        cells[(index_of(pat, idx_a), index_of(pat, idx_b))] = val
    return {k: v for k, v in cells.items() if v != 0}


# ---------------------------------------------------------------------------------------------
# pair tables
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", sorted(SIZES))
def test_pair_tables_from_count_mapping(sp, oracle, cases, n):
    c, eng = cases[n], sp.engine
    ref_counts, ref_usable = oracle.get_pattern_counts_wide(c.codes)
    assert list(c.counts.items()) == list(ref_counts.items()) and c.usable == ref_usable  # first-occurrence order
    table = eng.table_from_mapping(c.counts)
    assert isinstance(table, eng.WidePatternTable) and table.n == n
    pt = eng.pair_tables_from_table(table)
    planes = eng.pair_tables_from_alignment(eng.pack(c.codes), as_counts=True)
    ref, usable = oracle.pair_tables_from_codes(c.codes, as_counts=True)
    assert usable == c.usable
    N = pt.N.cpu().numpy()
    np.testing.assert_array_equal(N, planes.N.cpu().numpy())
    np.testing.assert_array_equal(N, ref.astype(np.float64))
    np.testing.assert_array_equal(pt.T.cpu().numpy(), planes.T.cpu().numpy())
    assert float(pt.total.item()) == float(planes.total.item()) == float(usable)
    again = eng.pair_tables_from_table(eng.table_from_mapping(dict(c.counts)))  # a fresh table: no cache hit
    assert again.N.cpu().numpy().tobytes() == N.tobytes()


@pytest.mark.parametrize("n", sorted(SIZES))
def test_pair_tables_from_probabilities(sp, oracle, cases, n):
    c, eng = cases[n], sp.engine
    pt = eng.pair_tables_from_table(eng.table_from_mapping(c.probs))
    ref, _ = oracle.pair_tables_from_codes(c.codes)
    np.testing.assert_allclose(pt.N.cpu().numpy(), ref, rtol=1e-14, atol=1e-14)
    again = eng.pair_tables_from_table(eng.table_from_mapping(dict(c.probs)))
    assert again.N.cpu().numpy().tobytes() == pt.N.cpu().numpy().tobytes()  # bitwise reproducible
    assert again.T.cpu().numpy().tobytes() == pt.T.cpu().numpy().tobytes()


def test_narrow_table_through_the_wide_kernels(sp, oracle):
    """A 20-taxon table with its keys widened to {key, 0}: the wide kernels give the narrow results bit for bit."""
    eng = sp.engine
    codes = random_codes(20, 20_000, seed=3)
    counts = oracle.get_pattern_counts_wide(codes)[0]
    narrow = eng.table_from_mapping(counts)
    assert isinstance(narrow, eng.PatternTable)
    keys = torch.stack([narrow.keys, torch.zeros_like(narrow.keys)], dim=1).contiguous()
    wide = eng.WidePatternTable(20, keys, narrow.values)
    a, b = eng.pair_tables_from_table(wide), eng.pair_tables_from_table(narrow)
    for x, y in ((a.N, b.N), (a.T, b.T), (a.total, b.total)):
        np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy())
    for ia, ib in (([0, 5, 3], list(range(6, 20))), ([19, 2], [4, 7, 1]), (list(range(20)), [])):
        for x, y in zip(eng.flatten_coo(wide, ia, ib), eng.flatten_coo(narrow, ia, ib)):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy())


# ---------------------------------------------------------------------------------------------
# subflattening + split_score
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", sorted(SIZES))
def test_subflattening_every_side_size(sp, oracle, cases, n):
    c = cases[n]
    ref_tables, _ = oracle.pair_tables_from_codes(c.codes)
    total = ref_tables[0, 0].trace()
    aln = sp.Alignment(c.probs, c.taxa)
    rng = np.random.default_rng(n)
    for a in range(1, n // 2 + 1):
        perm = rng.permutation(n)
        ia, ib = sorted(perm[:a].tolist()), sorted(perm[a:].tolist())
        if a % 2:
            ia = ia[::-1]  # the order of a side is the row order of the subflattening
        split = ([c.taxa[i] for i in ia], [c.taxa[i] for i in ib])
        S = sp.subflattening(split, aln)
        ref = oracle.subflattening_from_tables(ref_tables, total, ia, ib)
        assert S.shape == ref.shape == (3 * a + 1, 3 * (n - a) + 1)
        np.testing.assert_allclose(S, ref, rtol=1e-12, atol=1e-13)
        if a > 1:  # a 4-row matrix has at most 4 singular values: score 0 against LAPACK's rounding noise
            assert_score(sp.split_score(S), oracle.split_score(ref))


def test_subflattening_string_split_at_33_taxa(sp, oracle, cases):
    c = cases[33]
    ref_tables, _ = oracle.pair_tables_from_codes(c.codes)
    aln = sp.Alignment(c.probs, c.taxa)
    ia, ib = [3, 0, 17, 32, 9], [i for i in range(33) if i not in (3, 0, 17, 32, 9)]
    split = "".join(c.taxa[i] for i in ia) + "|" + "".join(c.taxa[i] for i in ib)
    S = sp.subflattening(split, aln)
    ref = oracle.subflattening_from_tables(ref_tables, ref_tables[0, 0].trace(), ia, ib)
    np.testing.assert_allclose(S, ref, rtol=1e-12, atol=1e-13)
    assert_score(sp.split_score(S), oracle.split_score(ref))
    with pytest.raises(KeyError):  # a taxon on neither side (__reconstruct_pattern, constructions.py:192-198)
        sp.subflattening(split[:-1], aln)
    with pytest.raises(KeyError):  # a plain dict counts '|' as a taxon (constructions.py:114-117)
        sp.subflattening(split, c.probs)
    with pytest.raises(IndexError):  # 33-taxon patterns against 34 taxa
        sp.subflattening(split + "Y", sp.Alignment(c.probs, c.taxa + ["Y"]))


# ---------------------------------------------------------------------------------------------
# flattening
# ---------------------------------------------------------------------------------------------
def _check_flattening(sp, oracle, mapping, taxa, ia, ib, dense=True):
    aln = sp.Alignment(mapping, taxa)
    split = ([taxa[i] for i in ia], [taxa[i] for i in ib])
    R = sp.flattening(split, aln, sp.FlatFormat.reduced)
    np.testing.assert_array_equal(R, oracle.flattening_reduced_from_dict(mapping, ia, ib))
    F = sp.flattening(split, aln, sp.FlatFormat.sparse)
    assert F.shape == (4 ** len(ia), 4 ** len(ib))
    assert dict(F.items()) == cells_from_dict(mapping, ia, ib)
    if dense:
        np.testing.assert_array_equal(sp.flattening(split, aln, sp.FlatFormat.dense), dense_from_dict(mapping, ia, ib))


def test_flattening_covering_split_at_40_taxa(sp, oracle, cases):
    c = cases[40]
    mapping = dict(itertools.islice(c.probs.items(), 1500))
    ia, ib = list(range(0, 40, 2)), list(range(1, 40, 2))  # 20 | 20
    _check_flattening(sp, oracle, mapping, c.taxa, ia, ib, dense=False)  # a dense 4^20 x 4^20 matrix does not fit anywhere
    ia, ib = [5, 0, 9], [1, 2, 3, 4, 6, 39]  # and a split that leaves taxa out, in all three formats
    _check_flattening(sp, oracle, mapping, c.taxa, ia, ib)


@pytest.mark.parametrize("sides", [([7, 2, 40], [63, 0, 11, 30]), ([1], [2, 3]), ([60, 61, 62, 63], [0, 1, 2])])
def test_flattening_non_covering_split_at_64_taxa(sp, oracle, cases, sides):
    c = cases[64]
    ia, ib = sides
    for mapping in (c.counts, c.probs):
        cells = {(index_of(p, ia), index_of(p, ib)) for p in mapping}
        assert len(cells) < len(mapping)  # several patterns collide on a cell: the last one wins it
        _check_flattening(sp, oracle, mapping, c.taxa, ia, ib)


def test_flattening_side_above_31_taxa_raises(sp, cases):
    c = cases[64]
    aln = sp.Alignment(c.probs, c.taxa)
    for split in ((c.taxa[:32], c.taxa[32:]), (c.taxa[:2], c.taxa[2:])):
        for fmt in (sp.FlatFormat.sparse, sp.FlatFormat.reduced, sp.FlatFormat.dense):
            with pytest.raises(NotImplementedError, match="31 taxa"):
                sp.flattening(split, aln, fmt)


# ---------------------------------------------------------------------------------------------
# Alignment.sub_alignment
# ---------------------------------------------------------------------------------------------
def restated_sub_alignment(mapping, idx):
    acc = {}
    for pat, val in mapping.items():
        sub = "".join(pat[i] for i in idx)
        acc[sub] = acc.get(sub, 0) + val  # alignment.py:26-28
    return {k: acc[k] for k in sorted(acc)}  # ascending keys = lexicographic A<C<G<T order


@pytest.mark.parametrize("keep", [10, 35])
def test_sub_alignment_of_40_taxa(sp, oracle, cases, keep):
    c = cases[40]
    rng = np.random.default_rng(keep)
    idx = sorted(rng.choice(40, size=keep, replace=False).tolist())
    sub_taxa = [c.taxa[i] for i in idx]
    for mapping in (c.counts, c.probs):
        aln = sp.Alignment(mapping, c.taxa)
        sub = aln.sub_alignment(sub_taxa[::-1])
        assert aln.sub_alignment(sub_taxa) is sub  # memoised per taxa tuple in parent order (alignment.py:11,30)
        assert sub.taxa == tuple(sub_taxa)
        ref = restated_sub_alignment(mapping, idx)
        assert list(sub.keys()) == list(ref.keys())
        if mapping is c.counts:
            assert sub.data == ref and all(type(v) is int for v in sub.values())
        else:
            got, want = np.array(list(sub.values())), np.array(list(ref.values()))
            np.testing.assert_allclose(got, want, rtol=1e-13, atol=0)
    sub = sp.Alignment(c.counts, c.taxa).sub_alignment(sub_taxa)
    a = keep // 2
    ia, ib = list(range(a)), list(range(a, keep))
    split = ([sub_taxa[i] for i in ia], [sub_taxa[i] for i in ib])
    np.testing.assert_array_equal(sp.flattening(split, sub, sp.FlatFormat.reduced),
                                  oracle.flattening_reduced_from_dict(sub.data, ia, ib))
    codes = c.codes[idx]
    ref_tables, _ = oracle.pair_tables_from_codes(codes, as_counts=True)
    S = sp.subflattening(split, sub)
    np.testing.assert_array_equal(S, oracle.subflattening_from_tables(ref_tables.astype(np.float64), float(c.usable), ia, ib))


# ---------------------------------------------------------------------------------------------
# erickson_SVD(Method.subflattening)
# ---------------------------------------------------------------------------------------------
def _leaves(cluster):
    return (cluster,) if isinstance(cluster, str) else tuple(cluster)


def restated_erickson(oracle, tables, taxa):
    """The agglomeration of phylogenetics.py:99-171 with oracle subflattenings of the oracle's pair tables and LAPACK scores."""
    pos = {t: i for i, t in enumerate(taxa)}
    total = tables[0, 0].trace()
    clusters, known, chosen = list(taxa), {}, []
    while len(chosen) < len(taxa) - 2:
        cands = []
        for pair in itertools.combinations(clusters, 2):
            joined = tuple(sorted(leaf for cl in pair for leaf in _leaves(cl)))
            rest = tuple(sorted(leaf for cl in clusters for leaf in _leaves(cl) if leaf not in joined))
            cands.append((pair, (joined, rest)))
        for _, s in cands:
            if s not in known:
                S = oracle.subflattening_from_tables(tables, total, [pos[t] for t in s[0]], [pos[t] for t in s[1]])
                known[s] = oracle.split_score(S)
        best = min(cands, key=lambda cand: known[cand[1]])
        chosen.append(tuple(sorted(best[1])))
        merged = best[1][0]
        clusters = [cl for cl in clusters if cl not in merged and not set(cl).issubset(merged)] + [merged]
    return chosen


def informative(picks):
    return {frozenset(map(frozenset, s)) for s in picks if min(len(side) for side in s) > 1}


@pytest.mark.parametrize("n", [40, 64])
def test_erickson_subflattening(sp, oracle, cases, n):
    c = cases[n]
    true = {frozenset(map(frozenset, s)) for s in c.tree.splits()}
    tables, _ = oracle.pair_tables_from_codes(c.codes)
    restated = informative(restated_erickson(oracle, tables, c.taxa))
    assert restated == true  # the sizes are chosen so that the restatement recovers the tree
    aln = sp.Alignment(c.probs, c.taxa)
    got = sp.erickson_SVD(aln, taxa=list(c.taxa), method=sp.Method.subflattening)
    assert len(got) == n - 2
    assert informative(got) == restated  # a set: near-ties between cherries make the order noise
    if n == 64:  # a plain dict: default names t0..t63, positions = their sorted order, which is the tree's taxon order here
        assert sorted(f"t{i}" for i in range(n)) == list(c.taxa)
        assert informative(sp.erickson_SVD(c.probs, method=sp.Method.subflattening)) == restated


# ---------------------------------------------------------------------------------------------
# routes that stay limited to 31 taxa
# ---------------------------------------------------------------------------------------------
def test_unsupported_wide_routes_raise(sp, cases):
    c = cases[40]
    aln = sp.Alignment(c.probs, c.taxa)
    for method in (sp.Method.flattening, sp.Method.mutual_information):
        with pytest.raises(NotImplementedError, match="31 taxa"):
            sp.erickson_SVD(aln, method=method)
    split = (c.taxa[:20], c.taxa[20:])
    with pytest.raises(NotImplementedError, match="31 taxa"):
        sp.phylogenetics.flattening_rank_k_approximation(split, aln)
    table = sp.engine.table_from_mapping(aln)
    with pytest.raises(NotImplementedError, match="31 taxa"):
        sp.engine.rank1_divergence(table, list(range(20)), list(range(20, 40)))
    with pytest.raises(NotImplementedError, match="31 taxa"):
        sp.constructions.sparse_flattening_with_banned_patterns(split, aln, c.taxa, "A", "C")
