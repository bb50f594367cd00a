"""GPU tests of the split scorers at the top of their taxon ranges, against host references.  Run with `-m gpu`.

  * Flattening scores at 13..16 taxa (batch.score_splits, Method.flattening: engine.CountScorer, dense count flattenings
    up to 6|n-6, sparse_flattening_scores for 7|7 .. 8|8) for every size class 1 .. n/2, true and random splits, on both
    sides of 32,768 distinct patterns at 15 and 16 taxa, against tests/sparse_reference.score on the host pattern counts;
    at 16 taxa also one window_scores row and one bootstrap_scores replicate, against the reference on the window's and
    the replicate's counts, and a window without usable sites.
  * Subflattening scores at 33..64 taxa against oracle.split_score(oracle.subflattening_from_tables(...)): the default
    route (triple-table warp kernel up to 43 taxa, k = 3 * 21 + 1 = 64 at 42 and 43; the staged kernels from 44 taxa,
    k up to 97), the staged entry point spb_subflatten_score at 42 and 43 taxa, non-covering splits, taxon 63 at 64 taxa,
    and the multi-table scorers fed with the pair tables of bootstrap count rows (spb_pair_tables_count_rows up to 48
    taxa, spb_pair_tables_wide above).

The alignments are simulated on the host (bench_inputs.simulate_codes: a balanced tree; odd taxon counts drop the last
leaf of the tree on n + 1 taxa).  The flattening inputs add uniformly random sites: they raise the number of distinct
patterns past 32,768 while every host eigenproblem stays a few thousand rows (a random pattern rarely joins the
connected component of the tree's patterns).

Tolerance: rel <= max(1e-9, 64 eps / score^2) (tests/test_gpu_parity.py header); a side of one taxon scores exactly 0.0.
"""
import numpy as np
import pytest

import bench_inputs as BI
from tests import sparse_reference as SR
from tests.test_gpu_bootstrap import expanded, key_codes
from tests.test_gpu_parity import assert_score, score_tol

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0x5C0E
PATTERN_EDGE = 32768  # above this many patterns the dense Gram of a 15- or 16-taxon class splits its K dimension


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401  (score_splits, window_scores, bootstrap_scores)
    return splitp_b200


def simulated(n, N, random_sites, seed, bl):
    """uint8 codes [n, N + random_sites]: N sites simulated on the balanced tree (n + 1 leaves for odd n, last row
    dropped), then random_sites uniformly random sites."""
    codes = BI.simulate_codes(n + n % 2, bl, "JC", N, seed)[:n]
    noise = np.random.default_rng(seed + 1).integers(0, 4, size=(n, random_sites), dtype=np.uint8)
    return np.ascontiguousarray(np.concatenate([codes, noise], axis=1))


def true_sides(n):
    """The shorter side (sorted positions) of every non-trivial split of the simulating tree restricted to n taxa."""
    parent, names = BI.balanced_parents(n + n % 2)
    pos = {t: i for i, t in enumerate(BI.taxa_of(names))}
    below = {v: {pos[name]} for v, name in names.items()}
    for v in range(len(parent) - 1, 0, -1):  # children are numbered after their parents
        below.setdefault(parent[v], set()).update(below[v])
    out = set()
    for v in range(1, len(parent)):
        side = below[v] - {n}
        other = set(range(n)) - side
        short = min(sorted(side), sorted(other), key=len)
        if len(short) >= 2:
            out.add(tuple(short))
    return out


def stratified(n, per_size, seed, extra=()):
    """[(side a, side b, is_true)]: for every side size 1 .. n/2 the tree's true splits of that size plus random ones,
    at least per_size in all; then the sides in `extra`."""
    rng = np.random.default_rng(seed)
    true = true_sides(n)
    out = []
    for a in range(1, n // 2 + 1):
        chosen = [s for s in sorted(true) if len(s) == a]
        want = max(per_size, len(chosen) + 2)
        while len(chosen) < want:
            side = tuple(sorted(rng.choice(n, size=a, replace=False).tolist()))
            if side not in chosen:
                chosen.append(side)
        out += [(list(s), [t for t in range(n) if t not in s], s in true) for s in chosen]
    out += [(sorted(s), [t for t in range(n) if t not in s], False) for s in extra]
    return out


# ---------------------------------------------------------------------------------------------
# A. flattening scores at 13..16 taxa
# ---------------------------------------------------------------------------------------------
def host_patterns(codes):
    """(codes of every distinct pattern [P, n], counts [P]) of a code matrix."""
    pats, counts = np.unique(codes.T, axis=0, return_counts=True)
    return pats, counts


def flattening_reference(pats, counts, ia, ib):
    """tests/sparse_reference.score of the count flattening of (ia | ib)."""
    def side(idx):
        return pats[:, idx].astype(np.int64) @ (4 ** np.arange(len(idx), dtype=np.int64))
    return SR.score(side(ia), side(ib), counts.astype(np.float64))


def check_flattening(got, pats, counts, picks):
    worst = 0.0
    for s, (ia, ib, _) in enumerate(picks):
        if min(len(ia), len(ib)) == 1:
            assert got[s] == 0.0, (ia, got[s])
            continue
        ref = flattening_reference(pats, counts, ia, ib)
        assert_score(got[s], ref)
        worst = max(worst, abs(got[s] - ref) / ref / score_tol(ref))
    return worst


# (n, simulated sites, random sites, P above the 32,768-pattern edge or None when n < 15)
FLATTENING_CASES = [(13, 20_000, 2_000, None), (14, 20_000, 2_000, None), (15, 40_000, 8_000, False),
                    (15, 60_000, 33_000, True), (16, 40_000, 8_000, False), (16, 60_000, 30_000, True)]


@pytest.mark.parametrize("n,N,random_sites,above", FLATTENING_CASES)
def test_dense_flattening_scores_against_host_reference(sp, n, N, random_sites, above):
    """score_splits(Method.flattening) at 13..16 taxa, every size class, against the connected-component reference."""
    codes = simulated(n, N, random_sites, seed=100 + n, bl=0.02)
    pats, counts = host_patterns(codes)
    if above is not None:
        assert (len(counts) > PATTERN_EDGE) == above, len(counts)
    picks = stratified(n, 3, seed=n)
    got = sp.batch.score_splits(codes, [(ia, ib) for ia, ib, _ in picks], sp.Method.flattening)
    worst = check_flattening(got, pats, counts, picks)
    print(f"flattening n={n} P={len(counts)}: {len(picks)} splits, worst error = {worst:.3f} x tolerance")


def test_window_and_bootstrap_flattening_scores_at_16_taxa(sp):
    """window_scores and bootstrap_scores go through the same scorer as score_splits: one window row and one replicate
    of the 16-taxon alignment with more than 32,768 patterns, every size class, against the reference on the window's
    counts and on the replicate's counts."""
    eng = sp.engine
    n = 16
    codes = simulated(n, 60_000, 30_000, seed=116, bl=0.02)
    picks = [p for p in stratified(n, 1, seed=17) if not p[2]]
    picks = [next(p for p in picks if len(p[0]) == a) for a in range(1, n // 2 + 1)]
    splits = [(ia, ib) for ia, ib, _ in picks]
    b, e = 1_000, codes.shape[1]
    row = sp.batch.window_scores(codes, splits, [[b, e]], sp.Method.flattening)
    assert row.shape == (1, len(splits))
    pats, counts = host_patterns(codes[:, b:e])
    assert len(counts) > PATTERN_EDGE
    check_flattening(row[0], pats, counts, picks)
    got = sp.batch.bootstrap_scores(codes, splits, sp.Method.flattening, replicates=1, seed=SEED)
    table = eng.count_patterns(eng.pack(codes))
    rep = eng.bootstrap_counts(table, 0, 1, SEED)[0].cpu().numpy().view(np.uint32).astype(np.int64)
    keys = table.keys.cpu().numpy().view(np.uint64)
    drawn = rep > 0
    check_flattening(got[0], key_codes(keys[drawn], n), rep[drawn], picks)


def test_window_without_usable_sites_at_16_taxa(sp):
    """An empty window scores as an all-zero count flattening in both routes of the scorer: 0.0 for a one-taxon side,
    NaN for the dense classes and for the classes scored from the pattern list."""
    n = 16
    codes = simulated(n, 3_000, 0, seed=160, bl=0.05)
    codes[5, 1_000:1_100] = 255
    splits = [(list(range(a)), list(range(a, n))) for a in (1, 3, 6, 7, 8)]
    got = sp.batch.window_scores(codes, splits, [[1_000, 1_100], [0, 1_000]], sp.Method.flattening)
    assert got[0, 0] == 0.0 and np.isnan(got[0, 1:]).all()
    assert np.isfinite(got[1]).all()


# ---------------------------------------------------------------------------------------------
# B. subflattening scores at 33..64 taxa
# ---------------------------------------------------------------------------------------------
SUBFLATTENING_TAXA = [33, 42, 43, 44, 48, 49, 64]


def subflattening_picks(n, seed):
    """>= 8 splits per side size 1 .. n/2, true splits included; at 64 taxa also sides with and without taxon 63."""
    extra = ()
    if n == 64:
        extra = [(63,), (0, 63), (1, 2, 63), tuple(range(48, 64)), tuple(range(32, 64)), tuple(range(31)) + (63,),
                 tuple(range(2, 20)), tuple(range(0, 62, 2))]
    return stratified(n, 8, seed, extra)


def check_subflattening(got, picks, reference, label):
    worst = 0.0
    for s, (ia, ib, _) in enumerate(picks):
        if min(len(ia), len(ib)) == 1:
            assert got[s] == 0.0, (label, ia, got[s])
            continue
        ref = reference(ia, ib)
        assert_score(got[s], ref)
        worst = max(worst, abs(got[s] - ref) / ref / score_tol(ref))
    return worst


@pytest.fixture(scope="module")
def wide_inputs():
    """n -> code matrix [n, 20,000]."""
    return {n: simulated(n, 20_000, 0, seed=200 + n, bl=0.05) for n in SUBFLATTENING_TAXA}


@pytest.mark.parametrize("n", SUBFLATTENING_TAXA)
def test_subflatten_scores_against_oracle(sp, oracle, wide_inputs, n):
    """engine.subflatten_scores on the pair tables of the alignment (probabilities), both mask orders, and at 42 and 43
    taxa the staged entry point spb_subflatten_score, against the oracle; then splits whose side B is a strict subset of
    the complement of side A."""
    eng = sp.engine
    codes = wide_inputs[n]
    pt = eng.pair_tables_from_alignment(eng.pack(codes, want_sm=False))
    tables, usable = oracle.pair_tables_from_codes(codes)
    assert usable == codes.shape[1]
    picks = subflattening_picks(n, seed=n)
    ma, mb = eng.masks_from_splits([(ia, ib) for ia, ib, _ in picks])

    def reference(ia, ib):
        return oracle.split_score(oracle.subflattening_from_tables(tables, 1.0, ia, ib))
    got = eng.subflatten_scores(pt, ma, mb).cpu().numpy()
    worst = check_subflattening(got, picks, reference, "default")
    swapped = eng.subflatten_scores(pt, mb, ma).cpu().numpy()
    worst = max(worst, check_subflattening(swapped, [(ib, ia, t) for ia, ib, t in picks], reference, "swapped"))
    if n in (42, 43):  # below 44 taxa the engine routes to the triple-table kernel: call the staged one directly
        dev = eng.device()
        da, db = (torch.from_numpy(m.view(np.int64)).to(dev) for m in (ma, mb))
        staged = torch.empty(len(picks), dtype=torch.float64, device=dev)
        eng.call("spb_subflatten_score", eng._p(pt.T), eng._p(pt.total), pt.n, eng._p(da), eng._p(db), len(picks), eng._p(staged),
                 eng._st())
        worst = max(worst, check_subflattening(staged.cpu().numpy(), picks, reference, "staged"))
    rng = np.random.default_rng(n + 1)
    partial = []
    for ia, ib, _ in picks:
        if len(ia) >= 2 and len(ib) >= 3:
            keep = sorted(rng.choice(ib, size=int(rng.integers(2, len(ib))), replace=False).tolist())
            partial.append((ia, keep, False))
    if n == 64:
        partial += [([5, 9, 63], [0, 1, 2, 3], False), ([0, 1, 2], [60, 61, 62, 63], False),
                    (list(range(32, 64)), list(range(0, 31)), False)]
    pa, pb = eng.masks_from_splits([(ia, ib) for ia, ib, _ in partial])
    got = eng.subflatten_scores(pt, pa, pb).cpu().numpy()
    worst = max(worst, check_subflattening(got, partial, reference, "non-covering"))
    n_true = sum(t for _, _, t in picks)
    assert n_true >= len(true_sides(n)) > 0
    print(f"subflatten n={n}: {len(picks)} + {len(partial)} non-covering splits, {n_true} true, "
          f"worst error = {worst:.3f} x tolerance")


@pytest.mark.parametrize("n", SUBFLATTENING_TAXA)
def test_subflatten_scores_multi_against_oracle(sp, oracle, wide_inputs, n):
    """subflatten_scores_multi on the SubflattenTables of three bootstrap replicates (bootstrap_group_tables: the pair
    tables of their count rows) against the oracle on each replicate's pair tables of counts."""
    eng = sp.engine
    codes = wide_inputs[n]
    R = 3
    table = eng.count_patterns_wide(*eng.pack_wide(codes))
    stack = eng.bootstrap_group_tables(eng.bootstrap_sources([table], [SEED]), R, 0, R, n, own=False)
    picks = subflattening_picks(n, seed=n + 2)
    K = len(picks)
    ma, mb = eng.masks_from_splits([(ia, ib) for ia, ib, _ in picks])
    dev = eng.device()
    da, db = (torch.from_numpy(m.view(np.int64)).to(dev) for m in (ma, mb))
    got = eng.subflatten_scores_multi(stack, da.repeat(R), db.repeat(R), K).view(R, K).cpu().numpy()
    keys, _ = table.compact()
    keys = keys.cpu().numpy().view(np.uint64)
    rows = eng.bootstrap_counts(table, 0, R, SEED).cpu().numpy().view(np.uint32).astype(np.int64)
    worst = 0.0
    for r in range(R):
        tables, usable = oracle.pair_tables_from_codes(expanded(keys, rows[r], n), as_counts=True)
        assert usable == codes.shape[1]

        def reference(ia, ib, tables=tables, usable=usable):
            return oracle.split_score(oracle.subflattening_from_tables(tables, usable, ia, ib))
        worst = max(worst, check_subflattening(got[r], picks, reference, f"replicate {r}"))
    print(f"subflatten multi n={n}: {R} replicates x {K} splits, worst error = {worst:.3f} x tolerance")
