"""GPU tests of the sparse flattening route (csrc/sparse.cu, engine.sparse_flattening_scores): the F (F^T Q) product kernels,
the small Gram from the CSC, scores against the host reference of tests/sparse_reference.py at 12 to 64 taxa, closed forms
and hard spectra, agreement with the dense routes, and the public routes that use it.  Run with `-m gpu`.

Tolerances: products and small Grams of integer values are BIT-EXACT; scores rel <= max(1e-9, 64 * eps / score^2), as in
test_gpu_parity.py.
"""
import itertools
import os
import sys
import warnings

import numpy as np
import pytest
import scipy.sparse

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sparse_reference  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    return splitp_b200


def assert_score(got, ref):
    got, ref = float(got), float(ref)
    tol = max(1e-9, 64 * EPS / max(ref * ref, 1e-300))
    assert abs(got - ref) <= tol * max(abs(ref), 1e-300) or (ref == 0.0 and got == 0.0), (got, ref)


def simulated_codes(sp, n, N, seed, bl=0.1):
    tree = sp.trees.balanced_tree(n, bl)
    codes = sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=seed).cpu().numpy().astype(np.uint8)
    return tree, codes


def host_patterns(codes):
    """(U uint8 [P, n], counts float64 [P]) of a code matrix [n, N] (codes 0..3 only)."""
    U, cnt = np.unique(codes.T, axis=0, return_counts=True)
    return U, cnt.astype(np.float64)


def side_ids(U, idx):
    if len(idx) == 0:
        return np.zeros(len(U), dtype=np.int64)
    return np.unique(U[:, list(idx)], axis=0, return_inverse=True)[1].reshape(-1)


def ref_score(U, cnt, ia, ib):
    return sparse_reference.score(side_ids(U, ia), side_ids(U, ib), cnt)


def random_splits(n, sizes, per, seed):
    rng = np.random.default_rng(seed)
    out = []
    for a in sizes:
        for _ in range(per):
            perm = rng.permutation(n)
            out.append((sorted(perm[:a].tolist()), sorted(perm[a:].tolist())))
    return out


def plan(sp, rows, cols, vals):
    eng = sp.engine
    dev = eng.device()
    r, c = torch.as_tensor(rows, dtype=torch.int64, device=dev), torch.as_tensor(cols, dtype=torch.int64, device=dev)
    R, C = int(r.max()) + 1, int(c.max()) + 1
    return eng.SparsePlan(r, c, R, C, torch.as_tensor(vals, dtype=torch.float64, device=dev))


def run_product(sp, plans, k, Q):
    eng = sp.engine
    a = eng.sparse_batch_arrays(plans, k)
    B = len(plans)
    ws = eng._empty(int(eng.lib.spb_sparse_product_ws(k, B, a["ncols"], a["nnz"])), torch.float64)
    Qd = torch.from_numpy(Q).to(eng.device())
    AQ = torch.full_like(Qd, float("nan"))
    eng.call("spb_sparse_product", eng._p(a["row_off"]), eng._p(a["row_col"]), eng._p(a["row_val"]), eng._p(a["col_off"]),
             eng._p(a["col_row"]), eng._p(a["col_val"]), a["ncols"], a["nnz"], k, B, eng._p(Qd), eng._p(AQ), eng._p(ws), eng._st())
    return AQ.cpu().numpy()


def unique_pairs(rows, cols, rng, vmax=6):
    key = np.unique(rows.astype(np.int64) * (1 << 32) + cols)
    return key >> 32, key & 0xFFFFFFFF, rng.integers(1, vmax, size=len(key)).astype(np.float64)


def product_cases():
    rng = np.random.default_rng(1)
    P = 300_000
    long_rows = unique_pairs(rng.integers(0, 16, P), rng.integers(0, 100_000, P), rng)                 # 16 x 1e5: long segments
    perm = rng.permutation(100_000)
    extra = rng.integers(0, 100_000, 2000)
    near_perm = unique_pairs(np.concatenate([np.arange(100_000), extra]),
                             np.concatenate([perm, rng.integers(0, 100_000, 2000)]), rng)          # 1e5 x 1e5 near-permutation
    rand = unique_pairs(rng.integers(0, 3000, 60_000), rng.integers(0, 5000, 60_000), rng)            # random sparse
    return {"long": long_rows, "perm": near_perm, "random": rand}


# ---------------------------------------------------------------------------------------------
# 1. product kernel
# ---------------------------------------------------------------------------------------------
def test_sparse_product_exact_and_reproducible(sp):
    cases = product_cases()
    rng = np.random.default_rng(2)
    for name, (r, c, v) in cases.items():
        p = plan(sp, r, c, v)
        k = int(r.max()) + 1
        Q = rng.integers(-8, 9, size=(1, 8, k)).astype(np.float64)
        got = run_product(sp, [p], k, Q)
        F = scipy.sparse.csr_matrix((v, (r, c)), shape=(k, int(c.max()) + 1))
        want = (F @ (F.T @ Q[0].T)).T
        assert np.array_equal(got[0], want), name
        assert np.array_equal(run_product(sp, [p], k, Q), got), name  # bitwise reproducible
    # a batch of two matrices of different row counts: rows past a matrix's own count stay zero
    (r1, c1, v1), (r2, c2, v2) = cases["random"], cases["long"]
    k = int(r1.max()) + 1
    Q = rng.integers(-8, 9, size=(2, 8, k)).astype(np.float64)
    got = run_product(sp, [plan(sp, r1, c1, v1), plan(sp, r2, c2, v2)], k, Q)
    for b, (r, c, v) in enumerate([(r1, c1, v1), (r2, c2, v2)]):
        F = scipy.sparse.csr_matrix((v, (r, c)), shape=(k, int(c.max()) + 1))
        assert np.array_equal(got[b], (F @ (F.T @ Q[b].T)).T)


# ---------------------------------------------------------------------------------------------
# 2. small Gram
# ---------------------------------------------------------------------------------------------
def sparse_gram(sp, plans, k):
    eng = sp.engine
    a = eng.sparse_batch_arrays(plans, k)
    B, maxc = len(plans), max(p.C for p in plans)
    G = eng._empty((B, k, k), torch.float64)
    ws = eng._empty(max(int(eng.lib.spb_sparse_gram_small_ws(k, B, maxc)), 1), torch.float64)
    eng.call("spb_sparse_gram_small", eng._p(a["col_off"]), eng._p(a["col_row"]), eng._p(a["col_val"]), eng._p(a["colbase"]), k, B,
             maxc, eng._p(G), eng._p(ws), eng._st())
    return G.cpu().numpy()


def test_small_gram_exact_against_numpy(sp):
    rng = np.random.default_rng(3)
    mats = [unique_pairs(rng.integers(0, k, nnz), rng.integers(0, cols, nnz), rng, vmax=300)
            for k, cols, nnz in ((128, 40_000, 200_000), (16, 100_000, 100_000), (70, 9, 500))]
    plans = [plan(sp, r, c, v) for r, c, v in mats]
    G = sparse_gram(sp, plans, 128)
    for b, (r, c, v) in enumerate(mats):
        F = scipy.sparse.csr_matrix((v, (r, c)), shape=(128, int(c.max()) + 1)).toarray()
        assert np.array_equal(G[b], F @ F.T), b
    assert np.array_equal(sparse_gram(sp, plans, 128), G)


def test_small_gram_matches_count_scorer_and_thin_wide_gram(sp):
    eng = sp.engine
    _, codes = simulated_codes(sp, 12, 200_000, seed=12)
    table = eng.count_patterns(eng.pack(codes))
    cs = eng.CountScorer(table)
    for ia, ib in (([0, 5, 9], [1, 2, 3, 4, 6, 7, 8, 10, 11]), ([3, 4], [0, 1, 2, 5, 6, 7, 8, 9, 10, 11])):
        G, R = cs.gram(ia, ib)
        used = torch.unique(eng.flatten_coo(table, ia, ib)[0]).cpu().numpy()
        p = eng.sparse_plan(table, ia, ib)
        assert p.k == len(used)
        got = sparse_gram(sp, [p], p.k)[0]
        assert np.array_equal(got, G[:R, :R].cpu().numpy()[np.ix_(used, used)])
    _, codes = simulated_codes(sp, 64, 50_000, seed=64)
    wide, valid, n, N = eng.pack_wide(codes)
    wt = eng.count_patterns_wide(wide, valid, n, N)
    keys, counts = wt.compact()
    wtab = eng.WidePatternTable(n, keys, counts.to(torch.float64))
    for side in ([5, 17, 40], [0, 63]):
        a = len(side)
        Gt = eng._empty(4 ** (2 * a), torch.float64)
        eng.call("spb_thin_gram_wide", eng._p(wt.hkeys), eng._p(wt.hcounts), wt.cap, eng._p(wt.special), n, bytes(side), a, eng._p(Gt),
                 eng._st())
        Gt = Gt[:4 ** (2 * a)].reshape(4 ** a, 4 ** a).cpu().numpy()
        used = torch.unique(eng.project_keys(wtab, side)).cpu().numpy()
        p = eng.sparse_plan(wtab, side, [t for t in range(n) if t not in side])
        assert p.k == len(used)
        assert np.array_equal(sparse_gram(sp, [p], p.k)[0], Gt[np.ix_(used, used)])


# ---------------------------------------------------------------------------------------------
# 3. scores against the host reference
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sim20(sp):
    tree, codes = simulated_codes(sp, 20, 3000, seed=20)
    return tree, codes, *host_patterns(codes)


def true_split_positions(tree):
    pos = {t: i for i, t in enumerate(tree.taxa)}
    return [([pos[t] for t in a], [pos[t] for t in b]) for a, b in tree.splits()]


def test_scores_20_taxa_against_reference(sp, sim20):
    eng = sp.engine
    tree, codes, U, cnt = sim20
    splits = true_split_positions(tree) + random_splits(20, range(1, 11), 2, seed=21)
    table = eng.count_patterns(eng.pack(codes))
    got = eng.sparse_flattening_scores(table, splits).cpu().numpy()
    for s, (ia, ib) in enumerate(splits):
        assert_score(got[s], ref_score(U, cnt, ia, ib))


@pytest.mark.parametrize("n", [40, 64])
def test_scores_wide_against_reference(sp, n):
    eng = sp.engine
    _, codes = simulated_codes(sp, n, 2500, seed=n)
    U, cnt = host_patterns(codes)
    wide, valid, _, N = eng.pack_wide(codes)
    keys, counts = eng.count_patterns_wide(wide, valid, n, N).compact()
    table = eng.WidePatternTable(n, keys, counts.to(torch.float64))
    splits = random_splits(n, (4, 9, 16, 25, 32 if n == 64 else 20), 2, seed=n + 1)
    splits.append((list(range(n // 2)), list(range(n // 2, n))))  # 32|32 at 64 taxa
    got = eng.sparse_flattening_scores(table, splits).cpu().numpy()
    for s, (ia, ib) in enumerate(splits):
        assert_score(got[s], ref_score(U, cnt, ia, ib))


# ---------------------------------------------------------------------------------------------
# 4. closed forms and hard spectra
# ---------------------------------------------------------------------------------------------
def scored_converged(sp, rows, cols, vals):
    eng = sp.engine
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)  # an unconverged matrix warns
        out = float(eng.sparse_matrix_score(*(torch.as_tensor(x, device=eng.device()) for x in (rows, cols, vals)))[0])
    if min(len(np.unique(rows)), len(np.unique(cols))) > eng.JACOBI_MAX_K:
        assert int(eng.lib.spb_score_last_unconverged()) == 0
    return out


def test_diagonal_gram_closed_form(sp):
    rng = np.random.default_rng(5)
    for m in (60, 2000):
        v = rng.permutation(np.arange(1, m + 1)).astype(np.float64)
        idx = np.arange(m, dtype=np.int64)
        want = np.sqrt(1 - np.sort(v ** 2)[-4:].sum() / np.sum(v ** 2))
        assert_score(scored_converged(sp, idx, rng.permutation(idx), v), want)


def test_reducible_top4_in_different_components(sp):
    rng = np.random.default_rng(6)
    rows, cols, vals = [], [], []
    r0 = c0 = 0
    for scale in (9.0, 8.0, 7.0, 6.0):  # four rank-1 blocks carry the 4 largest eigenvalues
        a, b = rng.integers(1, 4, size=12), rng.integers(1, 4, size=30)
        rr, cc = np.meshgrid(np.arange(12), np.arange(30), indexing="ij")
        rows.append(r0 + rr.ravel()); cols.append(c0 + cc.ravel()); vals.append(scale * np.outer(a, b).ravel())
        r0 += 12; c0 += 30
    m = 400  # many small singletons
    rows.append(r0 + np.arange(m)); cols.append(c0 + np.arange(m)); vals.append(rng.integers(1, 5, size=m).astype(np.float64))
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    assert_score(scored_converged(sp, rows, cols, vals), sparse_reference.score(rows, cols, vals))


def test_fully_degenerate_spectrum(sp):
    m = 500
    idx = np.arange(m, dtype=np.int64)
    assert_score(scored_converged(sp, idx, idx[::-1].copy(), np.full(m, 3.0)), np.sqrt(1 - 4 / m))


# ---------------------------------------------------------------------------------------------
# 5. agreement with the dense routes
# ---------------------------------------------------------------------------------------------
def all_splits(n):
    out = []
    for mask in range(1, 1 << (n - 1)):
        a = [t for t in range(n) if mask >> t & 1]
        if 2 <= len(a) <= n - 2:
            out.append((a, [t for t in range(n) if not mask >> t & 1]))
    return out


def test_all_splits_of_12_taxa_match_count_scorer(sp):
    eng = sp.engine
    _, codes = simulated_codes(sp, 12, 100_000, seed=121)
    table = eng.count_patterns(eng.pack(codes))
    splits = all_splits(12)
    assert len(splits) == 2035
    want = eng.CountScorer(table).score_many(splits).cpu().numpy()
    got = eng.sparse_flattening_scores(table, splits).cpu().numpy()
    for g, w in zip(got, want):
        assert_score(g, w)


@pytest.mark.parametrize("n", [14, 16])
def test_sample_matches_reduced_route(sp, n):
    eng = sp.engine
    _, codes = simulated_codes(sp, n, 20_000, seed=n)
    table = eng.count_patterns(eng.pack(codes))
    splits = random_splits(n, (2, 4, 6, n // 2), 2, seed=n + 7)
    got = eng.sparse_flattening_scores(table, splits).cpu().numpy()
    for s, (ia, ib) in enumerate(splits):
        F = eng.flatten_reduced(table, ia, ib)
        want = 0.0 if min(F.shape) <= 4 else float(eng.score_matrix(F)[0])
        assert_score(got[s], want)


# ---------------------------------------------------------------------------------------------
# 6. invariances
# ---------------------------------------------------------------------------------------------
def test_counts_and_probabilities_agree_and_repeat_bitwise(sp, sim20):
    eng = sp.engine
    tree, codes, U, cnt = sim20
    splits = true_split_positions(tree) + random_splits(20, (3, 7, 10), 2, seed=22)
    counts = eng.count_patterns(eng.pack(codes))
    a = eng.sparse_flattening_scores(counts, splits).cpu().numpy()
    b = eng.sparse_flattening_scores(counts, splits).cpu().numpy()
    assert np.array_equal(a, b)
    probs = eng.PatternTable(20, counts.keys, values=eng._table_values(counts) / float(cnt.sum()))
    c = eng.sparse_flattening_scores(probs, splits).cpu().numpy()
    for x, y in zip(c, a):
        assert_score(x, y)


# ---------------------------------------------------------------------------------------------
# 7. public routes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [20, 64])
def test_score_splits_against_reference(sp, n):
    _, codes = simulated_codes(sp, n, 3000 if n == 20 else 2000, seed=70 + n)
    U, cnt = host_patterns(codes)
    splits = random_splits(n, (2, 5, n // 2), 3, seed=n + 3)
    from splitp_b200 import batch
    got = batch.score_splits(codes, splits, sp.Method.flattening)
    assert got.shape == (len(splits),)
    for s, (ia, ib) in enumerate(splits):
        assert_score(got[s], ref_score(U, cnt, ia, ib))


def informative(chosen):
    return {frozenset((frozenset(a), frozenset(b))) for a, b in chosen if min(len(a), len(b)) >= 2}


def restated_erickson(U, cnt, n):
    """phylogenetics.erickson_SVD(Method.flattening) with the host reference scores, on taxon positions."""
    clusters = [(t,) for t in range(n)]
    known, chosen = {}, []
    while len(chosen) < n - 2:
        best = None
        for x, y in itertools.combinations(clusters, 2):
            joined = tuple(sorted(x + y))
            rest = tuple(t for t in range(n) if t not in joined)
            key = (joined, rest)
            if key not in known:
                known[key] = ref_score(U, cnt, list(joined), list(rest))
            if best is None or known[key] < known[best]:
                best = key
        chosen.append(best)
        clusters = [c for c in clusters if not set(c) <= set(best[0])] + [best[0]]
    return chosen


def test_erickson_flattening_sparse_candidates(sp, monkeypatch):
    n = 16
    _, codes = simulated_codes(sp, n, 4000, seed=160, bl=0.15)
    U, cnt = host_patterns(codes)
    names = [str(np.base_repr(i, base=max(i + 1, 2))) for i in range(n)]  # erickson_SVD's default names, in position order
    mapping = {"".join("ACGT"[c] for c in row): int(k) for row, k in zip(U, cnt)}
    dense = sp.erickson_SVD(mapping, method=sp.Method.flattening)
    monkeypatch.setattr(sp.phylogenetics, "SPARSE_MIN_CELLS", 0)
    sparse = sp.erickson_SVD(mapping, method=sp.Method.flattening)
    pos = {t: i for i, t in enumerate(names)}
    to_pos = lambda ch: [(tuple(pos[t] for t in a), tuple(pos[t] for t in b)) for a, b in ch]  # noqa: E731
    assert informative(sparse) == informative(dense)
    assert informative(to_pos(sparse)) == informative(restated_erickson(U, cnt, n))


def test_split_score_of_sparse_flattening(sp, monkeypatch, sim20):
    tree, codes, U, cnt = sim20
    mapping = {"".join("ACGT"[c] for c in row): float(k) for row, k in zip(U, cnt)}
    taxa = [str(np.base_repr(i, base=max(i + 1, 2))) for i in range(20)]  # sorted names = position order ('0'..'9', 'A'..'J')
    splits = [([taxa[t] for t in a], [taxa[t] for t in b]) for a, b in random_splits(20, (5, 8, 10), 1, seed=23)]
    want = [sp.split_score(sp.flattening(s, mapping)) for s in splits]  # FlatFormat.sparse: a scipy sparse matrix
    monkeypatch.setattr(sp.phylogenetics, "SPARSE_MIN_CELLS", 0)
    got = [sp.split_score(sp.flattening(s, mapping)) for s in splits]
    for g, w in zip(got, want):
        assert type(g) is float
        assert_score(g, w)


# ---------------------------------------------------------------------------------------------
# 8. errors
# ---------------------------------------------------------------------------------------------
def test_non_covering_split_and_empty_table(sp, sim20):
    eng = sp.engine
    _, codes, _, _ = sim20
    table = eng.count_patterns(eng.pack(codes))
    with pytest.raises(ValueError, match="every taxon"):
        eng.sparse_flattening_scores(table, [([0, 1], [2, 3])])
    empty = eng.PatternTable(20, eng._empty(0, torch.int64), values=eng._empty(0, torch.float64))
    out = eng.sparse_flattening_scores(empty, [([0, 1], list(range(2, 20)))])
    assert out.cpu().numpy().tolist() == [0.0]
