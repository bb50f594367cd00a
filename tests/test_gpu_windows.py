"""GPU tests of site windows (spb_pair_tables_segments / spb_pair_finalize_rows in csrc/pairs.cu, engine.pair_raw_segments /
window_tables / window_subflatten_scores / window_tree_masks, batch.window_scores / window_trees).  Run with `-m gpu`.

Row w of window_scores must be score_splits of the alignment restricted to window w's sites, and tree w of window_trees
must be erickson_SVD's agglomeration (tests/erickson_reference.py) under those scores.
"""
import numpy as np
import pytest

import bench_inputs as BI
from tests import erickson_reference as ER

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TILE = 2048  # sites per tile of the pair kernels


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401
    return splitp_b200


def raw_model(codes):
    """numpy model of the raw pair statistics (spb_pair_raw_words layout) of a code matrix: usable sites only."""
    n = codes.shape[0]
    c = codes[:, (codes <= 3).all(axis=0)].astype(np.int64)
    raw = np.zeros(n * n * 9 + n * 3 + 1, np.int64)
    for i in range(n):
        for x in range(3):
            raw[n * n * 9 + i * 3 + x] = int((c[i] == x).sum())
        for j in range(i + 1, n):
            for x in range(3):
                for y in range(3):
                    raw[(i * n + j) * 9 + x * 3 + y] = int(((c[i] == x) & (c[j] == y)).sum())
    raw[-1] = c.shape[1]
    return raw


BOUNDS = [0, 5, 31, 32, 33, 64, 64, 65, TILE - 1, TILE, TILE + 1, 2 * TILE, 2 * TILE, 2 * TILE + 37, 3 * TILE + 100,
          3 * TILE + 101, 3 * TILE + 400]


@pytest.mark.parametrize("n", [2, 5, 20, 33, 64])
def test_segments_equal_slices(sp, n):
    eng = sp.engine
    N = 3 * TILE + 400
    codes = np.ascontiguousarray(BI.simulate_codes(n + n % 2, 0.2, "JC", N, n)[:n])  # balanced trees: even leaf counts
    for site in (30, 31, 32, 64, TILE - 1, TILE, 2 * TILE, 3 * TILE + 100):  # invalid sites next to boundaries
        codes[site % n, site] = 255
    aln = eng.pack(codes)
    for bounds in (BOUNDS, [100, 3000, 3001, 5000], [7, 7], [0, N]):
        rows = eng.pair_raw_segments(aln, bounds).cpu().numpy()
        assert rows.shape == (len(bounds) - 1, int(eng.lib.spb_pair_raw_words(n)))
        for s in range(len(bounds) - 1):
            b, e = bounds[s], bounds[s + 1]
            model = raw_model(codes[:, b:e])
            assert np.array_equal(rows[s], model), (bounds, s)
            if e > b:
                ref = eng.pair_raw(eng.pack(np.ascontiguousarray(codes[:, b:e]))).cpu().numpy()
                assert np.array_equal(rows[s], ref), (bounds, s)


def cta_runs(sp, N, site0, site1):
    """Sites per CTA run of spb_pair_tables_segments over the segments [site0, site1) of an N-site alignment: it launches
    min(2 SMs, tiles of the alignment) CTAs and CTA c takes `per` consecutive tiles from the first tile of site0."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    grid = min(2 * sm, -(-int(sp.engine.lib.spb_plane_words(N)) // 64))
    tile0, tile1 = (site0 // 32) // 64, -(-(-(-site1 // 32)) // 64)
    per = -(-(tile1 - tile0) // grid)
    return tile0 * TILE, per * TILE


@pytest.mark.parametrize("site0", [0, 3 * TILE + 77])
def test_segments_across_tiles_of_one_cta(sp, site0):
    """Segments long enough that every CTA owns several tiles: counters and the current segment carry over from tile to
    tile, a segment ends inside a CTA's run, on tile edges and on the edges between two CTAs' runs, and some span many
    tiles and several CTAs."""
    eng = sp.engine
    n, N = 5, 2_000_123
    rng = np.random.default_rng(site0 + 1)
    codes = rng.integers(0, 4, size=(n, N), dtype=np.uint8)
    start, run = cta_runs(sp, N, site0, N)
    assert run >= 4 * TILE  # several tiles per CTA
    edges = [start + k * run for k in range(1, 6)]
    for site in [edges[0] - 1, edges[0], edges[1] + 1, start + 2 * TILE - 1, N - 1]:  # unusable sites next to boundaries
        codes[site % n, site] = 255
    bounds = sorted([site0, site0 + 1000, start + 3 * TILE,  # inside the first tile, then on a tile edge in the first run
                     edges[0] - 1, edges[0], edges[0], edges[0] + 1,  # around the edge of the first two runs (one empty)
                     edges[1] - TILE, edges[1] + 5,  # a segment crossing a run edge
                     edges[1] + 2 * TILE + 300,  # several tiles inside one run
                     edges[4] + 17,  # a segment several runs long
                     N - 40, N])
    aln = eng.pack(codes, want_sm=False)
    rows = eng.pair_raw_segments(aln, bounds).cpu().numpy()
    for s in range(len(bounds) - 1):
        b, e = bounds[s], bounds[s + 1]
        assert np.array_equal(rows[s], raw_model(codes[:, b:e])), (bounds, s)
    for s in (3, 7, 10):  # the slice packed on its own: a run edge, a multi-tile segment, a multi-run segment
        b, e = bounds[s], bounds[s + 1]
        ref = eng.pair_raw(eng.pack(np.ascontiguousarray(codes[:, b:e]), want_sm=False)).cpu().numpy()
        assert np.array_equal(rows[s], ref), (bounds, s)


def test_window_scores_long_alignment(sp):
    n, N = 8, 2_000_000
    codes = np.ascontiguousarray(BI.simulate_codes(n, 0.1, "JC", N, 17))
    codes[3, 700_000:700_050] = 255
    splits = splits_for(n, 30, 4)
    wins = np.concatenate([sp.batch.sliding_windows(N, 300_000, 170_000), [[0, N], [650_000, 1_900_001], [12, 40]]])
    got = sp.batch.window_scores(codes, splits, wins, sp.Method.subflattening)
    for w, (b, e) in enumerate(wins.tolist()):
        ref = sp.batch.score_splits(np.ascontiguousarray(codes[:, b:e]), splits, sp.Method.subflattening)
        assert_rows_equal(got[w], ref)


def window_codes(n, seed, N=6000):
    codes = np.ascontiguousarray(BI.simulate_codes(n + n % 2, 0.1, "JC", N, seed)[:n])
    codes[n // 2, 4000:4100] = 255  # a window without usable sites
    codes[0, 1000:1010] = 255
    return codes


WINDOWS = [(100, 2500), (2000, 4500), (0, 6000), (100, 2500), (4000, 4100), (5, 6), (3000, 3001), (4099, 5999), (1000, 1011)]


def splits_for(n, count, seed):
    out = BI.random_splits_idx(n, count, seed) if n >= 4 else []
    out.append(([0], list(range(1, n))))  # a one-taxon side
    return out


def assert_rows_equal(got, ref, tol=False):
    if not tol:
        assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
        return
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    with np.errstate(divide="ignore", over="ignore"):
        bound = np.maximum(1e-9, 64 * np.finfo(float).eps / ref[ok] ** 2)
    assert (np.abs(got[ok] - ref[ok]) <= bound * np.maximum(np.abs(ref[ok]), 1e-300)).all()


@pytest.mark.parametrize("method", ["subflattening", "mutual_information"])
@pytest.mark.parametrize("n", [4, 12, 20, 40, 64])
def test_window_scores_equal_score_splits(sp, n, method):
    m = getattr(sp.Method, method)
    codes = window_codes(n, 3 * n)
    splits = splits_for(n, 40, n)
    wins = [w for w in WINDOWS if method == "subflattening" or w != (4000, 4100)]
    got = sp.batch.window_scores(codes, splits, wins, m)
    assert got.shape == (len(wins), len(splits)) and got.dtype == np.float64
    for w, (b, e) in enumerate(wins):
        ref = sp.batch.score_splits(np.ascontiguousarray(codes[:, b:e]), splits, m)
        assert_rows_equal(got[w], ref)


@pytest.mark.parametrize("n", [8, 12, 20])
def test_window_scores_flattening(sp, n):
    codes = window_codes(n, 5 * n)
    splits = splits_for(n, 12, n)
    wins = [w for w in WINDOWS if w != (4000, 4100)]
    got = sp.batch.window_scores(codes, splits, wins, sp.Method.flattening)
    for w, (b, e) in enumerate(wins):
        ref = sp.batch.score_splits(np.ascontiguousarray(codes[:, b:e]), splits, sp.Method.flattening)
        assert_rows_equal(got[w], ref, tol=True)


def outcome(fn):
    try:
        return fn()
    except Exception as e:  # noqa: BLE001  the outcome of score_splits on such a slice, whatever it is
        return type(e)


@pytest.mark.parametrize("method,n", [("subflattening", 12), ("subflattening", 40), ("mutual_information", 12),
                                      ("mutual_information", 40), ("flattening", 8), ("flattening", 20)])
def test_window_without_usable_sites(sp, method, n):
    m = getattr(sp.Method, method)
    codes = window_codes(n, 7 * n)
    splits = splits_for(n, 6, n)
    got = outcome(lambda: sp.batch.window_scores(codes, splits, [(4000, 4100)], m))
    ref = outcome(lambda: sp.batch.score_splits(np.ascontiguousarray(codes[:, 4000:4100]), splits, m))
    if isinstance(ref, type):
        assert got is ref
        return
    assert np.array_equal(got[0].view(np.uint64), ref.view(np.uint64))
    if method == "subflattening":  # all-zero pair tables: NaN where both sides hold two taxa or more, 0.0 otherwise
        two = np.array([min(len(a), len(b)) >= 2 for a, b in splits])
        assert np.isnan(ref[two]).all() and (ref[~two] == 0.0).all()


def test_window_scores_edge_cases(sp):
    codes = window_codes(12, 1)
    splits = splits_for(12, 5, 1)
    for m in (sp.Method.subflattening, sp.Method.mutual_information, sp.Method.flattening):
        assert sp.batch.window_scores(codes, splits, np.zeros((0, 2), np.int64), m).shape == (0, len(splits))
        assert sp.batch.window_scores(codes, [], [(0, 10)], m).shape == (1, 0)
    assert sp.batch.window_trees(codes, []) == []


def test_groups_do_not_change_results(sp, monkeypatch):
    codes = window_codes(20, 9)
    splits = splits_for(20, 30, 2)
    wins = sp.batch.sliding_windows(6000, 1500, 700)[::-1]
    a = sp.batch.window_scores(codes, splits, wins, sp.Method.subflattening)
    ta = sp.batch.window_trees(codes, wins)
    with monkeypatch.context() as mp:
        mp.setattr(sp.engine, "WINDOW_BATCH_BYTES", 1)  # one window per group
        b = sp.batch.window_scores(codes, splits, wins, sp.Method.subflattening)
        tb = sp.batch.window_trees(codes, wins)
    assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    assert ta == tb


def names_for(n, seed):
    perm = np.random.default_rng(seed).permutation(n)
    return [f"x{int(p):02d}" for p in perm]


@pytest.mark.parametrize("n", [2, 3, 12, 33, 64])
def test_window_trees_equal_restatement(sp, n):
    codes = window_codes(n, 11 * n, N=5000)
    taxa = names_for(n, n)
    wins = [(0, 5000), (1200, 3300), (4000, 4100)] if n <= 12 else [(1200, 3300)]
    trees = sp.batch.window_trees(codes, wins, taxa=taxa)
    assert len(trees) == len(wins)
    for (b, e), tree in zip(wins, trees):
        assert len(tree) == max(n - 2, 0)

        def score_many(splits):  # the lockstep agglomeration orders NaN (a window without usable sites) as +inf
            sc = sp.batch.window_scores(codes, splits, [(b, e)], sp.Method.subflattening, taxa=taxa)[0]
            return np.where(np.isnan(sc), np.inf, sc).tolist()

        chosen, _ = ER.agglomerate(taxa, score_many)
        assert tree == chosen, (b, e)


def informative(tree):
    return {frozenset(s) for s in tree if min(len(s[0]), len(s[1])) >= 2}


def test_window_trees_of_a_well_resolved_tree(sp):
    from splitp_b200.alignment import Alignment
    from splitp_b200.phylogenetics import erickson_SVD
    from tests.test_gpu_bootstrap_trees import true_splits
    n, N = 20, 60_000
    codes = BI.simulate_codes(n, 0.05, "JC", N, 11)
    _, truth = true_splits(n)  # leaf names as erickson_SVD names the rows by default
    taxa = sp.batch._default_taxa(n)
    wins = sp.batch.sliding_windows(N, 20_000, 10_000)
    trees = sp.batch.window_trees(codes, wins)
    lut = np.array(list("ACGT"))
    for (b, e), tree in zip(wins.tolist(), trees):
        cols, counts = np.unique(codes[:, b:e].T, axis=0, return_counts=True)
        mapping = {"".join(lut[c]): int(k) / (e - b) for c, k in zip(cols, counts)}
        host = erickson_SVD(Alignment(mapping, taxa), taxa=taxa, method=sp.Method.subflattening)
        assert informative(tree) == informative(host) == {frozenset(s) for s in truth}
