"""GPU tests of bootstrap trees along site windows: the count-row pair tables (spb_pair_tables_count_rows, csrc/pair_rows.cu),
the stacked tables of engine.bootstrap_group_tables and batch.window_bootstrap_trees.  Run with `-m gpu`."""
import numpy as np
import pytest

import bench_inputs as BI

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0xB007


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401
    return splitp_b200


def keys_of(codes):
    """Keys of a code matrix [P, n] in the layout of the pattern tables: uint64 [P] up to 31 taxa, {lo, hi} [P, 2] above."""
    P, n = codes.shape
    lo, hi = np.zeros(P, np.uint64), np.zeros(P, np.uint64)
    for t in range(n):
        sh = 2 * (n - 1 - t)
        d = codes[:, t].astype(np.uint64)
        if sh < 64:
            lo |= d << np.uint64(sh)
        else:
            hi |= d << np.uint64(sh - 64)
    return lo if n <= 31 else np.stack([lo, hi], axis=1)


def reference_tables(sp, keys, rows, n):
    """N of every row through the single-table routes (spb_pair_tables_weighted / spb_pair_tables_wide)."""
    eng = sp.engine
    out = []
    for r in range(rows.shape[0]):
        vals = (rows[r].to(torch.int64) & 0xFFFFFFFF).to(torch.float64).contiguous()
        P = int(vals.shape[0])
        if n <= 31:
            N = eng._zeros((n, n, 4, 4), torch.float64)
            eng.call("spb_pair_tables_weighted", eng._p(keys), eng._p(vals), P, n, eng._p(N), eng._st())
        else:
            N = eng._empty((n, n, 4, 4), torch.float64)
            ws = eng._empty(max(int(eng.lib.spb_pair_tables_wide_ws(P, n)), 1), torch.float64)
            eng.call("spb_pair_tables_wide", eng._p(keys), eng._p(vals), P, n, eng._p(N), eng._p(ws), eng._st())
        out.append(N)
    return torch.stack(out) if out else eng._empty((0, n, n, 4, 4), torch.float64)


def count_rows(rng, R, P, big_row=None):
    rows = rng.integers(0, 7, size=(R, P)).astype(np.uint32)
    rows[rng.random((R, P)) < 0.4] = 0
    if R > 2:
        rows[1] = 0  # a row of zeros
    if big_row is not None and P > 0:  # a row summing to 2^32 - 1
        rows[big_row] = 1
        rows[big_row, P // 2] = np.uint32(2 ** 32 - 1 - (P - 1))
    return rows


@pytest.mark.parametrize("n", [2, 3, 12, 20, 31, 32, 44, 64])
@pytest.mark.parametrize("R,P", [(1, 1), (1, 777), (5, 1), (9, 4099), (101, 3001), (37, 20_011)])
def test_count_rows_equal_single_table_routes(sp, n, R, P):
    eng = sp.engine
    rng = np.random.default_rng(n * 1000 + R + P)
    codes = rng.integers(0, 4, size=(P, n)).astype(np.uint8)
    keys = torch.from_numpy(keys_of(codes).view(np.int64)).to(eng.device()).contiguous()
    rows_np = count_rows(rng, R, P, big_row=R - 1 if R > 1 else None)
    rows = torch.from_numpy(rows_np.view(np.int32)).to(eng.device())
    got = eng.pair_tables_count_rows(keys, rows, n)
    want = reference_tables(sp, keys, rows, n)
    assert got.shape == (R, n, n, 4, 4)
    assert torch.equal(got.view(torch.int64), want.view(torch.int64))  # bit for bit
    again = eng.pair_tables_count_rows(keys, rows, n)
    assert torch.equal(again.view(torch.int64), got.view(torch.int64))
    # the diagonal blocks hold the row sums
    sums = rows_np.astype(np.float64).sum(axis=1)
    assert np.array_equal(got[:, 0, 0].sum(dim=(1, 2)).cpu().numpy(), sums)


@pytest.mark.parametrize("n", [4, 40])
def test_count_rows_empty_inputs(sp, n):
    eng = sp.engine
    dev = eng.device()
    keys = torch.zeros((0, 2) if n > 31 else (0,), dtype=torch.int64, device=dev)
    got = eng.pair_tables_count_rows(keys, torch.zeros((3, 0), dtype=torch.int32, device=dev), n)
    assert got.shape == (3, n, n, 4, 4) and not got.any()
    assert eng.pair_tables_count_rows(keys, torch.zeros((0, 0), dtype=torch.int32, device=dev), n).shape == (0, n, n, 4, 4)


def test_count_rows_argument_checks(sp):
    eng = sp.engine
    dev = eng.device()
    keys = torch.zeros((8, 2), dtype=torch.int64, device=dev)
    rows = torch.ones((2, 7), dtype=torch.int32, device=dev)
    N = eng._empty((2, 40, 40, 4, 4), torch.float64)
    with pytest.raises(ValueError, match="16-byte aligned"):  # keys starting 8 bytes into an allocation
        eng.call("spb_pair_tables_count_rows", keys.data_ptr() + 8, eng._p(rows), 2, 7, 40, eng._p(N), eng._st())
    for n in (1, 65):
        with pytest.raises(ValueError, match="n_taxa"):
            eng.call("spb_pair_tables_count_rows", eng._p(keys), eng._p(rows), 2, 7, n, eng._p(N), eng._st())
    with pytest.raises(ValueError, match="bad sizes"):
        eng.call("spb_pair_tables_count_rows", eng._p(keys), eng._p(rows), -1, 7, 40, eng._p(N), eng._st())
    with pytest.raises(ValueError, match="NULL"):
        eng.call("spb_pair_tables_count_rows", None, eng._p(rows), 2, 7, 40, eng._p(N), eng._st())
    with pytest.raises(ValueError, match="NULL"):
        eng.call("spb_pair_tables_count_rows", eng._p(keys), eng._p(rows), 2, 7, 40, None, eng._st())


def counted(sp, codes):
    eng = sp.engine
    if codes.shape[0] <= eng.NARROW_MAX_TAXA:
        return eng.count_patterns(eng.pack(codes))
    return eng.count_patterns_wide(*eng.pack_wide(codes))


@pytest.mark.parametrize("n", [12, 20, 40, 44, 64])
def test_group_tables_equal_table_by_table(sp, n):
    eng = sp.engine
    B = 6
    tables = [counted(sp, BI.simulate_codes(n + n % 2, 0.1, "JC", sites, n + sites)[:n]) for sites in (3_000, 1_000)]
    seeds = [SEED, 2 ** 64 - 3]
    srcs = eng.bootstrap_sources(tables, seeds)
    ref = eng.SubflattenTables(n, 2 * (B + 1))
    for s, (table, seed) in enumerate(zip(tables, seeds)):
        keys, counts = eng._counted(table)
        ref.add(s * (B + 1), eng._table_of_counts(table, keys, counts, srcs[s][3]))
        for b, tb in enumerate(eng.bootstrap_tables(table, B, seed)):
            ref.add(s * (B + 1) + b + 1, tb)
    # up to 43 taxa a slot ends in 8 doubles of padding that no kernel writes
    used = ref.data.shape[1] - (8 if n <= eng.SUBFLATTEN_TABLES_MAX_TAXA else 0)
    for f0, f1 in ((0, 2 * (B + 1)), (3, 11), (7, 8)):  # all rows; a group across both sources; one replicate
        got = eng.bootstrap_group_tables(srcs, B + 1, f0, f1, n)
        assert torch.equal(got.data[:, :used].view(torch.int64), ref.data[f0:f1, :used].view(torch.int64))
        assert torch.equal(got.total.view(torch.int64), ref.total[f0:f1].view(torch.int64))


def assert_same(a, b):
    assert a.tree == b.tree
    assert a.replicate_trees == b.replicate_trees
    assert a.support.dtype == b.support.dtype == np.float64
    assert np.array_equal(a.support, b.support)


WINDOWS = [[1_000, 2_500], [0, 1_000], [500, 1_700], [0, 1_000], [2_999, 3_000], [0, 3_000]]


@pytest.mark.parametrize("n,reps", [(12, 20), (20, 20), (40, 8), (64, 5)])
def test_entries_equal_bootstrap_trees_on_slices(sp, n, reps):
    codes = BI.simulate_codes(n, 0.05, "JC", 3_000, 3 * n)
    taxa = [f"s{(7 * i + 3) % n:02d}" for i in range(n)]  # the smallest name is not in row 0
    got = sp.batch.window_bootstrap_trees(codes, WINDOWS, replicates=reps, seed=SEED, taxa=taxa)
    assert len(got) == len(WINDOWS)
    for (b, e), res in zip(WINDOWS, got):
        want = sp.batch.bootstrap_trees(np.ascontiguousarray(codes[:, b:e]), reps, seed=sp.engine.window_bootstrap_seed(SEED, b, e),
                                        taxa=taxa)
        assert_same(res, want)
        assert len(res.replicate_trees) == reps and len(res.tree) == n - 2
    assert_same(got[1], got[3])  # a repeated window
    # fixed splits: every entry equals the slice's bootstrap_trees with the same splits
    splits = [s for s in got[-1].tree if min(len(s[0]), len(s[1])) >= 2][:5] + [(taxa[:n // 2], taxa[n // 2:])]
    got_s = sp.batch.window_bootstrap_trees(codes, WINDOWS[:3], replicates=reps, seed=SEED, taxa=taxa, splits=splits)
    for (b, e), res in zip(WINDOWS[:3], got_s):
        want = sp.batch.bootstrap_trees(np.ascontiguousarray(codes[:, b:e]), reps, seed=sp.engine.window_bootstrap_seed(SEED, b, e),
                                        taxa=taxa, splits=splits)
        assert_same(res, want)
        assert res.support.shape == (len(splits),)


def test_dict_input_and_grouping(sp, monkeypatch):
    n = 16
    codes = BI.simulate_codes(n, 0.1, "JC", 4_000, 9)
    taxa = [f"t{i:02d}" for i in range(n)]
    aln = BI.codes_to_sequences(codes, taxa)
    wins = sp.batch.sliding_windows(4_000, 1_500, 500)
    a = sp.batch.window_bootstrap_trees(aln, wins, replicates=12, seed=7)
    with monkeypatch.context() as mp:
        mp.setattr(sp.engine, "BOOTSTRAP_TREES_BATCH_BYTES", 1)  # one table per lockstep group
        b = sp.batch.window_bootstrap_trees(aln, wins, replicates=12, seed=7)
    eng = sp.engine
    packed = eng.pack(codes)
    P_max = max(eng.count_patterns(packed, b, e).num for b, e in wins.tolist())
    groups = []
    lockstep = eng.erickson_lockstep

    def spy(n_, reps, *args, **kw):
        groups.append(reps)
        return lockstep(n_, reps, *args, **kw)
    with monkeypatch.context() as mp:  # groups of 5 rows: cut inside the windows' 13 rows
        mp.setattr(eng, "BOOTSTRAP_TREES_BATCH_BYTES", 5 * eng.bootstrap_row_bytes(n, P_max))
        mp.setattr(eng, "erickson_lockstep", spy)
        c = sp.batch.window_bootstrap_trees(aln, wins, replicates=12, seed=7)
    assert groups == [5] * (len(wins) * 13 // 5) + ([len(wins) * 13 % 5] if len(wins) * 13 % 5 else [])
    for x, y, z in zip(a, b, c):
        assert_same(x, y)
        assert_same(x, z)
    # the windows' own position does not matter: the reversed list gives the reversed entries
    r = sp.batch.window_bootstrap_trees(aln, wins[::-1], replicates=12, seed=7)
    for x, y in zip(a, r[::-1]):
        assert_same(x, y)


def test_window_without_usable_sites(sp):
    codes = BI.simulate_codes(6, 0.1, "JC", 500, 1)
    codes[:, 100:140] = 255  # no usable site in [100, 140)
    with pytest.raises(ValueError, match=r"window 1 \[100, 140\) has no usable site"):
        sp.batch.window_bootstrap_trees(codes, [[0, 500], [100, 140]], replicates=2)


def test_bootscan_finds_the_recombinant_halves(sp):
    from splitp_b200 import simulation, trees
    n, half = 8, 6_000
    t1 = trees.balanced_tree(n, 0.05)
    node = {name: i for i, name in t1.names.items()}
    names2 = dict(t1.names)
    names2[node["1"]], names2[node["4"]] = "4", "1"  # swap two taxa of the two different clades
    t2 = trees.Tree(t1.parent, names2, t1.branch_length)
    model = simulation.GTR.JukesCantor(1.0)
    codes = torch.cat([simulation.simulate_codes(t1, model, half, seed=1), simulation.simulate_codes(t2, model, half, seed=2)], dim=1)
    taxa = sp.batch._default_taxa(n)
    s1 = (("0", "1", "2", "3"), ("4", "5", "6", "7"))
    s2 = (("0", "2", "3", "4"), ("1", "5", "6", "7"))
    wins = [[0, 2_000], [2_000, 4_000], [3_900, 5_900], [6_100, 8_100], [10_000, 12_000]]
    res = sp.batch.window_bootstrap_trees(codes, wins, replicates=100, seed=SEED, taxa=taxa, splits=[s1, s2])
    for (b, e), r in zip(wins, res):
        own, other = (0, 1) if e <= half else (1, 0)
        assert r.support[own] >= 0.95 and r.support[other] <= 0.05, (b, e, r.support)
