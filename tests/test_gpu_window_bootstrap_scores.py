"""GPU tests of bootstrap split scores along site windows: the count-row rank-1 divergence (spb_mi_row_slots +
spb_mi_row_scores, csrc/mi_batch.cu; engine.rank1_divergence_count_rows), engine.bootstrap_scores_multi through
batch.bootstrap_scores and batch.window_bootstrap_scores.  Every comparison is bit for bit.  Run with `-m gpu`."""
import types

import numpy as np
import pytest

import bench_inputs as BI

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0x5C0E
METHODS = ["flattening", "subflattening", "mutual_information"]


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401
    return splitp_b200


def method(name):
    from splitp_b200.enums import Method
    return getattr(Method, name)


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


def cover_splits(n, rng, count=12):
    """Covering splits of n taxa: 1-taxon sides, the n/2 | n/2 split, an empty side and random ones."""
    out = [([0], list(range(1, n))), (list(range(n - 1)), [n - 1]), (list(range(n // 2)), list(range(n // 2, n))),
           ([], list(range(n)))]
    for _ in range(count):
        perm = rng.permutation(n)
        k = int(rng.integers(1, n))
        out.append((sorted(perm[:k].tolist()), sorted(perm[k:].tolist())))
    return out


def pattern_list(rng, n, P):
    """Distinct codes [P', n] (P' <= P) that include the all-T pattern (the all-ones key at 64 taxa)."""
    codes = rng.integers(0, 4, size=(P, n)).astype(np.uint8)
    codes[0] = 3
    codes[1] = 0
    return np.unique(codes, axis=0)


@pytest.mark.parametrize("n", [12, 20, 40, 64])
def test_count_rows_equal_compacted_tables(sp, n, monkeypatch):
    eng = sp.engine
    rng = np.random.default_rng(n)
    codes = pattern_list(rng, n, 3_000)
    P = codes.shape[0]
    keys = torch.from_numpy(keys_of(codes).view(np.int64)).to(eng.device()).contiguous()
    R = 9
    rows_np = rng.integers(0, 9, size=(R, P)).astype(np.uint32)
    rows_np[rng.random((R, P)) < 0.5] = 0
    all_t = int(np.flatnonzero((codes == 3).all(axis=1))[0])
    rows_np[2] = 0          # a row of zeros
    rows_np[3] = 0          # one pattern only: the all-T pattern
    rows_np[3, all_t] = 5
    rows_np[4, ::2] = 0
    rows = torch.from_numpy(rows_np.view(np.int32)).to(eng.device())
    splits = cover_splits(n, rng)
    div = float(rows_np.astype(np.int64).sum(axis=1).max())
    got = eng.rank1_divergence_count_rows(keys, lambda r0, r1: rows[r0:r1], R, n, div, splits)
    assert got.shape == (R, len(splits))
    owner = types.SimpleNamespace(n=n, taxa=None)
    for r in range(R):
        nz = torch.from_numpy(np.flatnonzero(rows_np[r])).to(eng.device())
        tb = eng._table_of_counts(owner, keys[nz].contiguous(), rows[r][nz].contiguous(), div)
        want = eng.rank1_divergence_scores(tb, splits)
        assert torch.equal(got[r].view(torch.int64), want.view(torch.int64)), r
    assert (got[:, 3] == 0).all() and (got[2] == 0).all()  # the empty side; the row of zeros
    # a single pattern: v = r = c = 5 / div for every split with two non-empty sides, so the score is v log(1 / v)
    v = 5 / div
    live = [j for j in range(len(splits)) if j != 3]
    assert np.allclose(got[3, live].cpu().numpy(), v * np.log(1 / v), rtol=1e-12, atol=0)
    # batches of splits and groups of rows: more than four launches, the same bits
    launches = []
    call = eng.call

    def spy(name, *args):
        if name == "spb_mi_row_scores":
            launches.append(name)
        return call(name, *args)
    cmax = int(eng.lib.spb_mi_rows_ws(P, 1, 0, 1))
    slots = 2 * int(eng.lib.spb_mi_side_cap(P, n // 2))
    with monkeypatch.context() as mp:
        mp.setattr(eng, "call", spy)
        mp.setattr(eng, "MI_BATCH_BYTES", 8 * (2 * slots + 3 * P + 2 * cmax) + 16 * P)
        again = eng.rank1_divergence_count_rows(keys, lambda r0, r1: rows[r0:r1], R, n, div, splits)
    assert len(launches) > 4
    assert torch.equal(again.view(torch.int64), got.view(torch.int64))


def test_count_rows_checks(sp):
    eng = sp.engine
    dev = eng.device()
    keys = torch.zeros(4, dtype=torch.int64, device=dev)
    desc = torch.zeros(8, dtype=torch.int64, device=dev)
    tk, so = torch.zeros(8, dtype=torch.int64, device=dev), torch.zeros(8, dtype=torch.int32, device=dev)
    with pytest.raises(ValueError, match="key_words"):
        eng.call("spb_mi_row_slots", eng._p(keys), 3, 4, eng._p(desc), 1, 4, eng._p(tk), eng._p(so), eng._st())
    with pytest.raises(ValueError, match="NULL"):
        eng.call("spb_mi_row_slots", None, 1, 4, eng._p(desc), 1, 4, eng._p(tk), eng._p(so), eng._st())
    with pytest.raises(ValueError, match="16-byte"):
        eng.call("spb_mi_row_slots", keys.data_ptr() + 8, 2, 1, eng._p(desc), 1, 4, eng._p(tk), eng._p(so), eng._st())
    with pytest.raises(ValueError, match="negative"):
        eng.call("spb_mi_row_scores", None, -1, None, None, 1, 1.0, None, 1, 4, None, None, None, eng._st())
    with pytest.raises(ValueError, match="NULL"):
        eng.call("spb_mi_row_scores", None, 4, None, None, 1, 1.0, eng._p(desc), 1, 4, eng._p(so), eng._p(tk), eng._p(tk),
                 eng._st())
    with pytest.raises(ValueError, match="65535 rows"):
        eng.call("spb_mi_row_scores", None, 4, None, None, 65536, 1.0, None, 1, 4, None, None, None, eng._st())


def counted(sp, codes):
    eng = sp.engine
    if codes.shape[0] <= eng.NARROW_MAX_TAXA:
        return eng.count_patterns(eng.pack(codes))
    return eng.count_patterns_wide(*eng.pack_wide(codes))


@pytest.mark.parametrize("n", [12, 20, 40, 64])
def test_bootstrap_scores_equal_the_per_replicate_route(sp, n):
    """bootstrap_scores against the route it replaced: every bootstrap_tables table through pair_tables_from_table +
    subflatten_scores, or rank1_divergence_scores."""
    eng = sp.engine
    B = 7
    codes = BI.simulate_codes(n, 0.1, "JC", 2_000, n)
    rng = np.random.default_rng(n + 1)
    splits = cover_splits(n, rng, 6)[:3] + cover_splits(n, rng, 6)[4:]
    table = counted(sp, codes)
    ma, mb = eng.masks_from_splits(splits)
    want_sub = torch.stack([eng.subflatten_scores(eng.pair_tables_from_table(tb, as_counts=True), ma, mb)
                            for tb in eng.bootstrap_tables(table, B, SEED)]).cpu().numpy()
    want_mi = torch.stack([eng.rank1_divergence_scores(tb, splits) for tb in eng.bootstrap_tables(table, B, SEED)]).cpu().numpy()
    got_sub = sp.batch.bootstrap_scores(codes, splits, method("subflattening"), B, SEED)
    got_mi = sp.batch.bootstrap_scores(codes, splits, method("mutual_information"), B, SEED)
    assert np.array_equal(got_sub.view(np.int64), want_sub.view(np.int64))
    assert np.array_equal(got_mi.view(np.int64), want_mi.view(np.int64))


WINDOWS = [[1_000, 2_500], [0, 1_000], [500, 1_700], [0, 1_000], [2_999, 3_000], [0, 3_000]]


@pytest.mark.parametrize("name", METHODS)
@pytest.mark.parametrize("n", [12, 20, 40])
def test_windows_equal_bootstrap_scores_on_slices(sp, n, name):
    m, B = method(name), 5
    codes = BI.simulate_codes(n, 0.05, "JC", 3_000, 3 * n)
    rng = np.random.default_rng(3 * n)
    splits = [s for s in cover_splits(n, rng, 3) if s[0]]
    if name == "flattening" and n <= 16:  # keep the dense count flattenings small
        splits = [s for s in splits if min(len(s[0]), len(s[1])) <= 4]
    got = sp.batch.window_bootstrap_scores(codes, splits, WINDOWS, m, replicates=B, seed=SEED)
    assert got.shape == (len(WINDOWS), B, len(splits)) and got.dtype == np.float64
    for w, (b, e) in enumerate(WINDOWS):
        want = sp.batch.bootstrap_scores(np.ascontiguousarray(codes[:, b:e]), splits, m, B,
                                          seed=sp.engine.window_bootstrap_seed(SEED, b, e))
        assert np.array_equal(got[w].view(np.int64), want.view(np.int64)), (w, b, e)
    assert np.array_equal(got[1].view(np.int64), got[3].view(np.int64))  # a repeated window


@pytest.mark.parametrize("name", ["subflattening", "mutual_information"])
def test_dict_input_order_and_grouping(sp, monkeypatch, name):
    eng, m, n, B = sp.engine, method(name), 16, 6
    codes = BI.simulate_codes(n, 0.1, "JC", 4_000, 9)
    taxa = [f"t{i:02d}" for i in range(n)]
    aln = BI.codes_to_sequences(codes, taxa)
    splits = [(taxa[:8], taxa[8:]), (["t03"], [t for t in taxa if t != "t03"]), (taxa[::2], taxa[1::2])]
    wins = sp.batch.sliding_windows(4_000, 1_500, 500)
    a = sp.batch.window_bootstrap_scores(aln, splits, wins, m, replicates=B, seed=7)
    for w, (b, e) in enumerate(wins.tolist()):
        sl = {t: s[b:e] for t, s in aln.items()}
        want = sp.batch.bootstrap_scores(sl, splits, m, B, seed=eng.window_bootstrap_seed(7, b, e))
        assert np.array_equal(a[w].view(np.int64), want.view(np.int64))
    with monkeypatch.context() as mp:  # one replicate row per group; one split per batch and one row per launch
        mp.setattr(eng, "BOOTSTRAP_SCORES_BATCH_BYTES", 1)
        mp.setattr(eng, "MI_BATCH_BYTES", 1)
        b_ = sp.batch.window_bootstrap_scores(aln, splits, wins, m, replicates=B, seed=7)
    assert np.array_equal(a.view(np.int64), b_.view(np.int64))
    r = sp.batch.window_bootstrap_scores(aln, splits, wins[::-1], m, replicates=B, seed=7)  # reordered windows
    assert np.array_equal(a.view(np.int64), r[::-1].view(np.int64))


def test_window_without_usable_sites_and_no_splits(sp):
    codes = BI.simulate_codes(6, 0.1, "JC", 500, 1)
    codes[:, 100:140] = 255  # no usable site in [100, 140)
    for name in METHODS:
        with pytest.raises(ValueError, match=r"window_bootstrap_scores: window 1 \[100, 140\) has no usable site"):
            sp.batch.window_bootstrap_scores(codes, [([0, 1, 2], [3, 4, 5])], [[0, 500], [100, 140]], method(name), replicates=2)
        out = sp.batch.window_bootstrap_scores(codes, [], [[0, 500], [0, 100]], method(name), replicates=3)
        assert out.shape == (2, 3, 0) and out.dtype == np.float64
