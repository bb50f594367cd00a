"""GPU tests of the batched rank-1 divergence (csrc/mi_batch.cu, engine.rank1_divergence_scores, score_splits with
Method.mutual_information): agreement with the per-split route, the reference's golden divergences, erickson_SVD's traced
scores and a numpy restatement up to 64 taxa; bitwise reproducibility of count tables; edge cases; two NCCL processes.
Run with `-m gpu`.

Tolerance: |got - ref| <= 1e-12 * sum_p |v_p log(v_p / (r c))|, which bounds the rounding of any summation order.
"""
import itertools
import os
import tempfile

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    import splitp_b200.batch  # noqa: F401  (score_splits, SplitScorer)
    return splitp_b200


def simulated_codes(sp, n, N, seed, bl=0.1):
    """Codes of n taxa (balanced trees need an even number: an odd n drops the last taxon of n + 1)."""
    tree = sp.trees.balanced_tree(n + n % 2, bl)
    codes = sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=seed).cpu().numpy().astype(np.uint8)
    return np.ascontiguousarray(codes[:n])


def np_divergence(U, v, ia, ib):
    """(divergence, sum of |terms|) of the flattening of (ia | ib) of the patterns U [P, n] with values v: side sums by
    np.unique of the projected patterns and bincount."""
    v = np.asarray(v, dtype=np.float64)
    keep = v != 0
    U, v = U[keep], v[keep]
    if len(v) == 0 or not len(ia) or not len(ib):
        return 0.0, 0.0
    ra = np.unique(U[:, list(ia)], axis=0, return_inverse=True)[1].reshape(-1)
    rb = np.unique(U[:, list(ib)], axis=0, return_inverse=True)[1].reshape(-1)
    c, r = np.bincount(ra, weights=v)[ra], np.bincount(rb, weights=v)[rb]
    t = v * np.log(v / (r * c))
    return float(t.sum()), float(np.abs(t).sum())


def host_probs(codes):
    """(U uint8 [P, n], probabilities [P]) of the usable sites of a code matrix [n, N]."""
    ok = (codes <= 3).all(axis=0)
    U, cnt = np.unique(codes[:, ok].T, axis=0, return_counts=True)
    return U, cnt / max(int(ok.sum()), 1)


def assert_close(got, ref, bound):
    assert abs(float(got) - ref) <= 1e-12 * bound, (float(got), ref, bound)


def covering(n, a_side):
    a = sorted(a_side)
    return a, [t for t in range(n) if t not in a]


def sampled_splits(n, sizes, per_size, seed):
    rng = np.random.default_rng(seed)
    out = []
    for a in sizes:
        for _ in range(per_size):
            out.append(covering(n, rng.choice(n, size=a, replace=False).tolist()))
    return out


def all_splits(n):
    out = []
    for a in range(1, n // 2 + 1):
        for side in itertools.combinations(range(n), a):
            if 2 * a == n and 0 not in side:
                continue
            out.append(covering(n, side))
    return out


@pytest.mark.parametrize("n,N", [(6, 20_000), (12, 100_000), (17, 100_000), (24, 100_000)])
def test_batched_matches_per_split(sp, n, N):
    codes = simulated_codes(sp, n, N, seed=n)
    splits = all_splits(n) if n <= 12 else sampled_splits(n, [1, 2, 8, 12, n - 1], 3, seed=n)
    got = sp.batch.score_splits(codes, splits, sp.Method.mutual_information)
    table = sp.engine.count_patterns(sp.engine.pack(codes))
    U, v = host_probs(codes)
    for (ia, ib), g in zip(splits, got):
        ref = float(sp.engine.rank1_divergence(table, ia, ib)[0].item())
        assert_close(g, ref, np_divergence(U, v, ia, ib)[1])


def test_golden_divergences(sp, golden_rank1):
    for rec in golden_rank1["erickson"]:
        table = sp.engine.table_from_mapping(dict(zip(rec["patterns"], rec["values"])))
        names = list(rec["divergences"])
        idx = [tuple([int(ch) for ch in side] for side in name.split("|")) for name in names]
        got = sp.engine.rank1_divergence_scores(table, idx).cpu().numpy()
        for name, g in zip(names, got):
            assert g == pytest.approx(rec["divergences"][name], rel=1e-12)


@pytest.mark.parametrize("n", [8, 9, 10])
def test_erickson_trace(sp, n):
    codes = simulated_codes(sp, n, 50_000, seed=100 + n)
    aln = sp.engine.table_to_dict(sp.engine.count_patterns(sp.engine.pack(codes)))
    tr = []
    sp.erickson_SVD(aln, method=sp.Method.mutual_information, trace=tr)
    U = np.array([[("ACGT").index(ch) for ch in p] for p in aln], dtype=np.uint8)
    v = np.array(list(aln.values()))
    table = sp.engine.table_from_mapping(aln)
    for step in tr:
        splits = list(step["scores"])
        idx = [sp.engine.split_positions(s, sorted(set(s[0]) | set(s[1]))) for s in splits]
        got = sp.engine.rank1_divergence_scores(table, idx).cpu().numpy()
        for (ia, ib), s, g in zip(idx, splits, got):
            assert_close(g, float(step["scores"][s]), np_divergence(U, v, ia, ib)[1])


def wide_codes(sp, n, N, seed):
    codes = simulated_codes(sp, n, N, seed=seed, bl=0.02)
    codes[:, : N // 50] = 3  # all-T sites: at 64 taxa the all-ones key
    return codes


def wide_splits(n, seed):
    rng = np.random.default_rng(seed)
    out = [covering(n, [0]), covering(n, [n - 1]), covering(n, [3, 7]), covering(n, [1, 30, n - 2])]
    out += [covering(n, rng.choice(n, size=int(rng.integers(1, n)), replace=False).tolist()) for _ in range(12)]
    if n == 64:
        out += [covering(n, range(32)), covering(n, range(32, 64)), covering(n, range(31)), covering(n, range(1, 64, 2))]
    return out


@pytest.mark.parametrize("n", [33, 40, 64])
def test_wide_against_numpy(sp, n):
    codes = wide_codes(sp, n, 60_000, seed=n)
    splits = wide_splits(n, seed=n)
    U, v = host_probs(codes)
    refs = [np_divergence(U, v, ia, ib) for ia, ib in splits]
    chars = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    got = sp.batch.score_splits(chars, splits, sp.Method.mutual_information)
    for g, (ref, bound) in zip(got, refs):
        assert_close(g, ref, bound)
    pats = ["".join("ACGT"[c] for c in row) for row in U]
    table = sp.engine.table_from_mapping(dict(zip(pats, v.tolist())))
    assert isinstance(table, sp.engine.WidePatternTable)
    got = sp.engine.rank1_divergence_scores(table, splits).cpu().numpy()
    for g, (ref, bound) in zip(got, refs):
        assert_close(g, ref, bound)


@pytest.mark.parametrize("n", [12, 20, 40])
def test_count_tables_bitwise_reproducible(sp, n, monkeypatch):
    codes = simulated_codes(sp, n, 80_000, seed=7 * n)
    splits = sampled_splits(n, [1, 2, n // 2, n - 3], 4, seed=n)
    if n <= 31:
        table = sp.engine.count_patterns(sp.engine.pack(codes))
    else:
        wide, valid, _, N = sp.engine.pack_wide(codes)
        table = sp.engine.count_patterns_wide(wide, valid, n, N)
    first = sp.engine.rank1_divergence_scores(table, splits).cpu().numpy()
    assert np.array_equal(first, sp.engine.rank1_divergence_scores(table, splits).cpu().numpy())
    assert np.array_equal(first, sp.batch.score_splits(codes, splits, sp.Method.mutual_information))
    order = np.random.default_rng(n).permutation(len(splits))[: len(splits) // 2]
    sub = sp.engine.rank1_divergence_scores(table, [splits[i] for i in order]).cpu().numpy()
    assert np.array_equal(sub, first[order])
    monkeypatch.setattr(sp.engine, "MI_BATCH_BYTES", 1 << 20)
    P = table.compact()[0].shape[0] if n > 31 else table.num
    caps = [sp.engine.lib.spb_mi_side_cap(P, len(a)) + sp.engine.lib.spb_mi_side_cap(P, len(b)) for a, b in splits]
    assert len(sp.engine.mi_batches(caps, P, 2 if n > 31 else 1)) > 4
    assert np.array_equal(first, sp.engine.rank1_divergence_scores(table, splits).cpu().numpy())


def test_edge_cases(sp):
    n = 9
    codes = simulated_codes(sp, n, 5_000, seed=3)
    splits = all_splits(n)[:20]
    mi = sp.Method.mutual_information
    assert np.array_equal(sp.batch.score_splits(np.full((n, 100), 255, np.uint8), splits, mi), np.zeros(len(splits)))
    assert np.array_equal(sp.batch.score_splits(np.full((40, 100), ord("N"), np.uint8), wide_splits(40, 1), mi), np.zeros(16))
    assert np.array_equal(sp.batch.score_splits(np.zeros((n, 100), np.uint8), splits, mi), np.zeros(len(splits)))
    with pytest.raises(ValueError):
        sp.batch.score_splits(codes, [([0, 1], [2, 3])], mi)
    with pytest.raises(ValueError):
        sp.batch.score_splits(codes, [([0, 1], [1, 2, 3, 4, 5, 6, 7, 8])], mi)
    got = sp.batch.score_splits(codes, [([], list(range(n))), splits[5], (list(range(n)), []), splits[5]], mi)
    assert got[0] == 0.0 and got[2] == 0.0 and got[1] == got[3] != 0.0
    taxa = [f"t{i}" for i in range(n)]
    labelled = [([taxa[i] for i in a], [taxa[i] for i in b]) for a, b in splits]
    assert np.array_equal(sp.batch.score_splits(codes, labelled, mi, taxa=taxa), sp.batch.score_splits(codes, splits, mi))
    aln = {t: "".join("ACGT"[c] for c in row) for t, row in zip(taxa, codes)}
    assert np.array_equal(sp.batch.score_splits(aln, labelled, mi), sp.batch.score_splits(codes, splits, mi))
    with pytest.raises(NotImplementedError):
        sp.batch.SplitScorer(splits, method=sp.Method.distance)


def _worker(rank, world, init, n, sites, out_path):
    import torch.distributed as dist

    import splitp_b200 as sp
    import splitp_b200.batch  # noqa: F401
    import splitp_b200.distributed  # noqa: F401
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=init, rank=rank, world_size=world)
    try:
        codes = simulated_codes(sp, n, 40_000, seed=n)
        splits = wide_splits(n, seed=n) if n > 31 else all_splits(n)[:200]
        if sites == "shard":
            b, e = sp.distributed.shard_range(codes.shape[1], rank, world, 32)
            mine = codes[:, b:e]
        else:
            mine = codes
        scorer = sp.batch.SplitScorer(splits, method=sp.Method.mutual_information, rank=rank, world=world, sites=sites)
        res = scorer(np.ascontiguousarray(mine))
        if rank == 0:
            np.save(out_path, res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [10, 20, 40])
@pytest.mark.parametrize("sites", ["shard", "replicated"])
def test_two_processes_bitwise(sp, n, sites):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    codes = simulated_codes(sp, n, 40_000, seed=n)
    splits = wide_splits(n, seed=n) if n > 31 else all_splits(n)[:200]
    one = sp.batch.score_splits(codes, splits, sp.Method.mutual_information)
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "scores.npy")
        mp.spawn(_worker, args=(2, "file://" + os.path.join(tmp, "rendezvous"), n, sites, out), nprocs=2, join=True)
        two = np.load(out)
    assert np.array_equal(one, two)
