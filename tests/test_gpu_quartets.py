"""GPU tests of quartet split scores: the quartet tables (spb_quartet_tables, csrc/quartets.cu; engine.quartet_tables) bit for
bit against a numpy count, the flattening scores against the oracle's LAPACK split_score and the drop-in per-quartet loop, the
rank-1 divergences against the oracle, subflattening against score_splits, orientation, input forms, grouping and the full
64-taxon quartet set (batch.quartet_scores).  Run with `-m gpu`."""
import itertools

import numpy as np
import pytest

import bench_inputs as BI
from tests import quartet_reference as QR

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
TAXA_COUNTS = [4, 5, 12, 20, 31, 32, 33, 48, 64]


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


def noisy_codes(n, N, seed, gap_rate=0.002):
    """Simulated codes with unusable characters (code 255) scattered over every taxon."""
    rng = np.random.default_rng(seed)
    codes = BI.simulate_codes(n + n % 2, 0.1, "JC", N, seed)[:n].copy()
    codes[rng.random(codes.shape) < gap_rate] = 255
    return codes


def sequences(codes, taxa):
    """{taxon: string}, unusable codes written as N."""
    lut = np.frombuffer(b"ACGTN", np.uint8)
    return {t: lut[np.minimum(codes[i], 4)].tobytes().decode() for i, t in enumerate(taxa)}


def sample_quartets(n, count, seed, shuffle=True):
    rng = np.random.default_rng(seed)
    allq = list(itertools.combinations(range(n), 4))
    pick = [allq[i] for i in rng.choice(len(allq), min(count, len(allq)), replace=False)]
    return np.array([rng.permutation(q) if shuffle else q for q in pick], dtype=np.int64)


def assert_score(got, ref):
    if np.isnan(ref):
        assert np.isnan(got)
        return
    tol = max(1e-9, 64 * EPS / max(ref * ref, 1e-300))
    assert abs(got - ref) <= tol * max(abs(ref), 1e-300) or (ref == 0.0 and got == 0.0), (got, ref)


def oracle_flattening_scores(oracle, table):
    out = []
    for p in range(3):
        R = QR.reduced(QR.flattening(table, p))
        out.append(float("nan") if R.size == 0 else 0.0 if min(R.shape) <= 4 else oracle.split_score(R))
    return out


@pytest.mark.parametrize("n", TAXA_COUNTS)
@pytest.mark.parametrize("N", [19, 2048 + 77, 3 * 2048 * 8 + 1000])
def test_tables_bit_exact(sp, n, N):
    from splitp_b200 import engine
    codes = noisy_codes(n, N, seed=n * 1000 + N)
    q = sample_quartets(n, 300, seed=n + N)
    got = engine.quartet_tables(engine.pack(codes), q).cpu().numpy()
    np.testing.assert_array_equal(got, QR.tables(codes, q))


@pytest.mark.parametrize("n", [5, 12, 20, 33, 64])
def test_flattening_scores_against_oracle(sp, oracle, n):
    codes = noisy_codes(n, 20_000, seed=7 * n)
    q = sample_quartets(n, 120, seed=n) if n != 12 else np.array(list(itertools.combinations(range(12), 4)))
    got = sp.batch.quartet_scores(codes, q, method("flattening"))
    assert got.shape == (len(q), 3)
    for row, table in zip(got, QR.tables(codes, q)):
        for g, r in zip(row, oracle_flattening_scores(oracle, table)):
            assert_score(g, r)


def test_degenerate_and_empty(sp):
    rng = np.random.default_rng(3)
    codes = rng.integers(0, 4, size=(6, 3000), dtype=np.uint8)
    codes[1] = codes[0]  # x_b = x_a: the flattening of {0,1}|{2,3} has 4 non-empty rows
    got = sp.batch.quartet_scores(codes, [(0, 1, 2, 3)], method("flattening"))
    assert got[0, 0] == 0.0
    empty = np.full((6, 100), 255, np.uint8)
    assert np.isnan(sp.batch.quartet_scores(empty, [(0, 1, 2, 3), (5, 4, 3, 2)], method("flattening"))).all()
    mi = sp.batch.quartet_scores(empty, [(0, 1, 2, 3)], method("mutual_information"))
    np.testing.assert_array_equal(mi, np.zeros((1, 3)))


@pytest.mark.parametrize("n", [12, 40])
def test_drop_in_parity(sp, n):
    from splitp_b200 import Alignment, FlatFormat, flattening, split_score
    from splitp_b200.parsers.fasta import get_pattern_counts
    taxa = [f"t{i}" for i in range(n)]
    seqs = sequences(noisy_codes(n, 5000, seed=n), taxa)
    mapping, _ = get_pattern_counts(seqs)
    aln = Alignment(mapping, taxa)
    quartets = [("t3", "t0", "t7", "t5"), ("t1", "t2", "t9", "t11"), ("t11", "t4", "t6", "t8")]
    got = sp.batch.quartet_scores(seqs, quartets, method("flattening"))
    for row, (a, b, c, d) in zip(got, quartets):
        sub = aln.sub_alignment([a, b, c, d])
        for col, split in enumerate([((a, b), (c, d)), ((a, c), (b, d)), ((a, d), (b, c))]):
            assert_score(row[col], float(split_score(flattening(split, sub, FlatFormat.reduced))))


@pytest.mark.parametrize("n", [5, 20, 64])
def test_mutual_information_against_oracle(sp, oracle, n):
    codes = noisy_codes(n, 20_000, seed=11 * n)
    q = sample_quartets(n, 60, seed=2 * n)
    got = sp.batch.quartet_scores(codes, q, method("mutual_information"))
    for row, table in zip(got, QR.tables(codes, q)):
        for p in range(3):
            ref = oracle.rank_1_divergence(QR.flattening(table, p) / table.sum())
            assert abs(row[p] - ref) <= 1e-12 * abs(ref), (row[p], ref)


@pytest.mark.parametrize("n", [20, 64])
def test_subflattening_equals_score_splits(sp, n):
    codes = noisy_codes(n, 30_000, seed=5 * n)
    q = np.sort(sample_quartets(n, 80, seed=3 * n), axis=1)
    got = sp.batch.quartet_scores(codes, q, method("subflattening"))
    splits = [s for a, b, c, d in q.tolist() for s in (([a, b], [c, d]), ([a, c], [b, d]), ([a, d], [b, c]))]
    want = sp.batch.score_splits(codes, splits, method("subflattening")).reshape(-1, 3)
    np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("name", ["flattening", "subflattening", "mutual_information"])
def test_orientation(sp, name):
    codes = noisy_codes(20, 10_000, seed=17)
    base = [(2, 5, 11, 17), (0, 1, 2, 3), (19, 4, 8, 13)]
    written, expect = [], []
    for q in base:
        for perm in itertools.permutations(q):
            written.append(perm)
            expect.append([frozenset([frozenset((perm[0], perm[j])), frozenset(set(perm) - {perm[0], perm[j]})]) for j in (1, 2, 3)])
    got = sp.batch.quartet_scores(codes, written, method(name))
    ref = {}
    for row, bips in zip(got, expect):
        for v, bip in zip(row, bips):
            ref.setdefault(bip, v)
            assert v.tobytes() == ref[bip].tobytes()
    dup = sp.batch.quartet_scores(codes, [base[0], base[1], base[0]], method(name))
    assert dup[0].tobytes() == dup[2].tobytes()


def test_input_forms(sp):
    from splitp_b200 import engine
    n, N = 33, 4000
    codes = noisy_codes(n, N, seed=23)
    taxa = [f"x{i}" for i in range(n)]
    seqs = sequences(codes, taxa)
    lut = np.frombuffer(b"ACGTN", np.uint8)
    q = sample_quartets(n, 50, seed=1)
    labels = [tuple(taxa[i] for i in row) for row in q.tolist()]
    planes, valid = sp.batch.pack_planes_host(codes)
    forms = [
        (seqs, labels),
        (codes, q),
        (lut[np.minimum(codes, 4)], q),
        (torch.from_numpy(codes).cuda(), q),
        (sp.batch.HostPlanes(planes, valid, n, N), q),
        (engine.pack(codes), q),
    ]
    for name in ("flattening", "mutual_information", "subflattening"):
        outs = [sp.batch.quartet_scores(a, qq, method(name)) for a, qq in forms]
        for o in outs[1:]:
            assert o.tobytes() == outs[0].tobytes(), name


@pytest.mark.parametrize("name", ["flattening", "mutual_information", "subflattening"])
def test_grouping(sp, monkeypatch, name):
    from splitp_b200 import engine
    codes = noisy_codes(16, 8000, seed=29)
    whole = sp.batch.quartet_scores(codes, None, method(name))
    monkeypatch.setattr(engine, "QUARTET_BATCH_BYTES", 97 * engine._QUARTET_BYTES)  # 1,820 quartets in 19 groups
    grouped = sp.batch.quartet_scores(codes, None, method(name))
    assert grouped.tobytes() == whole.tobytes()


def test_full_64_taxa(sp, oracle):
    """All 635,376 quartets of a 64-taxon x 10^5-site alignment simulated on the balanced tree (branch length 0.05).  The
    numpy model of the tables with the oracle's scores picks the true topology for 400 of 400 sampled quartets of this
    alignment; the test asks for 99 % of all quartets."""
    n = 64
    codes = BI.simulate_codes(n, 0.05, "JC", 100_000, 3)
    got = sp.batch.quartet_scores(codes, None, method("flattening"))
    assert got.shape == (635_376, 3) and not np.isnan(got).any()
    allq = sp.engine.all_quartets(n)
    rng = np.random.default_rng(0)
    idx = rng.choice(len(allq), 40, replace=False)
    for i, table in zip(idx, QR.tables(codes, allq[idx])):
        for g, r in zip(got[i], oracle_flattening_scores(oracle, table)):
            assert_score(g, r)
    hit = (got.argmin(axis=1) == QR.true_pairing(QR.leaf_distances(n), allq)).mean()
    assert hit >= 0.99, hit
