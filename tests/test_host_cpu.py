"""CPU-only tests: the C-ABI library loads and exports every symbol include/splitp_b200.h declares, the
host logic (split enumeration, tree topology, pattern encoding, sharding) and the N>1 plumbing over gloo.
No compute calls are made here (there is no GPU in the build container)."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    from splitp_b200 import _lib
    header = open(os.path.join(ROOT, "include", "splitp_b200.h")).read()
    declared = set(re.findall(r"\b(spb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.PROTOTYPES), (declared ^ set(_lib.PROTOTYPES))
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert _lib.lib.spb_version() == 100
    assert _lib.lib.spb_plane_words(33) == 4 and _lib.lib.spb_sm_words(12, 32) >= 24
    assert _lib.lib.spb_pair_raw_words(20) == 20 * 20 * 9 + 60 + 1
    # argument errors are reported through the status code + message, never abort(): NULL buffers
    assert _lib.lib.spb_pack(None, 4, 10, 10, 0, None, None, None, None) == 1
    assert b"spb_pack" in _lib.lib.spb_last_error()
    with pytest.raises(ValueError):
        _lib.call("spb_count_direct", None, None, 20, 0, 10, None, None, None, None)


def test_no_cpu_fallback_in_product():
    """The product path must fail loudly without a device; nothing under splitp_b200/ imports the oracle."""
    import torch
    import splitp_b200 as sp
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            sp.flattening("01|23", {"ACGT": 1.0})
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            sp.split_score(np.eye(6))
    for dirpath, _, files in os.walk(os.path.join(ROOT, "splitp_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_product_reads_no_tuning_variable():
    """The input alone chooses every kernel and route: the CUDA sources read no environment variable, and the Python package
    reads no SPB_* variable (NVCC, RANK, WORLD_SIZE and LOCAL_RANK are not tuning switches)."""
    csrc = os.path.join(ROOT, "splitp_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh")):
            assert "getenv(" not in open(os.path.join(csrc, f)).read(), f
    spb_read = re.compile(r"""(?:environ\s*(?:\.get\s*\(|\[)|getenv\s*\()\s*[rbf]?["']SPB_""")
    for dirpath, _, files in os.walk(os.path.join(ROOT, "splitp_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not spb_read.search(src), (f, spb_read.search(src))


def test_all_splits_matches_golden(golden_small):
    from splitp_b200.splits import all_splits

    class T:
        def __init__(self, taxa):
            self.taxa = list(taxa)

        def get_taxa(self):
            return self.taxa
    g = golden_small["all_splits"]
    for taxa, d in g.items():
        if taxa == "named5":
            assert [[list(a), list(b)] for a, b in all_splits(T([f"t{i}" for i in range(5)]))] == d
            with pytest.raises(ValueError):
                list(all_splits(T([f"t{i}" for i in range(5)]), string_format=True))
            continue
        t = T(taxa)
        assert [[list(a), list(b)] for a, b in all_splits(t)] == d["default"]
        assert [[list(a), list(b)] for a, b in all_splits(t, trivial=True)] == d["trivial"]
        assert [[list(a), list(b)] for a, b in all_splits(t, size=2)] == d["size2"]
        assert list(all_splits(t, string_format=True)) == d["strings"]
    r = list(all_splits(T("012345"), randomise=True))
    assert sorted(r) == sorted(all_splits(T("012345")))
    with pytest.raises(ValueError):
        next(all_splits(T([str(i) for i in range(40)]), string_format=True))


def test_balanced_tree(golden_readme):
    from splitp_b200.trees import balanced_tree
    t = balanced_tree(10, 0.05)
    assert t.taxa == [str(x) for x in golden_readme["taxa"]]
    assert sorted(t.splits(as_strings=True)) == sorted(str(s) for s in golden_readme["true_splits"])
    assert len(list(balanced_tree(12, 0.05).splits())) == 9
    assert balanced_tree(38).taxa[:3] == ["t0", "t1", "t10"]
    with pytest.raises(ValueError):
        balanced_tree(7)


def test_encode_decode_and_simulator():
    import torch
    from splitp_b200 import engine, simulation, trees
    pats = ["ACGT", "TTTT", "AAAA", "GATC"]
    keys, n = engine.encode_patterns(pats)
    assert n == 4 and keys.tolist() == [0b00011011, 255, 0, 0b10001101]
    assert engine.decode_keys(keys, 4) == pats
    with pytest.raises(KeyError):
        engine.encode_patterns(["ACGU"])
    with pytest.raises(KeyError):
        engine.encode_patterns(["acgt"])  # the reference's __index_of only knows upper case
    tree = trees.balanced_tree(6, 0.1)
    m = simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6))
    Q = m.rate_matrix
    assert abs(-(m.init_dist @ np.diag(Q)) - 1) < 1e-12 and np.allclose(Q.sum(axis=1), 0)
    c = simulation.simulate_codes(tree, m, 20000, seed=1, device="cpu")
    assert c.shape == (6, 20000) and c.dtype == torch.uint8 and int(c.max()) <= 3
    c2 = simulation.simulate_codes(tree, m, 20000, seed=1, device="cpu")
    assert torch.equal(c, c2)
    # siblings agree more often than taxa across the root
    same = lambda i, j: float((c[i] == c[j]).float().mean())  # noqa: E731
    assert same(0, 1) > same(0, 5)


def test_count_scorer_geometry():
    from splitp_b200 import engine
    g = engine.CountScorer.geometry
    assert g(16, 1 << 20) == (2, 16, 1 << 20)
    assert g(64, 262144) == (1, 128, 262144)
    assert g(32, 100) == (2, 32, 112)
    assert g(7, 55) == (2, 8, 64)
    assert g(256, 65536) == (1, 256, 65536)
    assert g(4096, 4096) == (1, 4096, 4096)
    assert g(100, 1000) == (1, 128, 1024)
    assert g(1810, 1814) == (1, 2048, 1920)


def test_shard_range():
    from splitp_b200.distributed import shard_range
    for total, world, align in [(1_000_000, 8, 32), (33, 4, 32), (2035, 8, 1), (5, 8, 1), (0, 2, 32)]:
        cover = []
        for r in range(world):
            b, e = shard_range(total, r, world, align)
            assert 0 <= b <= e <= total and (b % align == 0 or b == total)
            cover += list(range(b, e))
        assert cover == list(range(total))


def test_gloo_world2_plumbing(tmp_path):
    """world_size=2 over gloo on CPU tensors: integer table allreduce, u32 min-reduce of first-site indices,
    variable-length gathers and the score gather are rank-order exact."""
    script = tmp_path / "w2.py"
    script.write_text(f'''
import os, sys
sys.path.insert(0, {ROOT!r})
import torch, torch.distributed as dist
from splitp_b200 import distributed as spd
rank, local, world = spd.init_from_env()
assert world == 2 and dist.get_backend() == "gloo"
fn = spd.make_reduce_fn()
t = torch.arange(10, dtype=torch.int32) * (rank + 1)
fn(t, "sum"); assert t.tolist() == [3 * i for i in range(10)]
f = torch.tensor([-1, 5 + rank, -1 if rank == 0 else 7, -2147483648 + rank], dtype=torch.int32)  # -1 = 0xFFFFFFFF = "unset"
fn(f, "min_u32"); assert f.tolist() == [-1, 5, 7, -2147483648], f.tolist()
v = torch.arange(3 + 4 * rank, dtype=torch.int64) + 100 * rank
g = spd.all_gather_varlen(v); assert g.tolist() == [0, 1, 2] + [100 + i for i in range(7)]
# compacted pattern lists of the direct-table merge: one size exchange, two payloads, rank order kept
gk, gc = spd.make_gather_fn()(v, (v * 2).to(torch.int32))
assert gk.tolist() == g.tolist() and gc.tolist() == [2 * x for x in g.tolist()]
# hash-partitioned exchange: every entry ends up on its owner, nothing is lost, duplicates from both ranks are kept
keys = torch.arange(50, dtype=torch.int64) * 7919 + rank * 3            # ranks share no key ...
keys = torch.cat([keys, torch.tensor([123456789, 42], dtype=torch.int64)])  # ... except these two
cnts = torch.ones_like(keys, dtype=torch.int32) * (rank + 1)
rk, rc = spd.exchange_by_owner(keys, cnts, world)
assert bool((spd._owner_of(rk, world) == rank).all())
tot = torch.tensor([rk.shape[0], int(rc.sum())], dtype=torch.int64); dist.all_reduce(tot)
assert tot.tolist() == [104, 52 * 1 + 52 * 2], tot.tolist()
wk = torch.stack([keys, keys * 31 + 5], dim=1)                             # 128-bit keys (lo, hi)
rk2, rc2 = spd.exchange_by_owner(wk, cnts, world)
assert rk2.shape[1] == 2 and bool((spd._owner_of(rk2, world) == rank).all())
S = 11
b, e = spd.shard_range(S, rank, world)
sc = spd.gather_scores(torch.arange(b, e, dtype=torch.float64), S, rank, world)
assert sc.tolist() == [float(i) for i in range(S)]
mine = spd.shard_strided(list(range(S)), rank, world)
sc = spd.gather_strided(torch.tensor(mine, dtype=torch.float64), S, rank, world)
assert sc.tolist() == [float(i) for i in range(S)]
# cost-balanced partition: arbitrary positions per rank, gathered by a SUM all-reduce of disjoint supports
pos = torch.tensor([10, 0, 3, 7] if rank == 0 else [1, 2, 4, 5, 6, 8, 9], dtype=torch.int64)
sc = spd.gather_by_position(pos.to(torch.float64) * 1.5, pos, S)
assert sc.tolist() == [1.5 * i for i in range(S)]
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
''')
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29517", str(script)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_bench_reference_arm_runs():
    """`bench.py --impl reference`: one JSON line, the unmodified reference from baseline/_ref when it is installed
    (kind "reference"), the oracle port beside it; the process imports neither torch nor splitp_b200."""
    env = dict(os.environ, OMP_NUM_THREADS="1", SPB_BENCH_REPORT_MODULES="1")  # torchrun's setting must not reach BLAS
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--sites", "20000"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr
    import json
    assert len(r.stdout.strip().splitlines()) == 1  # stdout carries exactly one JSON line
    line = json.loads(r.stdout.strip())
    have_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "splitp"))
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["cpu_baseline"]["port"]["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["threads"]["OMP_NUM_THREADS"] == str(line["threads"]["host_cores"])
    assert set(line["config"]) == {"workload", "name", "taxa", "sites", "splits", "model", "branch_length", "seed", "l2", "parallelism"}
    if have_ref:
        assert line["cpu_baseline"]["port_vs_reference_max_rel"] < 1e-9
    assert "torch" not in line["modules"] and "splitp_b200" not in line["modules"]


def test_bench_reference_arm_under_torchrun_env_prints_on_rank0_only():
    """Under torchrun the reference arm runs on rank 0 alone; the other ranks exit 0 without output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0", "--sites", "20000"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_make_splits_matches_make_split():
    """The vectorised split encoder (one numpy pass per batch) produces the same bytes as the per-split ctypes one."""
    from splitp_b200 import _lib
    sides_a = [[0, 1, 2], [3, 5, 7], [11, 0, 4]]
    sides_b = [[3, 4, 5, 6, 7, 8, 9, 10, 11], [0, 1, 2, 4, 6, 8, 9, 10, 11], [1, 2, 3, 5, 6, 7, 8, 9, 10]]
    arr, rec = _lib.make_splits(12, sides_a, sides_b)
    assert len(arr) == 3 and rec.itemsize == 140
    for i, (a, b) in enumerate(zip(sides_a, sides_b)):
        assert bytes(arr[i]) == bytes(_lib.make_split(12, a, b))
    sub = (_lib.SpbSplit * 2).from_buffer(rec, rec.itemsize)  # a batch slice shares the numpy buffer
    assert bytes(sub[1]) == bytes(_lib.make_split(12, sides_a[2], sides_b[2]))
    with pytest.raises(ValueError):
        _lib.make_splits(12, [[0, 12]], [[1, 2]])
    with pytest.raises(ValueError):
        _lib.make_splits(65, [[0]], [[1]])


def test_warp_scorer_model_against_lapack(oracle):
    """The arithmetic of the warp-per-split subflattening scorer (Gram -> Householder tridiagonalisation -> 9-section
    for the 4 largest eigenvalues -> sqrt((trace - top4) / trace)), modelled lane by lane in tests/warp_scorer_model.py,
    stays within the parity tolerance of the reference's LAPACK route: on subflattenings of a simulated 12-taxon
    alignment (true and random splits) and on random matrices up to k = 31, including a rank-deficient one."""
    import torch
    from splitp_b200 import simulation, splits as splits_mod, trees
    from tests.warp_scorer_model import score_warp_model
    eps = np.finfo(float).eps
    n = 12
    tree = trees.balanced_tree(n, 0.05)
    codes = simulation.simulate_codes(tree, simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6)), 100_000, seed=3,
                                      device=torch.device("cpu")).numpy()
    tables, total = oracle.pair_tables_from_codes(codes)
    pos = {t: i for i, t in enumerate(tree.taxa)}
    allsp = list(splits_mod.all_splits(tree))
    true = [s for s in allsp if s in set(tree.splits())]
    rng = np.random.default_rng(5)
    sample = true[:4] + [allsp[i] for i in rng.choice(len(allsp), 8, replace=False)]
    checked = 0
    for s in sample:
        M = oracle.subflattening_from_tables(tables, total, [pos[t] for t in s[0]], [pos[t] for t in s[1]])
        if M.shape[0] > M.shape[1]:
            M = M.T
        if M.shape[0] <= 4:
            continue
        ref = oracle.split_score(M)
        got, lams = score_warp_model(M)
        tol = max(1e-9, 64 * eps / max(ref * ref, 1e-300))
        assert abs(got - ref) <= tol * ref, (s, got, ref)
        sv = np.linalg.svd(M, compute_uv=False)[:4] ** 2
        np.testing.assert_allclose(lams, sv, rtol=0, atol=1e-13 * sv[0])
        checked += 1
    assert checked >= 8
    for k, L in ((31, 31), (7, 55), (5, 9)):
        A = rng.standard_normal((k, L))
        A[2] = 2.0 * A[1]  # exact dependency: a zero eigenvalue
        got, _ = score_warp_model(A)
        sv = np.linalg.svd(A, compute_uv=False) ** 2
        ref = float(np.sqrt(sv[4:].sum() / sv.sum()))
        tol = max(1e-9, 64 * eps / max(ref * ref, 1e-300))  # a vanishing score (k = 5 with a zero eigenvalue) is all rounding
        assert abs(got - ref) <= min(tol * ref, 1e-7) or abs(got - ref) <= 1e-9 * ref, (k, L, got, ref)


# ---------------------------------------------------------------------------------------------
# alignment simulators against the reference's pattern distribution (SURVEY section 8 f2)
# ---------------------------------------------------------------------------------------------
def _chi2_pvalue(observed, expected):
    import scipy.stats
    keep = expected > 0
    assert observed[~keep].sum() == 0
    # pool cells with an expectation below 5 into one (the usual validity rule of the chi-square approximation)
    small = keep & (expected < 5)
    obs = np.concatenate([observed[keep & ~small], [observed[small].sum()]])
    exp = np.concatenate([expected[keep & ~small], [expected[small].sum()]])
    if exp[-1] == 0:
        obs, exp = obs[:-1], exp[:-1]
    stat = ((obs - exp) ** 2 / exp).sum()
    return float(scipy.stats.chi2.sf(stat, len(exp) - 1)), float(stat), len(exp) - 1


def _pattern_counts(codes, patterns):
    n = codes.shape[0]
    keys = np.zeros(codes.shape[1], dtype=np.int64)
    for r in codes:
        keys = keys * 4 + r
    cnt = np.bincount(keys, minlength=4 ** n)
    lut = {c: i for i, c in enumerate("ACGT")}
    idx = [sum(lut[ch] * 4 ** (n - 1 - i) for i, ch in enumerate(p)) for p in patterns]
    return cnt[idx].astype(np.float64), int(cnt.sum() - cnt[idx].sum())


@pytest.fixture(scope="module")
def golden_patternprobs():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "golden_patternprobs.json")) as f:
        return json.load(f)


def test_simulators_match_reference_pattern_probabilities(golden_patternprobs):
    """Chi-square goodness of fit of both generators (splitp_b200.simulation.simulate_codes on the CPU device, and
    bench_inputs.simulate_codes) against the EXACT pattern probabilities the reference computes
    (simulation.get_pattern_probabilities, splitp/simulation.py:71-157) for 4- and 6-taxon Jukes-Cantor trees."""
    import bench_inputs as BI
    from splitp_b200 import simulation, trees
    for case in golden_patternprobs["exact"]:
        n, bl = case["n"], case["branch_length"]
        N = 400_000 if n == 4 else 1_500_000
        probs = np.asarray(case["probs"])
        tree = trees.balanced_tree(n, bl)
        assert list(tree.taxa) == case["taxa"]
        for name, codes in (("torch", simulation.simulate_codes(tree, simulation.GTR.JukesCantor(0.5), N, seed=11, device="cpu").numpy()),
                            ("numpy", BI.simulate_codes(n, bl, "JC", N, seed=11))):
            obs, missing = _pattern_counts(codes, case["patterns"])
            assert missing == 0
            p, stat, dof = _chi2_pvalue(obs, probs * N)
            assert p > 1e-4, (name, n, bl, p, stat, dof)


def test_simulators_match_reference_generate_alignment_gtr(golden_patternprobs):
    """GTR (non-symmetric transition matrix): two-sample chi-square of both generators against a seeded sample of the
    reference's own generate_alignment (splitp/simulation.py:9-56; 4 taxa, 40,000 sites).  The reference draws the child
    state from the NORMALISED column of expm(t Q); without that normalisation this test fails."""
    import bench_inputs as BI
    import scipy.stats
    from splitp_b200 import simulation, trees
    case = golden_patternprobs["sampled"][0]
    n, bl, Nref = case["n"], case["branch_length"], case["sites"]
    ref_counts = dict(zip(case["patterns"], case["counts"]))
    tree = trees.balanced_tree(n, bl)
    N = 2_000_000
    gens = (("torch", simulation.simulate_codes(tree, simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6)), N, seed=5, device="cpu").numpy()),
            ("numpy", BI.simulate_codes(n, bl, "GTR", N, seed=5)))
    import itertools
    patterns = ["".join(p) for p in itertools.product("ACGT", repeat=n)]
    ref = np.asarray([ref_counts.get(p, 0) for p in patterns], dtype=np.float64)
    for name, codes in gens:
        mine, _ = _pattern_counts(codes, patterns)
        expected = mine / N * Nref  # our large sample as the (nearly exact) model for the reference's 40,000 draws
        p, stat, dof = _chi2_pvalue(ref, expected)
        assert p > 1e-4, (name, p, stat, dof)
    # and the un-normalised column (round 1's generator) is rejected by the same test: the fixture has the power to tell
    M = simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6)).transition_matrix(bl)
    assert abs(M.sum(axis=0) - 1).max() > 0.02
    del scipy


def test_simulate_codes_accepts_reference_phylogeny_like_tree():
    """simulate_codes / generate_alignment take the reference's Phylogeny (duck-typed: .networkx_graph with branch_length
    node attributes, .taxa): same alignment as from the equivalent trees.Tree."""
    import networkx as nx
    from splitp_b200 import simulation, trees

    own = trees.balanced_tree(6, 0.07)

    class FakePhylogeny:  # the attributes of splitp.phylogeny.Phylogeny the simulator reads
        def __init__(self, tree):
            g = nx.DiGraph()
            label = {i: (tree.names[i] if i in tree.names else f"n{i}") for i in range(len(tree.parent))}
            for i, p in enumerate(tree.parent):
                g.add_node(label[i], branch_length=tree.branch_length[i] if p >= 0 else None)
            for i, p in enumerate(tree.parent):
                if p >= 0:
                    g.add_edge(label[p], label[i])
            self.networkx_graph = g
            self.taxa = sorted(tree.names.values())

    conv = trees.as_tree(FakePhylogeny(own))
    assert sorted(conv.names.values()) == sorted(own.names.values()) and conv.taxa == own.taxa
    assert sorted(conv.branch_length) == sorted(own.branch_length)
    a = simulation.simulate_codes(FakePhylogeny(own), simulation.GTR.JukesCantor(0.5), 200_000, seed=3, device="cpu").numpy()
    # same topology and branch lengths => same pattern distribution (node numbering, hence the random stream, differs)
    b = simulation.simulate_codes(own, simulation.GTR.JukesCantor(0.5), 4_000_000, seed=4, device="cpu").numpy()  # 20x: "the model"
    import itertools
    patterns = ["".join(p) for p in itertools.product("ACGT", repeat=6)]
    ca, _ = _pattern_counts(a, patterns)
    cb, _ = _pattern_counts(b, patterns)
    p, stat, dof = _chi2_pvalue(ca, np.maximum(cb, 1e-9) / cb.sum() * ca.sum())
    assert p > 1e-4, (p, stat, dof)


def _phylogeny_from_splits(taxa, splits, branch_length):
    """A Phylogeny-shaped object (the attributes trees.as_tree reads: .networkx_graph, a DiGraph parent -> child with the
    branch above each node in its `branch_length` attribute, leaves named by taxon; .taxa) of the rooted binary tree with
    these true splits, rooted on its one split into equal halves (the root of a balanced tree)."""
    import networkx as nx
    everyone = frozenset(taxa)
    halves = [frozenset(a) for a, b in splits if len(a) == len(b)]
    assert len(halves) == 1
    x, y = halves[0], everyone - halves[0]
    clades = {x, y} | {frozenset([t]) for t in taxa}
    for a, b in splits:
        a = frozenset(a)
        clades.add(a if a <= x or a <= y else everyone - a)  # the side that lies within one half hangs below the root
    label = {c: next(iter(c)) if len(c) == 1 else "(" + ",".join(sorted(c)) + ")" for c in clades}
    label[everyone] = "root"
    g = nx.DiGraph()
    g.add_node("root", branch_length=None)
    for c in clades:
        g.add_node(label[c], branch_length=branch_length)
    for c in clades:
        g.add_edge(label[min((p for p in clades | {everyone} if c < p), key=len)], label[c])

    class Phylogeny:
        networkx_graph = g
    Phylogeny.taxa = list(taxa)
    return Phylogeny()


def test_as_tree_on_the_real_reference_phylogeny(golden_readme):
    """The trees the unmodified reference's splitp.trees.balanced_newick_tree returned, as recorded in tests/golden by
    make_golden.py (taxa and true splits: n = 6 and 8 at branch length 0.1 in golden_erickson.json, n = 10 at 0.05 in
    golden_readme.npz), rebuilt as Phylogeny-shaped objects: trees.as_tree gives the reference's taxa, taxa order and splits
    and the branch lengths of the graph, and trees.balanced_tree gives the same taxa, splits and branch lengths.
    With the reference itself installed in baseline/_ref, its own Phylogeny objects for n = 4 .. 20 are converted too."""
    from splitp_b200 import trees
    with open(os.path.join(ROOT, "tests", "golden", "golden_erickson.json")) as f:
        cases = [(rec["n"], 0.1, [[list(a), list(b)] for a, b in rec["true_splits"]]) for rec in json.load(f)]
    cases.append((10, 0.05, [[list(a), list(b)] for a, b in (s.split("|") for s in golden_readme["true_splits"].tolist())]))
    for n, bl, splits in cases:
        taxa = sorted({t for s in splits for side in s for t in side})
        if n == 10:
            assert taxa == [str(t) for t in golden_readme["taxa"]]
        assert len(taxa) == n and len(splits) == n - 3
        conv, own = trees.as_tree(_phylogeny_from_splits(taxa, splits, bl)), trees.balanced_tree(n, bl)
        want = {(tuple(a), tuple(b)) for a, b in splits}
        assert list(conv.taxa) == list(own.taxa) == taxa
        assert set(conv.splits()) == set(own.splits()) == want
        assert sorted(conv.branch_length) == sorted(own.branch_length) == [0.0] + [bl] * (2 * n - 2)
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "splitp")):
        return
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import warnings; warnings.simplefilter('ignore')\n"
        "import splitp\n"
        "from splitp_b200 import trees\n"
        "for n in (4, 6, 10, 12, 20):\n"
        "    ref = splitp.trees.balanced_newick_tree(n, 0.05)\n"
        "    conv, own = trees.as_tree(ref), trees.balanced_tree(n, 0.05)\n"
        "    assert list(conv.taxa) == list(own.taxa) == list(ref.taxa)\n"
        "    assert set(conv.splits()) == set(own.splits()) == set(ref.splits())\n"
        "    assert sorted(conv.branch_length) == sorted(own.branch_length)\n"
        "print('ok')\n" % (ref_dir, ROOT))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_install_reference_is_offline_and_leaves_the_source_alone(tmp_path):
    """__graft_entry__.install_reference (what build() runs when SPLITP_REFERENCE names the reference's source tree) installs
    a pure-Python package without an index into the target, builds from a copy (the source tree stays untouched and may be
    read-only), and refuses a directory that holds no splitp/ package."""
    import __graft_entry__
    src = tmp_path / "SplitP"
    (src / "splitp").mkdir(parents=True)
    (src / "splitp" / "__init__.py").write_text("VERSION = '0.3.2'\n")
    (src / "setup.py").write_text("from setuptools import setup\nsetup(name='splitp', version='0.3.2', packages=['splitp'])\n")
    before = sorted(p.relative_to(src) for p in src.rglob("*"))
    for p in src.rglob("*"):
        p.chmod(p.stat().st_mode & ~0o222)
    src.chmod(src.stat().st_mode & ~0o222)
    try:
        __graft_entry__.install_reference(str(src), str(tmp_path / "_ref"))
    finally:
        for p in [src, *src.rglob("*")]:
            p.chmod(p.stat().st_mode | 0o200)
    assert (tmp_path / "_ref" / "splitp" / "__init__.py").read_text() == "VERSION = '0.3.2'\n"
    assert sorted(p.relative_to(src) for p in src.rglob("*")) == before
    with pytest.raises(FileNotFoundError):
        __graft_entry__.install_reference(str(tmp_path / "_ref" / "splitp"), str(tmp_path / "other"))


def test_warp2_scorer_model_against_lapack(oracle):
    """The arithmetic of the round-2 subflattening scorer (Gram matrix from triple tables -> Householder with two rows per
    lane -> division-free Sturm counts), modelled in tests/warp_scorer_model.py, against LAPACK: subflattenings of simulated
    12- and 20-taxon alignments (k up to 31) and random / rank-deficient Gram matrices up to k = 64."""
    import bench_inputs as BI
    from tests.warp_scorer_model import gram_from_triples, score_warp2_model, triple_tables
    eps = np.finfo(float).eps
    for n, model, N in ((12, "JC", 100_000), (20, "GTR", 150_000)):
        codes = BI.simulate_codes(n, 0.05, model, N, seed=n)
        tables, _ = oracle.pair_tables_from_codes(codes)
        H = oracle.H4.astype(float)
        T = np.einsum("cx,ijxy,dy->ijcd", H, tables, H)
        tabs = triple_tables(T, 1.0)
        rng = np.random.default_rng(n)
        sides = [sorted(rng.choice(n, size=a, replace=False).tolist()) for a in range(2, n // 2 + 1) for _ in range(2)]
        sides.append(list(range(n // 2)))  # the tree's balanced true split
        for side in sides:
            other = [t for t in range(n) if t not in side]
            la, lb = (side, other) if len(side) <= len(other) else (other, side)
            S = oracle.subflattening_from_tables(tables, 1.0, la, lb)
            G = gram_from_triples(tabs, 1.0, la, lb)
            assert np.array_equal(G, G.T)  # bitwise symmetric by construction (mirrored table, commutative products)
            np.testing.assert_allclose(G, S @ S.T, rtol=0, atol=4 * eps * np.abs(S @ S.T).max())
            ref = oracle.split_score(S)
            got, _ = score_warp2_model(G)
            assert abs(got - ref) <= max(1e-9, 64 * eps / ref ** 2) * ref, (n, side, got, ref)
    rng = np.random.default_rng(0)
    for k, L in ((5, 40), (17, 17), (33, 60), (49, 49), (64, 70)):
        M = rng.standard_normal((k, L))
        if k == 17:
            M[5:] = M[:12] * 0.5  # rank deficient
        G = M @ M.T
        lam = np.sort(np.linalg.eigvalsh(G))[::-1]
        ref = np.sqrt(max(lam[4:].sum(), 0.0) / lam.sum())
        got, _ = score_warp2_model(G)
        assert abs(got - ref) <= 1e-12 * max(ref, 1.0), (k, got, ref)


def test_partition_by_cost_balances_the_class_ordered_split_list():
    """distributed.partition_by_cost on the 2,035 splits of 12 taxa: the ranges cover the list once, every rank's modelled time
    (items + one fixed cost per class it touches) is within 3 % of the mean, and most ranks hold a single size class."""
    import bench_inputs as BI
    from splitp_b200 import distributed as spd
    idx = BI.all_splits_idx(12)
    cls = [min(len(a), len(b)) for a, b in idx]
    per = {a: spd.flattening_cost_us(12, a, 60000) for a in set(cls)}
    fixed = {a: spd.flattening_fixed_us(a) for a in per}
    assert per[6] > per[5] > per[4] and per[6] > 3 * per[5]
    order = sorted(range(len(idx)), key=lambda i: (-per[cls[i]], i))
    for world in (1, 2, 3, 8, 16):
        ranges = spd.partition_by_cost([cls[i] for i in order], [per[cls[i]] for i in order], fixed, world)
        assert len(ranges) == world and ranges[0][0] == 0 and ranges[-1][1] == len(idx)
        assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1))
        times, single = [], 0
        for b, e in ranges:
            cs = [cls[order[i]] for i in range(b, e)]
            times.append(sum(per[c] for c in cs) + sum(fixed[c] for c in set(cs)))
            single += len(set(cs)) == 1
        assert max(times) <= 1.03 * (sum(times) / world), (world, times)
        if world == 8:
            assert single >= 5
    # degenerate inputs: fewer items than ranks, one class
    ranges = spd.partition_by_cost([3, 3], [1.0, 1.0], {3: 0.5}, 4)
    assert [e - b for b, e in ranges] == [1, 1, 0, 0]


def test_refit_costs_recovers_class_costs_from_rank_times():
    """distributed.refit_costs: rank times generated from 'true' per-class costs that differ from the model by up to 30 % are
    fitted well enough that the re-cut partition is balanced under the TRUE costs (8 ranks); with 2 ranks the fit stays near
    the model where the data say nothing and still improves the balance."""
    import bench_inputs as BI
    from splitp_b200 import distributed as spd
    idx = BI.all_splits_idx(12)
    cls = [min(len(a), len(b)) for a, b in idx]
    model = {a: spd.flattening_cost_us(12, a, 60000) for a in set(cls)}
    fixed = {a: spd.flattening_fixed_us(a) for a in model}
    truth = {2: model[2] * 1.3, 3: model[3] * 0.8, 4: model[4] * 1.2, 5: model[5] * 0.9, 6: model[6] * 1.05}

    def cut(per, world):
        order = sorted(range(len(idx)), key=lambda i: (-per[cls[i]], i))
        ranges = spd.partition_by_cost([cls[i] for i in order], [per[cls[i]] for i in order], fixed, world)
        held = []
        for b, e in ranges:
            h = {}
            for i in order[b:e]:
                h[cls[i]] = h.get(cls[i], 0) + 1
            held.append(h)
        return held

    def true_times(held):
        return [spd.RANK_BASE_US + sum(n * truth[a] for a, n in h.items()) + sum(fixed[a] for a in h) for h in held]

    for world in (2, 8):
        held = cut(model, world)
        before = true_times(held)
        fitted, fixed_fit = spd.refit_costs(model, fixed, held, before)
        assert all(abs(fixed_fit[a] / fixed[a] - 1) < 0.25 for a in fixed)
        after = true_times(cut(fitted, world))
        assert max(after) < max(before)
        if world == 8:
            assert max(after) <= 1.03 * (sum(after) / world), after
            assert abs(fitted[6] / truth[6] - 1) < 0.03 and abs(fitted[5] / truth[5] - 1) < 0.05


def test_split_scorer_partition_covers_every_split_once():
    """batch.SplitScorer(world = N): the ranks' shares of the flattening scores are disjoint, cover all 2,035 splits of 12 taxa,
    are identical however often they are re-cut from the same costs, and a re-fit from made-up rank times keeps that property
    (host logic only: no device is touched before the first scoring call)."""
    import bench_inputs as BI
    from splitp_b200 import batch
    from splitp_b200 import distributed as spd
    from splitp_b200.enums import Method
    idx = BI.all_splits_idx(12)
    for world in (2, 5, 8):
        scorers = [batch.SplitScorer(idx, None, Method.flattening, r, world, sites="replicated") for r in range(world)]
        seen = sorted(p for s in scorers for p in s.positions)
        assert seen == list(range(len(idx)))
        assert all(len(s.idx_mine) == len(s.positions) for s in scorers)
        assert all(s._held == scorers[0]._held for s in scorers)            # every rank computes the same cut
        assert sum(sum(h.values()) for h in scorers[0]._held) == len(idx)
        # a re-fit with the same (made-up) rank times on every rank: still a partition, still identical on all ranks
        times = [spd.RANK_BASE_US + sum(c * scorers[0]._per[a] * (1.2 if a == 6 else 0.9) + scorers[0]._fixed[a] for a, c in h.items())
                 for h in scorers[0]._held]
        for s in scorers:
            per, fixed = spd.refit_costs(s._per, s._fixed, s._held, times)
            s._per = {a: s._per[a] + s.REFIT_DAMPING * (per[a] - s._per[a]) for a in per}
            s._fixed = {a: s._fixed[a] + s.REFIT_DAMPING * (fixed[a] - s._fixed[a]) for a in fixed}
            s._cut()
        assert sorted(p for s in scorers for p in s.positions) == list(range(len(idx)))
        assert all(s._held == scorers[0]._held for s in scorers)
    assert batch.replicate_sites(12, 1_000_000, 8) and not batch.replicate_sites(12, 1_000_000, 1)
    assert not batch.replicate_sites(20, 100_000_000, 8)
    with pytest.raises(ValueError):
        batch.SplitScorer(idx, None, Method.flattening, 0, 2, sites="everything")
