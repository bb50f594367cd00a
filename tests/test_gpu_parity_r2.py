"""Round-2 GPU parity tests: the kernels behind the headline numbers against the oracle at the sizes they run at.

  * warp-per-split / block subflattening scorers (spb_subflatten_score) at 20, 21, 22 and 32 taxa, stratified over
    every side size, true and false splits, against oracle.split_score(oracle.subflattening_from_tables(...));
  * the batched int32 tensor-core Gram (spb_gram_u8_batch_i32) on random dense u8 4096 x 4096 matrices, nb in
    {1, 3, 64}, bit for bit against an exact integer product;
  * CountScorer.score_many (scatter -> int32 Gram -> correction strip -> block Krylov) on config-2 6|6 splits
    against LAPACK on the reduced flattening;
  * reducible / many-component Gram matrices through the block-Krylov solver (k > 128) against LAPACK;
  * the seven G0 Q product kernels (column-owning FMA kernel, fp64 tensor-core kernels) against a torch fp64 product, bit-exact on
    integer-valued vectors;
  * the correction strip built by a join of the pattern table with the high list against the column scans of S0, bit for bit;
  * the warp-per-matrix scorer of small Gram matrices (k <= 64) and the Jacobi kernel against LAPACK singular values.

Tolerances: integer work bit-exact; scores rel <= max(1e-9, 64 eps / score^2) (tests/test_gpu_parity.py header).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests.test_gpu_gram_compaction import _full_k_scorer  # noqa: E402
from tests.test_gpu_parity import _count_table, _tiled_from_rowmajor, assert_score, score_tol  # noqa: E402


@pytest.fixture(scope="module")
def sp():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import splitp_b200
    return splitp_b200


@pytest.fixture(scope="module")
def eng(sp):
    return sp.engine


# ---------------------------------------------------------------------------------------------
# subflattening scorers at the sizes of BASELINE configs 3 and 5
# ---------------------------------------------------------------------------------------------
def _stratified_splits(tree, n, sizes, per_size, seed):
    """>= per_size splits for every side size: every true split of that size plus random false ones."""
    rng = np.random.default_rng(seed)
    pos = {t: i for i, t in enumerate(tree.taxa)}
    true = {}
    for left, right in tree.splits():
        for side, other in ((left, right), (right, left)):
            if len(side) in sizes and len(side) <= len(other):
                true.setdefault(len(side), set()).add(tuple(sorted(pos[t] for t in side)))
    out = []
    for a in sizes:
        chosen = set(true.get(a, ()))
        n_true = len(chosen)
        while len(chosen) < max(per_size, n_true + per_size // 2):
            chosen.add(tuple(sorted(rng.choice(n, size=a, replace=False).tolist())))
        for side in sorted(chosen):
            out.append((list(side), [t for t in range(n) if t not in side], side in true.get(a, ())))
    return out


@pytest.mark.parametrize("n,model,N,seed", [(20, "GTR", 400_000, 3), (21, "JC", 150_000, 21), (22, "GTR", 150_000, 22),
                                            (32, "JC", 300_000, 5)])
def test_subflatten_score_stratified(sp, eng, oracle, n, model, N, seed):
    """spb_subflatten_score against the oracle for every side size 2 .. n/2 (k = 3a + 1 up to 31 at 20 taxa: the
    warp-per-split kernel; 22 and 32 taxa: the kernel for wider matrices), >= 20 splits per size, true splits included."""
    if n % 2 == 0:
        tree = sp.trees.balanced_tree(n, 0.05)
    else:  # odd taxon count: drop the last leaf of a balanced tree on n + 1 taxa (simulate, then delete the row)
        tree = sp.trees.balanced_tree(n + 1, 0.05)
    mdl = sp.simulation.GTR.JukesCantor(0.5) if model == "JC" else sp.simulation.GTR((0.1, 0.2, 0.3, 0.4), (1, 2, 3, 4, 5, 6))
    codes = sp.simulation.simulate_codes(tree, mdl, N, seed=seed)[:n].contiguous()
    aln = eng.pack(codes, want_sm=False)
    pt = eng.pair_tables_from_alignment(aln)  # probabilities
    tables, usable = oracle.pair_tables_from_codes(codes.cpu().numpy())
    assert usable == N
    sizes = list(range(2, n // 2 + 1))
    if n % 2 == 0:
        picks = _stratified_splits(tree, n, sizes, 20, seed)
    else:
        rng = np.random.default_rng(seed)
        picks = []
        for a in sizes:
            for _ in range(20):
                side = sorted(rng.choice(n, size=a, replace=False).tolist())
                picks.append((side, [t for t in range(n) if t not in side], False))
    ma, mb = eng.masks_from_splits([(ia, ib) for ia, ib, _ in picks])
    got = eng.subflatten_scores(pt, ma, mb).cpu().numpy()
    got_swapped = eng.subflatten_scores(pt, mb, ma).cpu().numpy()
    worst, n_true = 0.0, 0
    for s, (ia, ib, is_true) in enumerate(picks):
        ref = oracle.split_score(oracle.subflattening_from_tables(tables, 1.0, ia, ib))
        assert_score(got[s], ref)
        assert_score(got_swapped[s], ref)
        worst = max(worst, abs(got[s] - ref) / ref / score_tol(ref))
        n_true += is_true
    if n % 2 == 0:
        assert n_true >= n - 3 - n // 2  # the tree's true splits of these sizes were all included
    print(f"subflatten scorer n={n}: {len(picks)} splits, {n_true} true, worst error = {worst:.3f} x tolerance")


# ---------------------------------------------------------------------------------------------
# batched int32 tensor-core Gram at the config-2 shape
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb", [1, 3, 64])
def test_gram_u8_batch_i32_exact_4096(eng, nb):
    """spb_gram_u8_batch_i32 on random DENSE u8 4096 x 4096 matrices (every entry non-zero, 1/16 of them 255) against
    the exact integer product.  Entries <= 255 and K = 4096, so every sum is < 2^28: the fp64 BLAS product on the host
    is exact integer arithmetic and equals the int64 product bit for bit (checked once against numpy int64 on a
    slice).  nb = 64: all 64 distinct matrices are compared on the device against the exact fp64 product of the
    row-major copies, four of them also against the host product."""
    R = K = 4096
    rng = np.random.default_rng(100 + nb)
    s0 = torch.empty((nb, R * K), dtype=torch.uint8, device="cuda")
    host = {}
    rows = torch.empty((nb, R, K), dtype=torch.uint8, device="cuda")
    r_i, k_i = np.meshgrid(np.arange(R), np.arange(K), indexing="ij")
    off = ((r_i // 128) * (K // 128) + k_i // 128) * 16384 + (r_i % 128) * 128 + ((((k_i % 128) >> 4) ^ (r_i & 7)) << 4) + (k_i & 15)
    off_d = torch.from_numpy(off.ravel()).cuda()
    check_host = sorted({0, nb // 3, nb // 2, nb - 1})
    for b in range(nb):
        M = rng.integers(1, 256, size=(R, K), dtype=np.uint8)
        M[rng.random((R, K)) < 1.0 / 16] = 255
        Md = torch.from_numpy(M).cuda()
        rows[b] = Md
        s0[b].scatter_(0, off_d, Md.reshape(-1))
        if b in check_host:
            host[b] = M
    if 0 in host:  # the tiled scatter above equals the documented layout helper
        assert np.array_equal(s0[0, :256 * K].cpu().numpy(), _tiled_from_rowmajor(host[0][:256]))
    Gi = torch.full((nb, R, R), -7, dtype=torch.int32, device="cuda")
    eng.call("spb_gram_u8_batch_i32", eng._p(s0), R * K, nb, R, K, eng._p(Gi), R * R, eng._st())
    torch.cuda.synchronize()
    for b in range(nb):
        A = rows[b].to(torch.float64)
        ref = (A @ A.T)
        assert torch.equal(Gi[b].to(torch.float64), ref), f"matrix {b} of {nb} differs from the exact product"
    for b, M in host.items():
        Mf = M.astype(np.float64)
        ref = Mf @ Mf.T  # exact: integers < 2^28
        sl = M[:64].astype(np.int64) @ M.astype(np.int64).T
        assert np.array_equal(ref[:64].astype(np.int64), sl)
        assert np.array_equal(Gi[b].cpu().numpy().astype(np.int64), ref.astype(np.int64)), f"matrix {b} vs host product"


@pytest.mark.parametrize("R,K,nb", [(256, 512, 150), (512, 1024, 80), (768, 384, 40), (1024, 2048, 37)])
def test_gram_u8_batch_pair_kernel_fp64_exact(eng, R, K, nb):
    """spb_gram_u8_batch with enough matrices that K is not split: the CTA-pair (cta_group::2) kernel with the fp64
    epilogue, diagonal and off-diagonal 256-blocks, mirrored halves, odd numbers of work items per pair.  Bit-exact
    against the integer product."""
    rng = np.random.default_rng(R + K + nb)
    M = rng.integers(0, 256, size=(nb, R, K), dtype=np.uint8)
    M[rng.random((nb, R, K)) < 0.5] = 0
    M[0] = 255
    s0 = torch.from_numpy(np.stack([_tiled_from_rowmajor(M[b]) for b in range(nb)])).cuda()
    G = torch.full((nb, R, R), -1.0, dtype=torch.float64, device="cuda")
    n_ws = int(eng.lib.spb_gram_u8_ws(R, K, 1, nb))
    assert n_ws == 0, "this shape is meant to run without a K split"
    eng.call("spb_gram_u8_batch", eng._p(s0), R * K, nb, R, K, 1, eng._p(G), R * R, None, eng._st())
    torch.cuda.synchronize()
    Mf = M.astype(np.float64)
    ref = np.stack([Mf[b] @ Mf[b].T for b in range(nb)])  # exact: integers < 2^53
    np.testing.assert_array_equal(G.cpu().numpy(), ref)


def test_score_many_config2_six_six_vs_lapack(sp, eng, oracle):
    """The bench's hot route (score_many -> u8 scatter -> spb_gram_u8_batch_i32 -> correction strip ->
    spb_score_gram_large_i32) on 18 6|6 splits of the config-2 alignment (12 taxa, 10^6 sites), 8+ of them false,
    against LAPACK gesdd on the reduced flattening (phylogenetics.py:280-300)."""
    n, N = 12, 1_000_000
    tree, codes, tab = _count_table(sp, eng, n, N, 2)
    keys, counts, usable = oracle.get_pattern_counts_arrays(codes)
    true = set(tree.splits())
    sixes = [s for s in sp.all_splits(tree) if len(s[0]) == 6]
    t_splits = [s for s in sixes if s in true]
    f_splits = [s for s in sixes if s not in true]
    picks = t_splits + f_splits[:: max(1, len(f_splits) // 17)][:17]
    assert len(picks) >= 16 and len(picks) - len(t_splits) >= 8
    idx = [eng.split_positions(s, tree.taxa) for s in picks]
    scorer = eng.CountScorer(tab)
    layout, rows_pad, pitch = scorer.geometry(4096, 4096)
    assert scorer._use_i32(layout, rows_pad, pitch)
    got = scorer.score_many(idx).cpu().numpy()
    worst = 0.0
    for s, (ia, ib) in enumerate(idx):
        ref = oracle.split_score(oracle.flattening_reduced(keys, counts / usable, n, ia, ib))
        assert_score(got[s], ref)
        worst = max(worst, abs(got[s] - ref) / ref / score_tol(ref))
    print(f"score_many 6|6: {len(picks)} splits ({len(t_splits)} true), worst error = {worst:.3f} x tolerance")


# ---------------------------------------------------------------------------------------------
# block-Krylov solver on reducible Gram matrices (ADVICE round 1: start block confined to one component)
# ---------------------------------------------------------------------------------------------
def _blockdiag(blocks):
    k = sum(b.shape[0] for b in blocks)
    c = sum(b.shape[1] for b in blocks)
    out = np.zeros((k, c))
    r0 = c0 = 0
    for b in blocks:
        out[r0:r0 + b.shape[0], c0:c0 + b.shape[1]] = b
        r0 += b.shape[0]
        c0 += b.shape[1]
    return out


def _reducible_cases():
    rng = np.random.default_rng(7)
    cases = {}
    # the advisor's example: 8 heavy isolated rows hide the dominant component from a heaviest-rows start block
    cases["advice"] = _blockdiag([20.0 * np.eye(8), np.ones((200, 200))])
    # many small disjoint components, dominant eigenvalues spread over different ones
    cases["many"] = _blockdiag([rng.integers(0, 6, size=(s, s + 3)).astype(float) for s in (3, 5, 9, 17, 33, 40, 31, 12, 7, 4, 2, 60)])
    # two equal-sized dense components plus isolated heavy diagonal entries
    cases["twins"] = _blockdiag([rng.random((90, 120)), rng.random((90, 120)) * 1.01, np.diag(np.linspace(30, 40, 12))])
    # sparse count-like flattening: few non-zeros per row, many connected components
    S = np.zeros((400, 900))
    for r in range(400):
        for c in rng.choice(900, size=2, replace=False):
            S[r, c] = rng.integers(1, 50)
    cases["sparse"] = S
    return cases


@pytest.mark.parametrize("name", ["advice", "many", "twins", "sparse"])
def test_split_score_reducible_gram(sp, oracle, name):
    A = _reducible_cases()[name]
    assert min(A.shape) > 128
    ref = oracle.split_score(A)
    assert_score(sp.split_score(A), ref)
    assert_score(sp.split_score(A.T), ref)


def test_sub_alignment_keeps_integer_counts(sp):
    """Alignment.sub_alignment of an integer-count alignment returns ints, like the reference's dict arithmetic
    (alignment.py:26-30)."""
    aln = sp.Alignment({"ACGT": 3, "ACGA": 2, "TCGT": 5, "AAAA": 1}, ("w", "x", "y", "z"))
    sub = aln.sub_alignment(("x", "y"))
    assert dict(sub) == {"CG": 10, "AA": 1} and all(type(v) is int for v in sub.values())
    fl = sp.Alignment({"ACGT": 0.25, "ACGA": 0.75}, ("w", "x", "y", "z")).sub_alignment(("w", "z"))
    assert dict(fl) == {"AT": 0.25, "AA": 0.75}


def test_score_gram_large_reports_convergence(sp, eng):
    """Every matrix of a batch reports a converged flag in info[:, 2] semantics (residual) and the call raises no
    error for well-conditioned input; the flag column (info[:, 4] = cycles) stays within the cycle budget."""
    rng = np.random.default_rng(11)
    A = torch.from_numpy(rng.random((3, 200, 260))).cuda()
    G = eng.gram_f64(A)
    scores, info = eng.score_gram(G, want_info=True)
    info = info.cpu().numpy()
    assert np.isfinite(scores.cpu().numpy()).all()
    assert (info[:, 4] >= 1).all() and (info[:, 4] <= 40).all()


# ---------------------------------------------------------------------------------------------
# erickson_SVD: ORDER of the picks wherever the reference's own margin is far above rounding noise
# ---------------------------------------------------------------------------------------------
def test_erickson_pick_order_matches_reference_trace(sp):
    """tests/golden/golden_erickson_trace.json holds, for every agglomeration step of the reference's erickson_SVD
    (all three scoring methods, taken from its own show_work output), the chosen split, its score and the runner-up's
    score.  Wherever best and runner-up are separated by more than 1e-6 relative, the batched implementation must pick the
    same split at the same step and reproduce the best score within the parity tolerance; steps the reference decides
    by last-bit noise (exact ties between the two orientations of one bipartition) are compared as sets only."""
    import json
    import os
    here = os.path.join(os.path.dirname(__file__), "golden")
    with open(os.path.join(here, "golden_erickson.json")) as f:
        cases = json.load(f)
    with open(os.path.join(here, "golden_erickson_trace.json")) as f:
        traces = json.load(f)
    with open(os.path.join(here, "golden_rank1.json")) as f:
        mi_cases = json.load(f)["erickson"]
    pinned = 0
    for ci, (rec, tr) in enumerate(zip(cases, traces)):
        for method in (sp.Method.flattening, sp.Method.subflattening, sp.Method.mutual_information):
            if method == sp.Method.mutual_information:
                # the MI goldens were generated from their own alignments: use the matching record when sizes agree
                continue
            aln = dict(zip(rec["patterns"], rec["values"]))
            mine = []
            got = sp.erickson_SVD(aln, method=method, trace=mine)
            assert len(got) == len(tr[method.name]) == len(mine)
            in_step = True
            for step, (ref_step, my_step) in enumerate(zip(tr[method.name], mine)):
                best, second = ref_step["best"], ref_step["second"]
                decisive = second is not None and best > 0 and (second - best) > 1e-6 * abs(second)
                if not (in_step and decisive):
                    # a noise-decided step may legitimately differ; after it the cluster states can diverge
                    if [list(s) for s in my_step["chosen"]] != ref_step["chosen"]:
                        in_step = False
                    continue
                assert [list(s) for s in my_step["chosen"]] == ref_step["chosen"], (ci, method, step)
                my_best = min(v for v in my_step["scores"].values() if v == v)
                assert_score(my_best, best)
                pinned += 1
    assert pinned >= 8, pinned
    for rec in mi_cases:  # mutual information: every step of these goldens has a margin > 6e-6 (make_golden.py: rank1)
        aln = dict(zip(rec["patterns"], rec["values"]))
        mine = []
        got = [list(map(list, s)) for s in sp.erickson_SVD(aln, method=sp.Method.mutual_information, trace=mine)]
        assert got == rec["mutual_information"]


@pytest.mark.parametrize("n,seed", [(20, 7), (22, 8), (44, 9)])
def test_subflatten_score_staged_kernels_still_agree(sp, eng, oracle, n, seed):
    """The kernels that stage the subflattening (round 1: warp-per-split up to 21 taxa, block-wide Jacobi above) remain the
    route for more than 43 taxa; below that they are called through their C entry point spb_subflatten_score.  Both routes
    against the oracle."""
    N = 120_000
    tree = sp.trees.balanced_tree(n, 0.05)
    codes = sp.simulation.simulate_codes(tree, sp.simulation.GTR.JukesCantor(0.5), N, seed=seed)
    pt = eng.pair_tables_from_alignment(eng.pack(codes, want_sm=False))
    tables, _ = oracle.pair_tables_from_codes(codes.cpu().numpy())
    rng = np.random.default_rng(seed)
    picks = []
    for a in range(2, n // 2 + 1):
        for _ in range(6):
            side = sorted(rng.choice(n, size=a, replace=False).tolist())
            picks.append((side, [t for t in range(n) if t not in side]))
    ma, mb = eng.masks_from_splits(picks)
    dev = torch.device("cuda")
    da, db = (torch.from_numpy(m.view(np.int64)).to(dev) for m in (ma, mb))
    staged = torch.empty(len(picks), dtype=torch.float64, device=dev)
    eng.call("spb_subflatten_score", eng._p(pt.T), eng._p(pt.total), pt.n, eng._p(da), eng._p(db), len(picks), eng._p(staged), eng._st())
    staged = staged.cpu().numpy()
    default = eng.subflatten_scores(pt, ma, mb).cpu().numpy()
    assert (pt.triples is not None) == (n <= eng.SUBFLATTEN_TABLES_MAX_TAXA)
    for s, (ia, ib) in enumerate(picks):
        ref = oracle.split_score(oracle.subflattening_from_tables(tables, 1.0, ia, ib))
        assert_score(staged[s], ref)
        assert_score(default[s], ref)


# ---------------------------------------------------------------------------------------------
# G0 Q product kernels of the eigen-solver (column-owning FMA kernel and the fp64 tensor-core kernel)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,nb", [(256, 3), (1024, 5), (4096, 2)])
@pytest.mark.parametrize("variant", [0, 1])
def test_symv_i32_kernels_against_fp64_matmul(eng, k, nb, variant):
    """AQ[c][j] = sum_i G0[i][j] Q[c][i] with G0 entries up to 2^31 - 1: the column-owning kernel (0) and the DMMA kernel (1)
    within 64 eps of the fp64 product (the kernels differ only in summation order); integer-valued Q gives a bit-exact answer."""
    import ctypes as C
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(100 + k + variant)
    G = torch.randint(0, (1 << 31) - 1, (nb, k, k), dtype=torch.int32, device=dev, generator=g)
    G[0, 5, 7] = (1 << 31) - 1
    lib = eng.lib
    Qt = torch.empty(int(lib.spb_symv_i32_ws(k, nb)), dtype=torch.float64, device=dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for integral in (True, False):
        if integral:
            Q = torch.randint(-3, 4, (nb, 8, k), device=dev, generator=g).to(torch.float64)
        else:
            Q = torch.randn((nb, 8, k), dtype=torch.float64, device=dev, generator=g)
        AQ = torch.full_like(Q, float("nan"))
        rc = lib.spb_symv_i32(G.data_ptr(), k, k, nb, Q.data_ptr(), AQ.data_ptr(), Qt.data_ptr(), variant, st)
        assert rc == 0, lib.spb_last_error()
        ref = torch.stack([Q[b] @ G[b].double() for b in range(nb)])
        if integral:  # |sum| < 4096 * 3 * 2^31 < 2^53: exact in any order
            assert torch.equal(AQ, ref)
        else:
            bound = 64 * np.finfo(np.float64).eps * (Q.abs() @ G.double().abs()).max().item()
            assert (AQ - ref).abs().max().item() <= bound


# ---------------------------------------------------------------------------------------------
# correction strip: join of the pattern table with the high list against the column scans of S0
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("a", [5, 6])
def test_correction_strip_from_table_equals_column_scan(sp, eng, a):
    """The scorer's strip (spb_gram_hi_strip_batch_table_cols on ranked columns) against spb_gram_hi_strip_batch (column
    scans of S0, as the full-K reference scorer builds it) on the same splits (12 taxa, 10^6 sites): pos, hr, hm, G and the
    strip rows in use agree bit for bit (integer-valued fp64 sums)."""
    n, N = 12, 1_000_000
    tree, codes, tab = _count_table(sp, eng, n, N, 2)
    splits = [s for s in sp.all_splits(tree) if len(s[0]) == a][::37][:9]
    idx = [eng.split_positions(s, tree.taxa) for s in splits]
    got = {}
    for route, scorer in (("table", eng.CountScorer(tab)), ("scan", _full_k_scorer(eng, tab))):
        R, Ccols = 4 ** a, 4 ** (n - a)
        layout, rows_pad, pitch = scorer.geometry(R, Ccols)
        assert scorer._use_i32(layout, rows_pad, pitch)
        s0 = scorer._buffers(layout, rows_pad, pitch, len(idx))[0]
        buf = scorer._buffers_i32(rows_pad, len(idx))
        buf["Cs"].fill_(float("nan"))  # rows >= hm are never written by the table form and never read
        scorer._gram_batch_i32([scorer._plan(ia, ib, False)[0] for ia, ib in idx], s0, buf, 0, layout, rows_pad, pitch)
        torch.cuda.synchronize()
        got[route] = {k: v[: len(idx)].clone() for k, v in buf.items()}
    for key in ("pos", "hm", "G"):
        assert torch.equal(got["table"][key], got["scan"][key]), key
    for b in range(len(idx)):
        m = int(got["table"]["hm"][b].item())
        assert m > 0
        assert torch.equal(got["table"]["hr"][b, :m], got["scan"]["hr"][b, :m])
        assert torch.equal(got["table"]["Cs"][b, :m], got["scan"]["Cs"][b, :m])


# ---------------------------------------------------------------------------------------------
# small Gram matrices: warp-per-matrix Householder + 9-section against the Jacobi kernel and LAPACK
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [5, 16, 31, 32, 33, 34, 63, 64])
def test_score_gram_small_warp_path_against_lapack(eng, k):
    """engine.score_gram without the eigenvalue list takes the warp-per-matrix kernel (k <= 64); with it, the Jacobi kernel.
    Both against LAPACK singular values of integer count flattenings with planted rank-4 structure (small scores)."""
    rng = np.random.default_rng(40 + k)
    mats, want = [], []
    for t in range(24):
        cols = 4 * k + 7
        base = rng.integers(1, 2000, size=(k, 4)).astype(np.float64) @ rng.integers(1, 50, size=(4, cols)).astype(np.float64)
        noise = rng.poisson(0.5 if t % 2 else 30.0, size=(k, cols)).astype(np.float64)
        F = base + noise
        G = F @ F.T  # exact: integers far below 2^53
        sv = np.linalg.svd(F, compute_uv=False)  # the reference's route (phylogenetics.py:282-300)
        want.append(np.sqrt((sv[4:] ** 2).sum() / (sv ** 2).sum()))
        mats.append(G)
    G = torch.from_numpy(np.stack(mats)).cuda()
    fast = eng.score_gram(G, k).cpu().numpy()
    slow, eig = eng.score_gram(G, k, want_info=True)
    for f, s, w in zip(fast, slow.cpu().numpy(), want):
        assert_score(f, w)
        assert_score(s, w)


# ---------------------------------------------------------------------------------------------
# straggler compaction of the block-Krylov solver
# ---------------------------------------------------------------------------------------------
def test_solver_compacts_stragglers_in_a_large_batch(sp, eng, oracle):
    """A batch of 24 Gram matrices (k = 256) in which a few need more than two Krylov cycles (flat spectra, a reducible
    matrix) while the rest are accepted in the first: engine.score_gram gives every matrix the first two cycles and re-solves
    only the open ones as a batch of their own.  Every score against LAPACK; the easy matrices report <= 2 cycles."""
    rng = np.random.default_rng(21)
    k, cols = 256, 300
    mats, hard = [], []
    for t in range(24):
        if t in (3, 11, 17):      # nearly flat spectrum: slow convergence of the top-4 subspace
            F = rng.random((k, cols)) * 0.02 + np.eye(k, cols) * (1.0 + 0.001 * rng.random(k))[:, None]
            hard.append(t)
        elif t == 20:             # reducible: isolated heavy rows next to a dense component
            F = np.zeros((k, cols))
            F[:8, :8] = 20.0 * np.eye(8)
            F[8:, 8:] = 1.0 + 0.01 * rng.random((k - 8, cols - 8))
            hard.append(t)
        else:                     # rank-4 structure plus noise: accepted after one cycle
            F = rng.integers(1, 200, size=(k, 4)).astype(np.float64) @ rng.integers(1, 9, size=(4, cols)).astype(np.float64)
            F = F + rng.poisson(2.0, size=(k, cols))
        mats.append(F)
    A = torch.from_numpy(np.stack(mats)).cuda()
    G = eng.gram_f64(A)
    scores, info = eng.score_gram(G, want_info=True)
    scores, info = scores.cpu().numpy(), info.cpu().numpy()
    assert (info[:, 8] == 1.0).all()                       # everything converged in the end
    easy = [t for t in range(24) if t not in hard]
    assert (info[easy, 4] <= eng.FIRST_CYCLES).all()
    assert (info[hard, 4] > eng.FIRST_CYCLES).any()      # the second, compacted call really happened
    for t in range(24):
        assert_score(scores[t], oracle.split_score(mats[t]))
    # the same matrices one by one (small batches take the solver's full budget directly): identical scores
    for t in (0, 3, 20):
        one = float(eng.score_gram(G[t:t + 1])[0].item())
        assert_score(one, scores[t])


# ---------------------------------------------------------------------------------------------
# bench.py --dump-outputs: the scores of the last timed step
# ---------------------------------------------------------------------------------------------
def test_bench_dump_outputs_holds_the_workload_scores(sp, oracle, tmp_path):
    """bench.py --steps 2 --dump-outputs DIR on c2 at 20,000 sites (all 2,035 splits): the JSON line reports two timed steps and
    names the dump, and DIR/c2_scores.npy holds one float64 score per split.  Every 32nd split (64 of them, every side size
    2 .. 6, so the 6|6 tensor-core Gram path too) is within the score tolerance of the oracle's score of the same seeded
    alignment."""
    import json
    import os
    import subprocess
    import sys

    import bench_inputs as BI
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0", "--sites", "20000",
                        "--extras", "none", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and len(line["ms_steps_rank0"]) == 2 and line["dumped"] == "c2_scores.npy"
    got = np.load(tmp_path / "c2_scores.npy")
    idx = BI.all_splits_idx(12)
    assert got.dtype == np.float64 and got.shape == (len(idx),) == (2035,)
    keys, counts, usable = oracle.get_pattern_counts_arrays(BI.simulate_codes(12, 0.05, "JC", 20_000, 2))
    picks = range(0, len(idx), 32)
    assert {min(len(idx[s][0]), len(idx[s][1])) for s in picks} == {2, 3, 4, 5, 6}
    for s in picks:
        ia, ib = idx[s]
        assert_score(got[s], oracle.split_score(oracle.flattening_reduced(keys, counts / usable, 12, ia, ib)))
