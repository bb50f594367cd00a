"""Drop-in `split_score` (reference: splitp/phylogenetics.py:280-328).

    score = sqrt(1 - sum_{i<4} sigma_i^2 / sum_i sigma_i^2),  sigma = singular values of the matrix

sigma_i^2 are the eigenvalues of the Gram matrix on the short side, computed on the device
(fp64 Gram kernel + shared-memory Jacobi / block-Krylov Rayleigh-Ritz, csrc/score.cu).  K = 4 is
hard-coded as in the reference.  Tolerance against the reference's LAPACK path: 1e-9 relative, or the
conditioning floor c*eps/score^2 when that is larger (DESIGN.md, "score conditioning").
"""
from __future__ import annotations

from itertools import combinations

import numpy as np
import scipy.sparse
import torch

from . import engine
from .enums import Method


def is_sparse(matrix):
    return scipy.sparse.issparse(matrix)


def split_score(matrix, return_singular_values=False, force_frob_norm_on_dense=False, data_table_for_frob_norm=None):
    """Split score of a flattening / subflattening.  The three keyword arguments are accepted for
    signature compatibility; the reference ignores them too (phylogenetics.py:321-328 passes them to
    parameters that are never read or are unreachable)."""
    if isinstance(matrix, torch.Tensor):
        return engine.score_matrix(matrix.to(engine.device(), torch.float64))[0]
    if is_sparse(matrix):
        if min(matrix.shape) <= 4:
            # scipy.sparse.linalg.svds(k=4) in the reference (phylogenetics.py:306) refuses these
            raise ValueError(f"`k` must be an integer satisfying `0 < k < min(A.shape)`: min(shape)={min(matrix.shape)}")
        coo = matrix.tocoo()
        ur, ri = np.unique(coo.row, return_inverse=True)
        uc, ci = np.unique(coo.col, return_inverse=True)
        dev = engine.device()
        dense = torch.zeros((len(ur), len(uc)), dtype=torch.float64, device=dev)
        if len(coo.data):
            dense[torch.from_numpy(ri).to(dev), torch.from_numpy(ci).to(dev)] = torch.from_numpy(
                np.asarray(coo.data, dtype=np.float64)).to(dev)
        if min(dense.shape) <= 4:
            return 0.0
        return float(engine.score_matrix(dense)[0].item())  # the sparse path returns a Python float (:312)
    m = np.array(matrix, dtype=np.float64)
    if m.ndim != 2:
        raise ValueError("expected a matrix")
    if min(m.shape) == 0:
        return np.float64("nan")
    dev = engine.device()
    return np.float64(engine.score_matrix(torch.from_numpy(np.ascontiguousarray(m)).to(dev))[0].item())


def _device_matrix(flattening):
    m = np.asarray(flattening.todense() if is_sparse(flattening) else flattening, dtype=np.float64)
    if m.ndim != 2:
        raise ValueError("expected a matrix")
    return torch.from_numpy(np.ascontiguousarray(m)).to(engine.device())


def flattening_rank_1_approximation(flattening, return_vectors=False, dont_compute_matrix=False):
    """r = column sums, c = row sums of the flattening; approximation = r^T c, a (#columns x #rows) array as in the
    reference (phylogenetics.py:331-341).  Sums and outer product are computed on the device."""
    F = _device_matrix(flattening)
    c, r = engine.marginals_dense(F)
    approximation = None if dont_compute_matrix else engine.outer(r, c).cpu().numpy()
    if return_vectors:
        return approximation, r.cpu().tolist(), c.cpu().tolist()
    return approximation


def flattening_rank_k_approximation(split, alignment):
    """Sum over the four states of (column sums with the state banned on the rows)^T (row sums with the state banned
    on the columns): a (4^|B| x 4^|A|) csr_matrix (phylogenetics.py:344-361).  The taxon order is the sorted union
    of both sides, as in the reference."""
    split = (list(split[0]), list(split[1]))
    taxa = sorted(set(split[0]) | set(split[1]))
    idx_a, idx_b = engine.split_positions(split, taxa)
    table = engine.table_from_mapping(alignment)
    if isinstance(table, engine.WidePatternTable):
        raise NotImplementedError(f"flattening_rank_k_approximation: at most {engine.NARROW_MAX_TAXA} taxa (the banned-state "
                                  f"marginals read uint64 pattern keys); this alignment has {table.n}")
    R, Cn = 4 ** len(idx_a), 4 ** len(idx_b)
    if R * Cn > 1 << 28 or R > engine.MI_DIRECT_CELLS or Cn > engine.MI_DIRECT_CELLS:
        raise MemoryError(f"flattening_rank_k_approximation: a dense {Cn} x {R} result does not fit")
    out = torch.zeros((Cn, R), dtype=torch.float64, device=engine.device())
    div = table.divisor if (table.counts is not None and table.divisor > 0) else 1.0
    for code in range(4):
        _, cs = engine.table_marginals(table, idx_a, idx_b, ban_row=code)
        rs, _ = engine.table_marginals(table, idx_a, idx_b, ban_col=code)
        colsum = torch.div(cs.sums, torch.full_like(cs.sums, div))
        rowsum = torch.div(rs.sums, torch.full_like(rs.sums, div))
        engine.outer(colsum, rowsum, out, accumulate=True)
    return scipy.sparse.csr_matrix(out.cpu().numpy())


def flattening_rank_1_approximation_divergence(flattening):
    """sum over the non-zero cells of F[x,y] log(F[x,y] / (r[y] c[x])) (phylogenetics.py:364-373), on the device."""
    return np.float64(engine.rank1_divergence_dense(_device_matrix(flattening)).item())


def _leaves(cluster):
    return (cluster,) if isinstance(cluster, str) else tuple(cluster)


FLATTENING_DENSE_MAX_TAXA = 12   # batched dense route of erickson_SVD(Method.flattening): 4^n cells per split (134 MB at 12 taxa)
FLATTENING_BATCH_BYTES = 4 << 30


def _flattening_scores_batched(table, idx_list):
    """split_score(flattening(split, aln, FlatFormat.reduced)) for many splits that cover all taxa, without a host round
    trip per split: the DENSE flattening of every split (rows = its shorter side; transposing changes no singular
    value, and the all-zero rows / columns the reduced format drops add only zero singular values) goes into one batch
    per side size, followed by ONE batched fp64 Gram and ONE batched eigen-solver call per batch.  A reduced matrix with
    min(shape) <= 4 scores exactly 0.0 (at most 4 singular values), as split_score gives for the materialised matrix."""
    dev = engine.device()
    out = torch.zeros(len(idx_list), dtype=torch.float64, device=dev)
    groups = {}
    for s, (ia, ib) in enumerate(idx_list):
        short, long_ = (ia, ib) if len(ia) <= len(ib) else (ib, ia)
        groups.setdefault(len(short), []).append((s, short, long_))
    n = table.n
    for a, members in groups.items():
        R, Cc = 4 ** a, 4 ** (n - a)
        if R <= 4:
            continue  # at most 4 rows: score 0
        per = max(1, int(FLATTENING_BATCH_BYTES // (R * Cc * 8 + R * R * 8)))
        for c0 in range(0, len(members), per):
            chunk = members[c0:c0 + per]
            F = engine._empty((len(chunk), R, Cc), torch.float64)
            vp, kind, div = table.val_args()
            for j, (_, short, long_) in enumerate(chunk):
                sp = engine.make_split(n, short, long_)
                engine.call("spb_flatten_dense_w", engine._p(table.keys), vp, kind, div, table.num, engine.C.byref(sp),
                            engine._p(F[j]), None, engine._st())
            G = engine.gram_f64(F)
            sc = engine.score_gram(G, R)
            used_rows = (torch.diagonal(G, dim1=1, dim2=2) > 0).sum(dim=1)
            used_cols = (F != 0).any(dim=1).sum(dim=1)
            sc = torch.where((used_rows <= 4) | (used_cols <= 4), torch.zeros_like(sc), sc)
            out.index_copy_(0, torch.tensor([s for s, _, _ in chunk], dtype=torch.int64, device=dev), sc)
            del F, G
    return out


def erickson_SVD(alignment, taxa=None, method=Method.flattening, show_work=False, trace=None):
    """Agglomerative tree inference from split scores (reference: splitp/phylogenetics.py:99-171).

    At every step each pair of current clusters is joined tentatively, the split (joined leaves | all other leaves)
    is scored -- reduced flattening + split score (`Method.flattening`) or subflattening + split score
    (`Method.subflattening`) -- and the best-scoring pair is merged; scores are memoised per split.  Returns the
    n - 2 chosen splits as sorted 2-tuples of leaf tuples, like the reference.  The candidate splits of a step are
    scored as ONE batch on the device: the batched subflattening kernel for `Method.subflattening`; for
    `Method.flattening` (up to 12 taxa) the dense flattenings of a whole side-size class, one batched fp64 Gram and one
    batched eigen-solver call; for `Method.mutual_information` the divergences are queued for all candidates and read back
    once per step.  `trace` (an optional list, not in the reference's signature) receives the candidate scores of every step.  `Method.mutual_information` scores a split by the rank-1 divergence of
    its flattening (phylogenetics.py:136-140, 364-373), computed straight from the pattern table.  `Method.distance`
    leaves every score at infinity, as the reference does.
    """
    table = engine.table_from_mapping(alignment)
    num_taxa = table.n
    if isinstance(table, engine.WidePatternTable) and method in (Method.flattening, Method.mutual_information):
        # every candidate split joins a few taxa against all others: above 31 taxa its long side has more than 4^31 indices
        raise NotImplementedError(f"erickson_SVD({method}): at most {engine.NARROW_MAX_TAXA} taxa; above that use "
                                  f"Method.subflattening (this alignment has {num_taxa} taxa)")
    if taxa is None:
        taxa = [str(np.base_repr(i, base=max(i + 1, 2))) if num_taxa <= 36 else f"t{i}" for i in range(num_taxa)]
    known = {}
    pair_tables = None

    def positions(split):
        # same taxa order as flattening(): the mapping's .taxa, else the sorted union of both sides (constructions.py:21-24)
        order = alignment.taxa if hasattr(alignment, "taxa") else sorted(set(split[0]) | set(split[1]))
        return engine.split_positions(split, order)

    def score_new(splits):
        nonlocal pair_tables
        if method == Method.subflattening:
            if pair_tables is None:
                pair_tables = engine.pair_tables_from_table(table)
            idx = [positions(s) for s in splits]
            for ia, ib in idx:
                if not engine.covers_all(table.n, ia, ib):
                    raise KeyError(min(set(range(table.n)) - set(ia) - set(ib)))  # as subflattening() would
            ma, mb = engine.masks_from_splits(idx)
            return [np.float64(v) for v in engine.subflatten_scores(pair_tables, ma, mb).cpu().numpy()]
        if method == Method.flattening:
            idx = [positions(s) for s in splits]
            if table.n <= FLATTENING_DENSE_MAX_TAXA and all(engine.covers_all(table.n, ia, ib) for ia, ib in idx):
                # one batch per side size: no per-split host synchronisation (ONE device -> host copy per step)
                return [np.float64(v) for v in _flattening_scores_batched(table, idx).cpu().numpy()]
            out = []
            for ia, ib in idx:
                F = engine.flatten_reduced(table, ia, ib)
                out.append(np.float64(0.0) if min(F.shape) <= 4 else np.float64(engine.score_matrix(F)[0].item()))
            return out
        if method == Method.mutual_information:
            # every divergence stays on the device until the whole step is queued: ONE device -> host copy per step
            vals = torch.cat([engine.rank1_divergence(table, *positions(s)).reshape(1) for s in splits])
            return [np.float64(v) for v in vals.cpu().numpy()]
        return [np.inf] * len(splits)  # the reference leaves the score at infinity for the other methods

    def score_canonical(splits):
        """Both orientations of one bipartition ((A, B) and (B, A)) get the SAME float: the score is orientation-free
        mathematically (transposed matrix), but computed twice it differs in the last bits (order of the atomic sums), and
        erickson's `min` over candidates that contain both orientations would then be decided by that noise -- the
        reference's own LAPACK results for F and F^T coincide exactly on its golden runs (best == runner-up in its
        show_work trace), where `min` keeps the first candidate.  Scoring each bipartition once reproduces that."""
        canon = [s if s[0] <= s[1] else (s[1], s[0]) for s in splits]
        todo = []
        for c in canon:
            if c not in canonical_scores and c not in todo:
                todo.append(c)
        if todo:
            canonical_scores.update(zip(todo, score_new(todo)))
        return [canonical_scores[c] for c in canon]

    canonical_scores = {}
    chosen = []
    while len(chosen) < num_taxa - 2:
        candidates = []
        for pair in combinations(taxa, 2):
            joined = tuple(sorted(leaf for cluster in pair for leaf in _leaves(cluster)))
            rest = tuple(sorted(leaf for cluster in taxa for leaf in _leaves(cluster) if leaf not in joined))
            candidates.append((pair, (joined, rest)))
        fresh = []
        for _, split in candidates:
            if split not in known and split not in fresh:
                fresh.append(split)
        if fresh:
            known.update(zip(fresh, score_canonical(fresh)))
        if show_work:
            print(f"Scores: { {pair: (pair, split, known[split]) for pair, split in candidates} }")
        best_pair, best_split = min(candidates, key=lambda c: known[c[1]])  # first minimum, like min() in the reference
        if trace is not None:
            trace.append({"chosen": tuple(sorted(best_split)), "scores": {split: known[split] for _, split in candidates}})
        chosen.append(tuple(sorted(best_split)))
        merged = best_split[0]
        taxa = tuple([c for c in taxa if c not in merged and not set(c).issubset(merged)] + [merged])
    return chosen
