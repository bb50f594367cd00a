"""Host reference for flattening scores of sparse matrices (tests/test_gpu_sparse_flattening.py,
tests/test_sparse_flattening_cpu.py).

score^2 = 1 - (sum of the 4 largest eigenvalues of F F^T) / sum v^2.  F is cut into the connected components of its
row / column graph: F F^T is block-diagonal over them, so the spectrum is the union of the components' spectra.  A
component with one row or one column has the single eigenvalue sum v^2; the others go through numpy.linalg.eigvalsh of
their Gram on the smaller side.
"""
import numpy as np
import scipy.sparse
from scipy.sparse.csgraph import connected_components


def spectrum(rows, cols, vals):
    """Non-zero part of the spectrum of F F^T (unsorted) for the non-zeros (rows, cols, vals) of F (no repeated cell)."""
    rows, cols, vals = (np.asarray(x) for x in (rows, cols, vals))
    if len(vals) == 0:
        return np.zeros(0)
    _, r = np.unique(rows, return_inverse=True)
    _, c = np.unique(cols, return_inverse=True)
    R, C = int(r.max()) + 1, int(c.max()) + 1
    F = scipy.sparse.csr_matrix((vals.astype(np.float64), (r, c)), shape=(R, C))
    graph = scipy.sparse.bmat([[None, F], [F.T, None]]).tocsr()
    graph.data[:] = 1.0
    ncomp, label = connected_components(graph, directed=False)
    lr, lc = label[:R], label[R:]
    nr = np.bincount(lr, minlength=ncomp)
    nc = np.bincount(lc, minlength=ncomp)
    comp_of_entry = lr[r]
    mass = np.bincount(comp_of_entry, weights=vals.astype(np.float64) ** 2, minlength=ncomp)
    rank1 = (nr <= 1) | (nc <= 1)
    eig = [mass[rank1]]
    for comp in np.flatnonzero(~rank1):
        sub = F[np.flatnonzero(lr == comp)][:, np.flatnonzero(lc == comp)]
        G = (sub @ sub.T) if sub.shape[0] <= sub.shape[1] else (sub.T @ sub)
        eig.append(np.linalg.eigvalsh(G.toarray()))
    return np.concatenate(eig)


def score(rows, cols, vals):
    """Flattening score of the sparse matrix; 0.0 when one side has at most 4 used indices."""
    if min(len(np.unique(rows)), len(np.unique(cols))) <= 4:
        return 0.0
    lam = np.sort(spectrum(rows, cols, vals))[::-1]
    total = float(np.sum(np.asarray(vals, dtype=np.float64) ** 2))
    return float(np.sqrt(max(1.0 - lam[:4].sum() / total, 0.0)))


def flattening_entries(mapping, idx_a, idx_b):
    """(rows, cols, vals) of the flattening of (idx_a | idx_b) of a {pattern: value} mapping: one entry per pattern, rows and
    columns as the side strings (any grouping of equal projections gives the same score)."""
    pats = list(mapping)
    rows = np.array(["".join(p[t] for t in idx_a) for p in pats])
    cols = np.array(["".join(p[t] for t in idx_b) for p in pats])
    return rows, cols, np.array([float(mapping[p]) for p in pats])
