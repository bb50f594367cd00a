"""Numpy model of the quartet tables and of the three pairings of a quartet (batch.quartet_scores, csrc/quartets.cu), and the
true quartet topologies of the balanced tree of bench_inputs.  The tests compare the device tables with `tables` and feed the
16 x 16 matrices of `flattening` to the oracle."""
import numpy as np

PAIRINGS = ((1, 2, 3), (2, 1, 3), (3, 1, 2))  # pairing p: {a, partner} | {u, v} as quartet slots (partner, u, v)


def tables(codes, quartets):
    """int64 [Q, 256]: counts of the states (x_a, x_b, x_c, x_d) at cell 64 x_a + 16 x_b + 4 x_c + x_d over the sites where
    EVERY row of `codes` (uint8 [n, N], anything above 3 unusable) holds A/C/G/T."""
    codes = np.asarray(codes)
    ok = (codes <= 3).all(axis=0)
    c = codes[:, ok].astype(np.int64)
    out = np.zeros((len(quartets), 256), np.int64)
    for i, (a, b, x, y) in enumerate(np.asarray(quartets, dtype=np.int64).reshape(-1, 4)):
        out[i] = np.bincount(64 * c[a] + 16 * c[b] + 4 * c[x] + c[y], minlength=256)
    return out


def flattening(table, p):
    """16 x 16 flattening of pairing p (0 {a,b}|{c,d}, 1 {a,c}|{b,d}, 2 {a,d}|{b,c}) of one table: row 4 x_a + x_partner,
    column 4 x_u + x_v."""
    t = np.asarray(table).reshape(4, 4, 4, 4)  # [x_a][x_b][x_c][x_d]
    partner, u, v = PAIRINGS[p]
    return np.transpose(t, (0, partner, u, v)).reshape(16, 16)


def reduced(F):
    """The reduced format: all-zero rows and columns dropped."""
    F = np.asarray(F)
    return F[F.any(axis=1)][:, F.any(axis=0)]


def leaf_distances(n):
    """Edge counts between the leaves of bench_inputs.balanced_parents(n), rows in sorted-taxa order (the rows of
    simulate_codes)."""
    import bench_inputs as BI
    parent, names = BI.balanced_parents(n)
    depth = np.zeros(len(parent), np.int64)
    for v in range(1, len(parent)):
        depth[v] = depth[parent[v]] + 1
    ancestors = []
    for v in range(len(parent)):
        chain, u = [], v
        while u >= 0:
            chain.append(u)
            u = parent[u]
        ancestors.append(set(chain))
    leaves = [node for _, node in sorted((name, node) for node, name in names.items())]
    D = np.zeros((n, n), np.int64)
    for i, a in enumerate(leaves):
        for j, b in enumerate(leaves):
            lca = max(ancestors[a] & ancestors[b], key=lambda u: depth[u])
            D[i, j] = depth[a] + depth[b] - 2 * depth[lca]
    return D


def true_pairing(D, quartets):
    """Column of the tree's bipartition for every quartet (a, b, c, d): the pairing with the smallest sum of path lengths
    (four-point condition)."""
    q = np.asarray(quartets, dtype=np.int64)
    a, b, c, d = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    sums = np.stack([D[a, b] + D[c, d], D[a, c] + D[b, d], D[a, d] + D[b, c]], axis=1)
    return np.argmin(sums, axis=1)
