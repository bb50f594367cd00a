"""Host model of the column ranks of csrc/flatten.cu (spb_col_ranks_batch): per split, occupancy bits of the 4^b long-side
columns and the exclusive prefix counts of the bit words; rank(c) = pre[c >> 5] + popc(bits[c >> 5] & ((1 << (c & 31)) - 1)).
The ranks must number the occupied columns 0 .. ncols - 1 in column order, which keeps every pattern of a split in its own
cell and leaves F F^T unchanged."""
import numpy as np
import pytest


def col_rank_words(b):
    return (4 ** b + 31) // 32


def col_ranks(cols, b):
    """numpy restatement of the rank pass: (bits, pre, ncols) of the long-side indices `cols` of one split."""
    words = col_rank_words(b)
    bits = np.zeros(words, dtype=np.uint32)
    np.bitwise_or.at(bits, cols >> 5, (np.uint32(1) << (cols & 31).astype(np.uint32)))
    pop = np.array([bin(int(w)).count("1") for w in bits], dtype=np.int64)
    pre = np.concatenate([[0], np.cumsum(pop)[:-1]]).astype(np.uint32)
    return bits, pre, int(pop.sum())


def rank_of(bits, pre, c):
    w = bits[c >> 5]
    mask = ((np.uint64(1) << (c & 31).astype(np.uint64)) - np.uint64(1)).astype(np.uint32)
    low = np.array([bin(int(x)).count("1") for x in (w & mask)], dtype=np.int64)
    return pre[c >> 5].astype(np.int64) + low


def side_index(keys, n, idx):
    r = np.zeros(keys.shape[0], dtype=np.int64)
    for i in idx:
        r = (r << 2) | ((keys >> np.uint64(2 * (n - 1 - i))) & np.uint64(3)).astype(np.int64)
    return r


@pytest.mark.parametrize("n,a,P,seed", [(6, 2, 1, 0), (6, 2, 40, 1), (8, 3, 500, 2), (8, 4, 4 ** 8, 3), (10, 4, 3000, 4),
                                        (12, 6, 5000, 5), (12, 2, 20000, 6)])
def test_col_ranks_number_the_occupied_columns(n, a, P, seed):
    rng = np.random.default_rng(seed)
    keys = rng.choice(4 ** n, size=P, replace=False).astype(np.uint64)
    perm = rng.permutation(n)
    ia, ib = sorted(perm[:a].tolist()), perm[a:].tolist()  # long side in any taxon order
    b = n - a
    cols = side_index(keys, n, ib)
    bits, pre, ncols = col_ranks(cols, b)
    occupied = np.unique(cols)
    assert ncols == occupied.shape[0] <= min(4 ** b, P)
    assert np.array_equal(rank_of(bits, pre, cols), np.searchsorted(occupied, cols))
    # F F^T over the ranked columns equals F F^T over the raw columns (sparse, exact integers)
    rows = side_index(keys, n, ia)
    counts = rng.integers(1, 3000, size=P)
    import scipy.sparse as ss
    F = ss.csr_matrix((counts, (rows, cols)), shape=(4 ** a, 4 ** b))
    Fc = ss.csr_matrix((counts, (rows, rank_of(bits, pre, cols))), shape=(4 ** a, max(ncols, 1)))
    assert ((F @ F.T) != (Fc @ Fc.T)).nnz == 0


@pytest.mark.parametrize("num,pitch,want", [(0, 4096, 128), (1, 4096, 128), (128, 4096, 128), (129, 4096, 256), (60203, 4096, 4096),
                                            (60203, 1048576, 65536), (60203, 16384, 16384), (70000, 262144, 131072)])
def test_col_pitch(num, pitch, want):
    """S0 pitch of a ranked batch: min(4^b-wide pitch, P rounded up to a power of two >= 128)."""
    import types
    engine = pytest.importorskip("splitp_b200.engine")
    fake = types.SimpleNamespace(table=types.SimpleNamespace(num=num))
    got = engine.CountScorer._col_pitch(fake, 1, pitch)
    assert got == want and got % 128 == 0 and got >= min(num, pitch)
