"""Count flattenings scattered with column ranks: S0 keeps only the occupied columns, and every batched Gram contracts over its
own occupied columns (spb_col_ranks_batch, spb_flatten_u8_batch_cols, spb_gram_u8_batch_cols, spb_gram_u8_batch_i32_cols,
spb_gram_hi_strip_batch_table_cols).

  * the per-matrix-K Gram entry points against the full-K ones and an exact product, for every kernel: dp4a, umma<128>,
    umma<256> with a K split and the CTA-pair kernel (fp64 and int32);
  * CountScorer batches of every class of 12 taxa (fp64 Gram and int32 Gram + strip) against the full-K single-split Gram
    and a sparse numpy F F^T;
  * edge tables: one occupied column, every column occupied, 128k and 128k + 1 occupied columns, high counts in sparse
    columns, more high counts than the int32 route takes;
  * score_many over all 2,035 splits of 12 taxa bit for bit against the same scorer building full-K Gram matrices.
All integer work is compared bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests.test_gpu_parity import _count_table  # noqa: E402


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
# per-matrix K: the Gram entry points on random matrices
# ---------------------------------------------------------------------------------------------
def _k4major(S):
    """Row-major u8 [R, pitch] -> the dp4a operand layout (word k/4 of row r at word index (k/4) * R + r)."""
    R, P = S.shape
    return np.ascontiguousarray(S.reshape(R, P // 4, 4).transpose(1, 0, 2)).reshape(-1)


def _tiled(M):
    """Row-major u8 [R, K] -> the 128 x 128-byte SWIZZLE_128B tiles of csrc/gram.cu (16-byte chunk q of row rr stored at q ^ (rr & 7))."""
    R, K = M.shape
    t = M.reshape(R // 128, 128, K // 128, 8, 16).transpose(0, 2, 1, 3, 4)  # [row tile, k tile, rr, chunk, 16]
    perm = np.arange(8)[None, :] ^ (np.arange(128)[:, None] & 7)
    return np.ascontiguousarray(np.take_along_axis(t, perm[None, None, :, :, None], axis=3)).reshape(-1)


def _random_batch(rows, pitch, ncols, seed):
    """u8 matrices [nb, rows, pitch] with random values in the first ncols[b] columns and zeros beyond."""
    rng = np.random.default_rng(seed)
    out = np.zeros((len(ncols), rows, pitch), dtype=np.uint8)
    for b, k in enumerate(ncols):
        out[b, :, :k] = rng.integers(0, 256, size=(rows, k), dtype=np.uint8)
        out[b, rng.random(rows) < 0.1, :] = 0  # some empty rows
    return out


def _exact_gram(S):
    A = S.astype(np.float64)  # integer products below 2^53: exact in fp64
    return A @ A.transpose(0, 2, 1)


def direct_checks(eng, layout, rows, pitch, ncols, seed, i32=False):
    """spb_gram_u8_batch{,_i32}_cols with per-matrix ncols == the full-K entry point == the exact product."""
    lib, call, _p, _st = eng.lib, eng.call, eng._p, eng._st
    S = _random_batch(rows, pitch, ncols, seed)
    nb = len(ncols)
    if layout == eng.SPB_S0_K4MAJOR:
        flat = np.concatenate([_k4major(S[b]) for b in range(nb)])
    else:
        flat = np.concatenate([_tiled(S[b]) for b in range(nb)])
    dev = torch.device("cuda")
    s0 = torch.from_numpy(flat).to(dev)
    nc = torch.tensor(ncols, dtype=torch.int32, device=dev)
    want = _exact_gram(S)
    if i32:
        got = {}
        for name in ("full", "cols"):
            G = torch.full((nb, rows, rows), -1, dtype=torch.int32, device=dev)
            if name == "full":
                call("spb_gram_u8_batch_i32", _p(s0), rows * pitch, nb, rows, pitch, _p(G), rows * rows, _st())
            else:
                call("spb_gram_u8_batch_i32_cols", _p(s0), rows * pitch, nb, rows, pitch, _p(nc), _p(G), rows * rows, _st())
            got[name] = G.cpu().numpy().astype(np.float64)
    else:
        n = int(lib.spb_gram_u8_ws(rows, pitch, layout, nb))
        ws = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        got = {}
        for name in ("full", "cols"):
            G = torch.full((nb, rows, rows), float("nan"), dtype=torch.float64, device=dev)
            if name == "full":
                call("spb_gram_u8_batch", _p(s0), rows * pitch, nb, rows, pitch, layout, _p(G), rows * rows, _p(ws), _st())
            else:
                call("spb_gram_u8_batch_cols", _p(s0), rows * pitch, nb, rows, pitch, layout, _p(nc), _p(G), rows * rows, _p(ws), _st())
            got[name] = G.cpu().numpy()
    assert np.array_equal(got["full"], want)
    assert np.array_equal(got["cols"], want)


# (layout name, rows_pad, pitch, ncols per matrix, int32 route); nb and shapes pick the kernel as noted
DIRECT_CASES = [
    ("k4", 16, 8192, [1, 4, 5, 1023, 1024, 1025, 8192, 0, 3000], False),        # dp4a
    ("tiled", 128, 16384, [1, 128, 129, 256, 4000, 16384, 0, 12001], False),     # umma<128>, K split (8 matrices)
    ("tiled", 256, 65536, [128, 129, 1, 65536, 33025, 40000], False),           # umma<256>, K split, > 256 tiles
    ("tiled", 1024, 4096, [256, 257, 1, 4096, 2000] * 2, False),                # CTA pair, fp64 (10 x 10 blocks)
    ("tiled", 1024, 16384, [8068, 8192, 8193, 1, 16384, 0] * 2, True),         # CTA pair, int32
    ("tiled", 4096, 4096, [3402, 3584, 3585], True),                            # CTA pair, int32, 6|6 of 12 taxa
]


@pytest.mark.parametrize("case", range(len(DIRECT_CASES)))
def test_gram_cols_matches_full_k(eng, case):
    name, rows, pitch, ncols, i32 = DIRECT_CASES[case]
    layout = eng.SPB_S0_K4MAJOR if name == "k4" else eng.SPB_S0_TILED
    direct_checks(eng, layout, rows, pitch, ncols, 100 + case, i32)


# ---------------------------------------------------------------------------------------------
# the scorer's batches against full-K Gram matrices
# ---------------------------------------------------------------------------------------------
class FullKScorer:
    """Mixin: CountScorer batches as they were built before column ranks (raw columns, K = pitch), for reference."""

    def _col_pitch(self, layout, pitch):
        return int(pitch)

    def _scatter_raw(self, arr, nb, s0, layout, rows_pad, pitch, clear=False):
        e = self._eng
        t = self.table
        if clear:
            e.call("spb_flatten_u8_clear_batch", e._p(t.keys), t.num, arr, nb, e._p(s0), rows_pad * pitch, rows_pad, pitch, layout, e._st())
        else:
            e.call("spb_flatten_u8_batch", e._p(t.keys), e._p(t.counts), t.num, arr, nb, e._p(s0), rows_pad * pitch, rows_pad, pitch,
                   layout, e.SPB_U8_NO_MEMSET, e._p(self.hi_rc), e._p(self.hi_val), e._p(self.hi_num), self.hi_cap, e._st())

    def _gram_batch(self, splits, s0, G, ws, layout, rows_pad, pitch):
        e = self._eng
        nb = len(splits)
        arr = splits if isinstance(splits, C.Array) else (e._lib.SpbSplit * nb)(*splits)
        self._scatter_raw(arr, nb, s0, layout, rows_pad, pitch)
        e.call("spb_gram_u8_batch", e._p(s0), rows_pad * pitch, nb, rows_pad, pitch, layout, e._p(G), rows_pad * rows_pad, e._p(ws), e._st())
        e.call("spb_gram_hi_correction_batch", e._p(s0), rows_pad * pitch, nb, rows_pad, pitch, layout, e._p(self.hi_rc),
               e._p(self.hi_val), e._p(self.hi_num), self.hi_cap, e._p(G), rows_pad * rows_pad, e._st())
        self._scatter_raw(arr, nb, s0, layout, rows_pad, pitch, clear=True)

    def _gram_batch_i32(self, splits, s0, buf, b0, layout, rows_pad, pitch):
        e = self._eng
        nb = len(splits)
        arr = splits if isinstance(splits, C.Array) else (e._lib.SpbSplit * nb)(*splits)
        cs_rows = int(buf["Cs"].shape[1])
        G, Cs, pos, hr, hm = (buf[k][b0:] for k in ("G", "Cs", "pos", "hr", "hm"))
        self._scatter_raw(arr, nb, s0, layout, rows_pad, pitch)
        e.call("spb_gram_u8_batch_i32", e._p(s0), rows_pad * pitch, nb, rows_pad, pitch, e._p(G), rows_pad * rows_pad, e._st())
        e.call("spb_gram_hi_strip_batch", e._p(s0), rows_pad * pitch, nb, rows_pad, pitch, layout, e._p(self.hi_rc), e._p(self.hi_val),
               e._p(self.hi_num), self.hi_cap, e._p(Cs), cs_rows, e._p(pos), e._p(hr), e._p(hm), e._st())
        self._scatter_raw(arr, nb, s0, layout, rows_pad, pitch, clear=True)


def _full_k_scorer(eng, tab):
    cls = type("FullK", (FullKScorer, eng.CountScorer), {"_eng": eng})
    return cls(tab)


def _numpy_gram(tab, ia, ib):
    """Exact F F^T (rows over the short side ia) from the pattern list, scipy sparse int64."""
    import scipy.sparse as ss
    keys = tab.keys.cpu().numpy().view(np.uint64)
    cnt = tab.counts.cpu().numpy().view(np.uint32).astype(np.int64)
    n = tab.n

    def side(idx):
        r = np.zeros(keys.shape[0], dtype=np.int64)
        for i in idx:
            r = (r << 2) | ((keys >> np.uint64(2 * (n - 1 - i))) & np.uint64(3)).astype(np.int64)
        return r

    F = ss.csr_matrix((cnt, (side(ia), side(ib))), shape=(4 ** len(ia), 4 ** len(ib)))
    return (F @ F.T).toarray()


def _batch_grams(scorer, idx):
    """Gram matrices [nb, R, R] (fp64) of splits of one class through the scorer's batched route (int32 Gram + strip expanded)."""
    a = min(len(idx[0][0]), len(idx[0][1]))
    n = scorer.table.n
    R, Cc = 4 ** a, 4 ** (n - a)
    layout, rows_pad, pitch = scorer.geometry(R, Cc)
    plans = [scorer._plan(ia, ib, False)[0] for ia, ib in idx]
    nb = len(plans)
    s0_pitch = scorer._col_pitch(layout, pitch)
    if scorer._use_i32(layout, rows_pad, pitch):
        s0 = scorer._buffers(layout, rows_pad, s0_pitch, 1)[0]
        buf = scorer._buffers_i32(rows_pad, nb)
        scorer._gram_batch_i32(plans, s0, buf, 0, layout, rows_pad, pitch)
        out = []
        for b in range(nb):
            m = int(buf["hm"][b].item())
            hr = buf["hr"][b, :m].to(torch.int64)
            Cf = torch.zeros((rows_pad, rows_pad), dtype=torch.float64, device=hr.device)
            Cf[:, hr] = buf["Cs"][b, :m].T
            Cf[hr, :] = buf["Cs"][b, :m]
            out.append((buf["G"][b].to(torch.float64) + Cf)[:R, :R])
        return torch.stack(out).cpu().numpy(), True
    s0, G, ws = scorer._buffers(layout, rows_pad, s0_pitch, nb)
    scorer._gram_batch(plans, s0, G[:nb], ws, layout, rows_pad, pitch)
    return G[:nb, :R, :R].cpu().numpy(), False


@pytest.fixture(scope="module")
def c2_small(sp, eng):
    """The c2 tree (12 taxa, JC, bl 0.05) at 10^5 sites: counts >= 256 on the near-constant patterns."""
    return _count_table(sp, eng, 12, 100_000, 2)


@pytest.mark.parametrize("a", [2, 3, 4, 5, 6])
def test_scorer_batches_every_class(sp, eng, c2_small, a):
    tree, _, tab = c2_small
    splits = [s for s in sp.all_splits(tree) if len(s[0]) == a][::11][:6]
    idx = [eng.split_positions(s, tree.taxa) for s in splits]
    scorer = eng.CountScorer(tab)
    assert scorer.n_hi > 0
    got, i32 = _batch_grams(scorer, idx)
    assert i32 == (a >= 5)
    for b, (ia, ib) in enumerate(idx):
        G, k = scorer.gram(ia, ib)  # single split: raw columns, full K
        assert np.array_equal(got[b], G[:k, :k].cpu().numpy()), b
    assert np.array_equal(got[0], _numpy_gram(tab, *idx[0]))


def _table(eng, n, keys, counts):
    keys = np.asarray(keys, dtype=np.uint64)
    assert np.unique(keys).shape[0] == keys.shape[0]
    dev = torch.device("cuda")
    return eng.PatternTable(n, torch.from_numpy(keys.view(np.int64)).to(dev),
                            torch.from_numpy(np.asarray(counts, dtype=np.uint32).view(np.int32)).to(dev))


def _keys(n, ia, ib, rows, cols):
    """Keys of the patterns with short-side index rows[i] and long-side index cols[i] of the split (ia | ib)."""
    keys = np.zeros(len(rows), dtype=np.uint64)
    for side, vals in ((ia, np.asarray(rows, dtype=np.uint64)), (ib, np.asarray(cols, dtype=np.uint64))):
        for d, t in enumerate(side):
            digit = (vals >> np.uint64(2 * (len(side) - 1 - d))) & np.uint64(3)
            keys |= digit << np.uint64(2 * (n - 1 - t))
    return keys


def _edge_table(eng, n, a, ncols, rng, hi_cols=0, n_hi=0, rows=None):
    """Table of one split (first a taxa | rest) occupying exactly `ncols` random columns, every column with at least one
    pattern; `hi_cols` of them hold a single pattern with a count >= 256; n_hi extra patterns with counts >= 256."""
    ia, ib = list(range(a)), list(range(a, n))
    R, Cc = 4 ** a, 4 ** (n - a)
    cols = rng.choice(Cc, size=ncols, replace=False)
    cells = set()
    for j, c in enumerate(cols):
        per = 1 if j < hi_cols else int(rng.integers(1, 4))
        for r in rng.choice(R if rows is None else rows, size=per, replace=False):
            cells.add((int(r), int(c)))
    cells = sorted(cells)
    counts = rng.integers(1, 256, size=len(cells))
    colset = {int(c): j for j, c in enumerate(cols)}
    for i, (r, c) in enumerate(cells):
        if colset[c] < hi_cols:
            counts[i] = int(rng.integers(256, 5000))
    # extra high counts on cells of already occupied columns
    extra, taken = [], set(cells)
    while len(extra) < n_hi:
        cell = (int(rng.integers(0, R)), int(cols[rng.integers(0, ncols)]))
        if cell not in taken:
            taken.add(cell)
            extra.append(cell)
    allc = cells + extra
    counts = np.concatenate([counts, rng.integers(256, 70000, size=len(extra))]).astype(np.uint32)
    keys = _keys(n, ia, ib, [r for r, _ in allc], [c for _, c in allc])
    return _table(eng, n, keys, counts), (ia, ib)


EDGE_CASES = [  # (n, a, occupied columns, columns holding one high count, extra high counts)
    (8, 2, 1, 0, 0), (8, 3, 1, 1, 0), (8, 4, 1, 0, 3),           # one occupied column (dp4a, umma<128>, umma<256>)
    (8, 2, 4096, 5, 0), (8, 3, 1024, 7, 0), (8, 4, 256, 3, 0),   # every column occupied
    (8, 3, 128, 0, 0), (8, 3, 129, 2, 0), (8, 4, 256, 0, 0),
    (12, 6, 256, 40, 0), (12, 6, 257, 40, 0), (12, 5, 1280, 300, 0), (12, 5, 1281, 0, 20),  # 128k, 128k + 1 (int32 route)
    (12, 4, 384, 50, 0), (12, 3, 385, 0, 0), (12, 2, 129, 60, 0),
    (12, 6, 3000, 0, 5000),                                       # more high counts than the int32 route takes: fp64 Gram
]


@pytest.mark.parametrize("case", range(len(EDGE_CASES)))
def test_edge_tables(eng, case):
    n, a, ncols, hi_cols, n_hi = EDGE_CASES[case]
    rng = np.random.default_rng(500 + case)
    tab, (ia, ib) = _edge_table(eng, n, a, ncols, rng, hi_cols, n_hi)
    scorer = eng.CountScorer(tab)
    if n_hi > scorer.I32_MAX_HI:
        assert not scorer._use_i32(*scorer.geometry(4 ** a, 4 ** (n - a)))
    want = _numpy_gram(tab, ia, ib)
    got, _ = _batch_grams(scorer, [(ia, ib)] * 3)  # the same split three times in one batch
    for b in range(3):
        assert np.array_equal(got[b], want), b
    G, k = scorer.gram(ia, ib)
    assert np.array_equal(G[:k, :k].cpu().numpy(), want)


def test_score_many_all_splits_equals_full_k(sp, eng, c2_small):
    """All 2,035 splits of 12 taxa at 10^5 sites: the scores of score_many are bit for bit those of the same scorer building
    every Gram over all 4^b columns."""
    tree, _, tab = c2_small
    idx = [eng.split_positions(s, tree.taxa) for s in sp.all_splits(tree)]
    assert len(idx) == 2035
    got = eng.CountScorer(tab).score_many(idx).cpu().numpy()
    ref = _full_k_scorer(eng, tab).score_many(idx).cpu().numpy()
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
