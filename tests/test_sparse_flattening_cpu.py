"""CPU tests of the sparse flattening route: route choice, batch chunking, the multi-GPU refusal above 16 taxa and the host
reference of tests/test_gpu_sparse_flattening.py."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sparse_reference  # noqa: E402


@pytest.fixture(scope="module")
def sp():
    import __graft_entry__
    __graft_entry__.build()
    import splitp_b200
    return splitp_b200


def test_route_choice_taxon_bound(sp):
    from splitp_b200 import batch
    assert not batch.uses_sparse_flattening(12)
    assert not batch.uses_sparse_flattening(16)
    assert batch.uses_sparse_flattening(17)
    assert batch.uses_sparse_flattening(64)


def test_route_choice_dense_size_classes(sp):
    """CountScorer keeps the dense route for Gram sides up to 4^6 rows (every class of 12 taxa) and scores 7|7 .. 8|8 from
    the pattern list."""
    from splitp_b200 import engine
    assert engine.CountScorer.SPARSE_MIN_ROWS == 4 ** 7
    assert not any(engine.CountScorer.sparse_class(a) for a in range(1, 7))
    assert engine.CountScorer.sparse_class(7) and engine.CountScorer.sparse_class(8)


def test_route_choice_cell_bound(sp):
    from splitp_b200 import phylogenetics
    assert phylogenetics.SPARSE_MIN_CELLS == 2 ** 27
    assert not phylogenetics.use_sparse_route(2 ** 13, 2 ** 14)
    assert phylogenetics.use_sparse_route(2 ** 13 + 1, 2 ** 14)
    assert phylogenetics.use_sparse_route(10 ** 5, 10 ** 5)


def test_chunking_by_workspace_bytes(sp):
    from splitp_b200 import engine
    sizes = [(k, 10 * k, 20 * k) for k in (200, 300, 400, 1000, 5000)]
    def ws(kmax, batch, ncols, nnz, max_cols):
        return kmax * batch * 100 + nnz
    chunks = engine.sparse_chunks(sizes, ws, cap=100_000)
    assert [i for c in chunks for i in c] == list(range(len(sizes)))  # consecutive, every split once
    for c in chunks:
        kmax = max(sizes[i][0] for i in c)
        assert len(c) == 1 or ws(kmax, len(c), 0, sum(sizes[i][2] for i in c), 0) <= 100_000
    assert chunks == [[0, 1], [2], [3], [4]]  # a matrix larger than the cap still gets a batch of its own
    assert engine.sparse_chunks(sizes, ws, cap=1 << 40, max_batch=2) == [[0, 1], [2, 3], [4]]
    assert engine.sparse_chunks([], ws, cap=1) == []


def test_multi_gpu_flattening_refused_above_16_taxa(sp):
    from splitp_b200 import batch
    from splitp_b200.enums import Method
    splits17 = [(list(range(3)), list(range(3, 17)))]
    with pytest.raises(NotImplementedError, match="16 taxa"):
        batch.SplitScorer(splits17, method=Method.flattening, rank=0, world=2)


def test_reference_against_dense_svd():
    rng = np.random.default_rng(7)
    for trial in range(12):
        R, C = rng.integers(5, 40), rng.integers(5, 60)
        dense = np.where(rng.random((R, C)) < rng.choice([0.03, 0.1, 0.5]), rng.integers(1, 50, size=(R, C)), 0).astype(np.float64)
        if trial % 3 == 0:  # block-diagonal: several components
            dense[: R // 2, C // 2:] = 0
            dense[R // 2:, : C // 2] = 0
        r, c = np.nonzero(dense)
        if min(len(np.unique(r)), len(np.unique(c))) <= 4:
            continue
        sv = np.linalg.svd(dense[np.unique(r)][:, np.unique(c)], compute_uv=False)
        want = np.sqrt(max(1 - np.sum(sv[:4] ** 2) / np.sum(sv ** 2), 0.0))
        got = sparse_reference.score(r, c, dense[r, c])
        assert abs(got - want) <= 1e-12 + 1e-10 * want, (trial, got, want)
