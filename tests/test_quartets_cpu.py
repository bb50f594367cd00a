"""Host tests of batch.quartet_scores: every argument check raises before any device work, the default quartet list, the
column map of written quartets, the numpy model of the cell index and the pairings (tests/quartet_reference.py) against the
oracle's sub-alignment and flattening, and the refusal inside a torch.distributed group of several processes."""
import itertools
from math import comb

import numpy as np
import pytest

from tests import quartet_reference as QR


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch as batch
    return batch


@pytest.fixture
def no_device(batch, monkeypatch):
    """Any step towards the device fails the test."""
    def refuse(*args, **kwargs):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(batch, "_as_alignment", refuse)
    monkeypatch.setattr(batch.engine, "device", refuse)
    return batch


def _codes(n, N=10):
    return np.zeros((n, N), np.uint8)


BAD_QUARTETS = [
    ([(0, 1, 1, 2)], "four distinct taxa"),
    ([(0, 1, 2, 6)], "out of range"),
    ([(0, 1, 2, -1)], "out of range"),
    (np.array([[0, 1, 2, 6]]), r"\[0, 6\)"),
    (np.array([[3, 1, 2, 3]]), "four distinct taxa"),
    (np.zeros((2, 3), np.int64), r"\[Q, 4\]"),
    ([(0, 1, 2)], "not a 4-tuple"),
    ([(0, 1, 2, 3, 4)], "not a 4-tuple"),
    ([(0, 1, 2, True)], "boolean"),
    ([(0, 1, 2, 2.0)], "unknown taxon"),
    ([(0, 1, 2, "e")], "unknown taxon"),
    (["abcd"], "not a 4-tuple"),
    ([5], "not a 4-tuple"),
    (5, "sequence of 4-tuples"),
    ("abcd", "sequence of 4-tuples"),
]


@pytest.mark.parametrize("quartets,match", BAD_QUARTETS, ids=[str(i) for i in range(len(BAD_QUARTETS))])
def test_rejects_quartets(no_device, quartets, match):
    with pytest.raises(ValueError, match="quartet_scores: .*" + match):
        no_device.quartet_scores(_codes(6), quartets)


def test_labels(no_device):
    taxa = ["a", "b", "c", "d", "e"]
    with pytest.raises(ValueError, match="unknown taxon 'x'"):
        no_device.quartet_scores({t: "ACGT" for t in taxa}, [("a", "b", "c", "x")])
    with pytest.raises(ValueError, match="labels need `taxa`"):
        no_device.quartet_scores(_codes(5), [("a", "b", "c", "d")])
    with pytest.raises(ValueError, match="four distinct taxa"):
        no_device.quartet_scores(_codes(5), [("a", "b", "c", "a")], taxa=taxa)


@pytest.mark.parametrize("n", [3, 65])
def test_taxa_bound(no_device, n):
    with pytest.raises(ValueError, match="quartet_scores: 4 to 64 taxa"):
        no_device.quartet_scores(_codes(n), [(0, 1, 2, 3)])


def test_rejects_method(no_device):
    from splitp_b200.enums import Method
    with pytest.raises(NotImplementedError, match="quartet_scores: Method.flattening"):
        no_device.quartet_scores(_codes(4), None, Method.distance)


@pytest.mark.parametrize("quartets", [[], np.zeros((0, 4), np.int64)])
def test_no_quartets(no_device, quartets):
    out = no_device.quartet_scores(_codes(6), quartets)
    assert out.shape == (0, 3) and out.dtype == np.float64


@pytest.mark.parametrize("n", [4, 5, 12, 33, 64])
def test_default_quartet_list(batch, n):
    q = batch.engine.all_quartets(n)
    assert q.shape == (comb(n, 4), 4)
    np.testing.assert_array_equal(q, np.array(list(itertools.combinations(range(n), 4))))


def test_column_map(batch):
    rng = np.random.default_rng(4)
    written = np.array([rng.choice(64, 4, replace=False) for _ in range(500)] + list(itertools.permutations(range(4))))
    srt, cmap = batch.engine.quartet_column_map(written)
    np.testing.assert_array_equal(srt, np.sort(written, axis=1))
    for q, s, cols in zip(written.tolist(), srt.tolist(), cmap.tolist()):
        for j, k in enumerate(cols):
            want = {frozenset((q[0], q[j + 1])), frozenset(set(q) - {q[0], q[j + 1]})}
            assert {frozenset((s[0], s[k + 1])), frozenset(set(s) - {s[0], s[k + 1]})} == want


def test_cell_index_and_pairings_model(oracle):
    """QR.tables + QR.flattening equal the oracle's flattening of the sub-alignment of the whole alignment's pattern counts
    (sites with an unusable character in ANY taxon dropped), for the three pairings of sorted quartets."""
    rng = np.random.default_rng(9)
    n = 7
    codes = rng.integers(0, 4, size=(n, 3000), dtype=np.uint8)
    codes[6, rng.random(3000) < 0.1] = 255  # gaps outside the quartets below
    keys, counts, _ = oracle.get_pattern_counts_arrays(codes)
    for q in [(0, 1, 2, 3), (1, 3, 4, 5), (0, 2, 4, 5)]:
        sub_keys, sub_vals = oracle.sub_alignment(keys, counts, n, list(q))
        table = QR.tables(codes, [q])[0]
        assert table.sum() == counts.sum()
        for p, (ia, ib) in enumerate([([0, 1], [2, 3]), ([0, 2], [1, 3]), ([0, 3], [1, 2])]):
            want = oracle.flattening_dense(sub_keys, sub_vals, 4, ia, ib)
            np.testing.assert_array_equal(QR.flattening(table, p), want)


def test_true_pairing_model():
    D = QR.leaf_distances(8)  # ((0,1),(2,3)),((4,5),(6,7)) in sorted-taxa rows
    got = QR.true_pairing(D, np.array([(0, 1, 2, 3), (0, 2, 1, 3), (0, 4, 1, 5), (4, 6, 5, 7)]))
    np.testing.assert_array_equal(got, [0, 1, 1, 1])


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        try:
            batch.quartet_scores(_codes(4), [(0, 1, 2, 3)])
            result = "returned"
        except NotImplementedError as e:
            result = "NotImplementedError" if "quartet_scores runs on one GPU" in str(e) else str(e)
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(result)


def test_refused_on_several_processes(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError"] * 2
