"""Host tests of batch.window_bootstrap_scores: every argument check (raised before any device work), the empty window
list and the refusal inside a torch.distributed group of several processes."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch as batch
    return batch


def _codes(n, N=10):
    return np.zeros((n, N), np.uint8)


SPLITS = [([0, 1], [2, 3])]
BAD_WINDOWS = [[[0.0, 5.0]], [0, 5], [[-1, 5]], [[0, 11]], [[5, 5]], [[6, 5]], [[0, 5], [2]], [[0, None]]]


@pytest.mark.parametrize("windows", BAD_WINDOWS, ids=[str(i) for i in range(len(BAD_WINDOWS))])
def test_rejects_windows(batch, windows):
    with pytest.raises(ValueError, match="window_bootstrap_scores"):
        batch.window_bootstrap_scores(_codes(4), SPLITS, windows)


@pytest.mark.parametrize("replicates", [0, -3, 2.0, True, "5", 2 ** 24 + 1])
def test_rejects_replicates(batch, replicates):
    with pytest.raises(ValueError, match="window_bootstrap_scores: (replicates|at most)"):
        batch.window_bootstrap_scores(_codes(4), SPLITS, [[0, 5]], replicates=replicates)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 1.5, True, "0"])
def test_rejects_seed(batch, seed):
    with pytest.raises(ValueError, match="bootstrap seed"):
        batch.window_bootstrap_scores(_codes(4), SPLITS, [[0, 5]], seed=seed)


@pytest.mark.parametrize("n", [1, 65])
def test_taxa_bound(batch, n):
    with pytest.raises(ValueError, match="window_bootstrap_scores: 2 to 64 taxa"):
        batch.window_bootstrap_scores(_codes(n), SPLITS, [[0, 5]])


def test_rejects_method(batch):
    from splitp_b200.enums import Method
    with pytest.raises(NotImplementedError, match="score_splits"):
        batch.window_bootstrap_scores(_codes(4), SPLITS, [[0, 5]], method=Method.distance)


def test_unknown_leaf(batch):
    with pytest.raises(KeyError):  # SplitScorer's lookup, as in score_splits
        batch.window_bootstrap_scores(_codes(4), [(("a", "b"), ("c", "x"))], [[0, 5]], taxa=["a", "b", "c", "d"])


@pytest.mark.parametrize("windows", [np.zeros((0, 2), np.int64), []])
def test_no_windows(batch, windows):
    out = batch.window_bootstrap_scores(_codes(4), SPLITS * 3, windows, replicates=7)
    assert out.shape == (0, 7, 3) and out.dtype == np.float64


def test_packed_input_above_31_taxa_refused(batch):
    from splitp_b200.enums import Method
    planes, valid = batch.pack_planes_host(np.zeros((40, 100), np.uint8))
    with pytest.raises(NotImplementedError, match="window_bootstrap_scores of 40 taxa needs the alignment as characters"):
        batch.window_bootstrap_scores(batch.HostPlanes(planes, valid, 40, 100), [([0], list(range(1, 40)))], [[0, 50]],
                                      Method.mutual_information, replicates=2)


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        try:
            batch.window_bootstrap_scores(_codes(4), SPLITS, [[0, 5]])
            result = "returned"
        except NotImplementedError as e:
            result = "NotImplementedError" if "window_bootstrap_scores runs on one GPU" in str(e) else str(e)
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(result)


def test_refused_on_several_processes(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError"] * 2
