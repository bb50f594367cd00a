"""Host tests of the site-window entry points (batch.sliding_windows, window_scores, window_trees): the window list, every
rejected `windows` form (raised before any device work) and the refusal inside a torch.distributed group of several
processes."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch as batch
    return batch


def _codes(n, N=10):
    return np.zeros((n, N), np.uint8)


@pytest.mark.parametrize("n_sites,width,step,want", [
    (10, 4, None, [[0, 4], [4, 8]]),
    (10, 4, 4, [[0, 4], [4, 8]]),
    (10, 4, 3, [[0, 4], [3, 7], [6, 10]]),
    (10, 4, 1, [[k, k + 4] for k in range(7)]),
    (10, 3, 5, [[0, 3], [5, 8]]),
    (10, 4, 7, [[0, 4]]),
    (10, 10, None, [[0, 10]]),
    (10, 11, None, []),
    (0, 1, None, []),
])
def test_sliding_windows(batch, n_sites, width, step, want):
    got = batch.sliding_windows(n_sites, width, step)
    assert got.dtype == np.int64 and got.shape == (len(want), 2)
    assert got.tolist() == want


@pytest.mark.parametrize("args", [(-1, 4), (10, 0), (10, 4, 0), (10, 2.0), (10.0, 2), (10, 4, True), (10, "4")])
def test_sliding_windows_bad_arguments(batch, args):
    with pytest.raises(ValueError, match="sliding_windows"):
        batch.sliding_windows(*args)


BAD_WINDOWS = [
    [[0.0, 5.0]],                       # floats
    np.array([[0, 5]], dtype=np.float32),
    [[True, False]],                    # booleans
    [0, 5],                             # one dimension
    [[0, 5, 7]],                        # three columns
    [[[0, 5]]],                         # three dimensions
    [[-1, 5]],                          # begin < 0
    [[0, 11]],                          # end > n_sites
    [[5, 5]],                           # empty window
    [[6, 5]],                           # begin > end
    [[0, 5], [2]],                      # ragged
    [["0", "5"]],                       # strings
    np.array([[0, 2 ** 63 + 1]], dtype=np.uint64),
    [[0, None]],
]


@pytest.mark.parametrize("windows", BAD_WINDOWS, ids=[str(i) for i in range(len(BAD_WINDOWS))])
def test_window_scores_rejects_windows(batch, windows):
    from splitp_b200 import Method
    with pytest.raises(ValueError, match="window_scores"):
        batch.window_scores(_codes(4), [([0, 1], [2, 3])], windows, Method.subflattening)


@pytest.mark.parametrize("windows", BAD_WINDOWS, ids=[str(i) for i in range(len(BAD_WINDOWS))])
def test_window_trees_rejects_windows(batch, windows):
    with pytest.raises(ValueError, match="window_trees"):
        batch.window_trees(_codes(4), windows)


@pytest.mark.parametrize("n", [1, 65])
def test_taxa_bound(batch, n):
    from splitp_b200 import Method
    with pytest.raises(ValueError, match="2 to 64 taxa"):
        batch.window_scores(_codes(n), [], [[0, 5]], Method.subflattening)
    with pytest.raises(ValueError, match="2 to 64 taxa"):
        batch.window_trees(_codes(n), [[0, 5]])


def test_window_trees_bad_taxa(batch):
    with pytest.raises(ValueError, match="distinct names"):
        batch.window_trees(_codes(4), [[0, 5]], taxa=["a", "b", "c"])
    with pytest.raises(ValueError, match="distinct names"):
        batch.window_trees(_codes(4), [[0, 5]], taxa=["a", "b", "c", "a"])


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    from splitp_b200 import Method
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    results = []
    try:
        for call in (lambda: batch.window_scores(_codes(4), [([0, 1], [2, 3])], [[0, 5]], Method.subflattening),
                     lambda: batch.window_trees(_codes(4), [[0, 5]])):
            try:
                call()
                results.append("returned")
            except NotImplementedError as e:
                results.append("NotImplementedError" if "runs on one GPU" in str(e) else str(e))
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(",".join(results))


def test_refused_on_several_processes(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError,NotImplementedError"] * 2
