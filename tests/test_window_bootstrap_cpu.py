"""Host tests of batch.window_bootstrap_trees and engine.window_bootstrap_seed: a numpy model of the window seed with known
answers, every argument check (raised before any device work) and the refusal inside a torch.distributed group of
several processes."""
import numpy as np
import pytest

from tests import bootstrap_reference as BR


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch as batch
    return batch


def seed_model(seed, begin, end):
    """Three SplitMix64 steps absorbing seed, begin and end (numpy uint64 arithmetic wraps mod 2^64)."""
    g = np.uint64(BR.GAMMA)
    with np.errstate(over="ignore"):
        h = BR.fmix(np.uint64(seed) + g)
        h = BR.fmix(h + np.uint64(begin) + g)
        h = BR.fmix(h + np.uint64(end) + g)
    return int(h)


def test_seed_model_first_step_is_splitmix64():
    # SplitMix64 seeded with 0 first outputs 0xE220A8397B1DCDAF: the first step of the model is that generator
    with np.errstate(over="ignore"):
        assert int(BR.fmix(np.uint64(0) + np.uint64(BR.GAMMA))) == 0xE220A8397B1DCDAF


KNOWN = [  # (seed, begin, end) -> window seed, from the model
    ((0, 0, 0), 0x238275BC38FCBE91),
    ((0, 0, 10), 12509544039547440554),
    ((2 ** 64 - 1, 5, 2 ** 64 - 1), 14770701935879361966),
]


@pytest.mark.parametrize("args,want", KNOWN)
def test_window_seed_known_answers(args, want):
    import splitp_b200.engine as eng
    assert seed_model(*args) == want
    assert eng.window_bootstrap_seed(*args) == want


def test_window_seed_matches_model():
    import splitp_b200.engine as eng
    rng = np.random.default_rng(5)
    for _ in range(200):
        seed = int(rng.integers(0, 2 ** 63)) * 2 + int(rng.integers(0, 2))
        b = int(rng.integers(0, 10 ** 9))
        e = b + int(rng.integers(1, 10 ** 6))
        got = eng.window_bootstrap_seed(seed, b, e)
        assert got == seed_model(seed, b, e) and 0 <= got < 2 ** 64
    # the window's bounds, not its position, select the seed; swapping begin and end changes it
    assert eng.window_bootstrap_seed(3, 10, 20) == eng.window_bootstrap_seed(3, 10, 20)
    assert eng.window_bootstrap_seed(3, 10, 20) != eng.window_bootstrap_seed(3, 20, 10)
    assert eng.window_bootstrap_seed(3, 10, 20) != eng.window_bootstrap_seed(4, 10, 20)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 1.0, True, "1", None])
def test_window_seed_rejects_seed(seed):
    import splitp_b200.engine as eng
    with pytest.raises(ValueError):
        eng.window_bootstrap_seed(seed, 0, 1)


def _codes(n, N=10):
    return np.zeros((n, N), np.uint8)


BAD_WINDOWS = [[[0.0, 5.0]], [0, 5], [[-1, 5]], [[0, 11]], [[5, 5]], [[6, 5]], [[0, 5], [2]], [[0, None]]]


@pytest.mark.parametrize("windows", BAD_WINDOWS, ids=[str(i) for i in range(len(BAD_WINDOWS))])
def test_rejects_windows(batch, windows):
    with pytest.raises(ValueError, match="window_bootstrap_trees"):
        batch.window_bootstrap_trees(_codes(4), windows)


@pytest.mark.parametrize("replicates", [0, -3, 2.0, True, "5", 2 ** 24 + 1])
def test_rejects_replicates(batch, replicates):
    with pytest.raises(ValueError, match="window_bootstrap_trees: (replicates|at most)"):
        batch.window_bootstrap_trees(_codes(4), [[0, 5]], replicates=replicates)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 1.5, True, "0"])
def test_rejects_seed(batch, seed):
    with pytest.raises(ValueError, match="bootstrap seed"):
        batch.window_bootstrap_trees(_codes(4), [[0, 5]], seed=seed)


@pytest.mark.parametrize("n", [1, 65])
def test_taxa_bound(batch, n):
    with pytest.raises(ValueError, match="window_bootstrap_trees: 2 to 64 taxa"):
        batch.window_bootstrap_trees(_codes(n), [[0, 5]])


def test_bad_taxa(batch):
    for taxa in (["a", "b", "c"], ["a", "b", "c", "a"]):
        with pytest.raises(ValueError, match="window_bootstrap_trees: taxa must be 4 distinct names"):
            batch.window_bootstrap_trees(_codes(4), [[0, 5]], taxa=taxa)


@pytest.mark.parametrize("splits,match", [
    ([(("a", "b"), ("c", "x"))], "unknown leaf 'x'"),
    ([(("a", "b"), ("b", "c", "d"))], "exactly one side"),
    ([(("a", "b"), ("c",))], "exactly one side"),
    ([(("a", "a", "b"), ("c", "d"))], "exactly one side"),
])
def test_bad_splits(batch, splits, match):
    with pytest.raises(ValueError, match=f"window_bootstrap_trees: .*{match}"):
        batch.window_bootstrap_trees(_codes(4), [[0, 5]], taxa=["a", "b", "c", "d"], splits=splits)


def test_no_windows(batch):
    assert batch.window_bootstrap_trees(_codes(4), np.zeros((0, 2), np.int64)) == []
    assert batch.window_bootstrap_trees(_codes(4), []) == []


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        try:
            batch.window_bootstrap_trees(_codes(4), [[0, 5]])
            result = "returned"
        except NotImplementedError as e:
            result = "NotImplementedError" if "window_bootstrap_trees runs on one GPU" in str(e) else str(e)
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(result)


def test_refused_on_several_processes(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError"] * 2
