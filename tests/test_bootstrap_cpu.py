"""Host tests of the bootstrap resampling rule (tests/bootstrap_reference.py, the model csrc/bootstrap.cu is checked against on
the GPU) and of the argument checks of batch.bootstrap_scores, which run before anything touches a device."""
import numpy as np
import pytest
from scipy.stats import chi2

from tests import bootstrap_reference as BR


def test_splitmix64_outputs_from_state_zero():
    got = BR.uniforms(0, 0, np.arange(3))
    assert [int(x) for x in got] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]


def test_known_replicate():
    counts = [5, 1, 994]
    assert BR.sites(7, 3, 1000)[:5].tolist() == [97, 539, 804, 316, 17]
    assert BR.replicate(counts, 7, 3).tolist() == [4, 1, 995]


def test_vectorised_model_equals_scalar_model():
    rng = np.random.default_rng(11)
    counts = rng.integers(0, 50, size=40)
    counts[[0, 7, 39]] = 0  # empty patterns are never drawn
    for seed in (0, 1, 2 ** 64 - 1, 0x123456789ABCDEF0):
        for b in (0, 1, 5, 2 ** 24 - 1):
            d = BR.draws(counts, seed, b)
            for s in (0, 1, 2, 100, len(d) - 1):
                assert d[s] == BR.draw_scalar(counts, seed, b, s), (seed, b, s)


def test_mulhi_matches_python_integers():
    rng = np.random.default_rng(3)
    a = rng.integers(0, 2 ** 63, size=1000, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    b = np.concatenate([rng.integers(1, 2 ** 32, size=500, dtype=np.uint64), rng.integers(0, 2 ** 63, size=500, dtype=np.uint64)])
    assert [int(x) for x in BR.mulhi(a, b)] == [(int(x) * int(y)) >> 64 for x, y in zip(a, b)]
    top = np.uint64(2 ** 64 - 1)
    assert int(BR.mulhi(top, top)) == ((2 ** 64 - 1) ** 2) >> 64


def test_every_replicate_sums_to_n():
    counts = np.array([3, 0, 17, 1, 250, 9])
    reps = BR.replicates(counts, 42, 0, 20)
    assert (reps.sum(axis=1) == counts.sum()).all()
    assert (reps[:, 1] == 0).all()


def test_replicate_does_not_depend_on_its_chunk():
    counts = np.array([10, 20, 30, 40])
    alone = BR.replicate(counts, 9, 6)
    assert np.array_equal(BR.replicates(counts, 9, 4, 5)[2], alone)
    assert np.array_equal(BR.replicates(counts, 9, 0, 8)[6], alone)


def test_pooled_chi_square():
    """4,000 replicates of N = 200 draws: the pooled counts are one multinomial draw of 800,000 from count / N."""
    counts = np.array([1, 2, 5, 12, 30, 50, 100])
    reps = BR.replicates(counts, 2024, 0, 4000)
    obs = reps.sum(axis=0)
    exp = 4000 * counts.astype(np.float64)
    stat = float(((obs - exp) ** 2 / exp).sum())
    assert chi2.sf(stat, len(counts) - 1) > 1e-3, stat


def test_atomics_after_aggregation():
    assert BR.atomics_after_aggregation(np.zeros(64, dtype=np.int64)) == 2
    assert BR.atomics_after_aggregation(np.arange(33)) == 33
    assert BR.atomics_after_aggregation([5, 5, 6]) == 2


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch
    return splitp_b200.batch


@pytest.mark.parametrize("replicates", [0, -1, 1.5, True])
def test_bad_replicates(batch, replicates):
    with pytest.raises(ValueError):
        batch.bootstrap_scores(np.zeros((4, 10), np.uint8), [([0, 1], [2, 3])], replicates=replicates)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 0.5, "1"])
def test_bad_seed(batch, seed):
    with pytest.raises(ValueError):
        batch.bootstrap_scores(np.zeros((4, 10), np.uint8), [([0, 1], [2, 3])], seed=seed)


def test_seed_range_ends_accepted(batch):
    from splitp_b200 import engine
    assert engine.bootstrap_seed(0) == 0
    assert engine.bootstrap_seed(np.uint64(2 ** 64 - 1)) == 2 ** 64 - 1


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        batch.bootstrap_scores(np.zeros((4, 10), np.uint8), [([0, 1], [2, 3])], replicates=2)
        result = "returned"
    except NotImplementedError:
        result = "NotImplementedError"
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(result)


def test_refused_on_several_processes(batch, tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError"] * 2
