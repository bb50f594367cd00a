"""Host tests of bootstrap_trees: the agglomeration restatement of tests/erickson_reference.py (the model the lockstep
kernels are checked against on the GPU) reproduces the reference's subflattening picks on the golden alignments when fed the
oracle's scores, and the argument checks of batch.bootstrap_trees raise before anything touches a device."""
import json
import os

import numpy as np
import pytest

from tests import erickson_reference as ER

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


@pytest.mark.parametrize("case", [0, 1])
def test_restatement_reproduces_golden_subflattening_picks(oracle, case):
    g, tr = _load("golden_erickson.json")[case], _load("golden_erickson_trace.json")[case]
    n = g["n"]
    keys, _ = oracle.patterns_to_keys(g["patterns"])
    vals = np.asarray(g["values"], dtype=np.float64)
    tables, total = oracle.pair_tables(keys, vals, n), vals.sum()
    taxa = [str(np.base_repr(i, base=max(i + 1, 2))) for i in range(n)]
    index = {t: i for i, t in enumerate(taxa)}

    def score_many(splits):
        return [oracle.split_score(oracle.subflattening_from_tables(tables, total, [index[t] for t in a], [index[t] for t in b]))
                for a, b in splits]

    chosen, trace = ER.agglomerate(taxa, score_many)
    steps = tr["subflattening"]
    assert len(chosen) == len(steps) == n - 2
    compared = 0
    for got, step, scores in zip(chosen, steps, trace):
        want = tuple(tuple(side) for side in step["chosen"])
        if step["second"] - step["best"] > 1e-6 * abs(step["second"]):
            assert got == want
            assert abs(min(scores.values()) - step["best"]) <= 1e-9 * max(abs(step["best"]), 1e-300) + 1e-15
            compared += 1
        elif got != want:
            break  # a near-tie decided differently: later steps start from different clusters
    assert compared >= 2
    if compared == n - 2:
        assert chosen == [tuple(tuple(side) for side in s) for s in g["subflattening"]]


def test_restatement_first_minimum_and_orientation():
    taxa = ["b", "a", "c", "d"]  # the smallest name is in row 1
    seen = []

    def score_many(splits):
        seen.extend(splits)
        return [0.0] * len(splits)  # all tied: the first candidate in combinations order wins

    chosen, _ = ER.agglomerate(taxa, score_many)
    assert all(a[0] == "a" for a, _ in seen)  # canonical orientation: the side with the smallest name first
    assert chosen[0] == (("a", "b"), ("c", "d"))  # pair (b, a) comes first
    # the clusters are now (c, d, (a, b)): the first pair (c, d) gives the step-0 bipartition again
    assert chosen[1] == (("a", "b"), ("c", "d"))


def _codes(n, N=10):
    return np.zeros((n, N), np.uint8)


@pytest.fixture(scope="module")
def batch():
    import splitp_b200.batch as batch
    return batch


@pytest.mark.parametrize("method", ["flattening", "mutual_information"])
def test_other_methods_refused(batch, method):
    from splitp_b200 import Method
    with pytest.raises(NotImplementedError, match="one pattern table per launch"):
        batch.bootstrap_trees(_codes(6), replicates=2, method=getattr(Method, method))


@pytest.mark.parametrize("replicates", [0, -1, 1.5, True, 2 ** 24 + 1])
def test_bad_replicates(batch, replicates):
    with pytest.raises(ValueError, match="bootstrap_trees"):
        batch.bootstrap_trees(_codes(6), replicates=replicates)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 0.5, "1"])
def test_bad_seed(batch, seed):
    with pytest.raises(ValueError):
        batch.bootstrap_trees(_codes(6), seed=seed)


@pytest.mark.parametrize("n", [1, 65])
def test_taxa_bound(batch, n):
    with pytest.raises(ValueError, match="2 to 64 taxa"):
        batch.bootstrap_trees(_codes(n), replicates=2)


def test_bad_taxa_and_splits(batch):
    with pytest.raises(ValueError, match="distinct names"):
        batch.bootstrap_trees(_codes(4), replicates=2, taxa=["a", "b", "c"])
    with pytest.raises(ValueError, match="distinct names"):
        batch.bootstrap_trees(_codes(4), replicates=2, taxa=["a", "b", "c", "a"])
    with pytest.raises(ValueError, match="unknown leaf"):
        batch.bootstrap_trees(_codes(4), replicates=2, taxa=list("abcd"), splits=[("ab", "cx")])
    with pytest.raises(ValueError, match="exactly one side"):
        batch.bootstrap_trees(_codes(4), replicates=2, taxa=list("abcd"), splits=[("ab", "c")])
    with pytest.raises(ValueError, match="exactly one side"):
        batch.bootstrap_trees(_codes(4), replicates=2, taxa=list("abcd"), splits=[("abc", "cd")])


def _refusal_worker(rank, world, init, out_dir):
    import os

    import torch.distributed as dist

    import splitp_b200.batch as batch
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        batch.bootstrap_trees(_codes(4), replicates=2)
        result = "returned"
    except NotImplementedError:
        result = "NotImplementedError"
    finally:
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}"), "w") as f:
        f.write(result)


def test_refused_on_several_processes(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_refusal_worker, args=(2, "file://" + str(tmp_path / "rendezvous"), str(tmp_path)), nprocs=2, join=True)
    assert [(tmp_path / f"rank{r}").read_text() for r in range(2)] == ["NotImplementedError"] * 2
