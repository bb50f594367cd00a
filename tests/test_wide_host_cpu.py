"""CPU-only tests of the host side of 32..64-taxon pattern mappings: 128-bit key encoding and decoding
(engine.encode_patterns / decode_keys) and their errors.  No device is needed."""
import random

import numpy as np
import pytest


def _as_int(key):
    """Python int of a key: uint64 scalar or {lo, hi} pair."""
    return int(key) if np.ndim(key) == 0 else (int(key[1]) << 64) | int(key[0])


def _reference_key(pattern):
    v = 0
    for c in pattern:
        v = v * 4 + "ACGT".index(c)  # __index_of (constructions.py:166-171): taxon 0 most significant
    return v


@pytest.mark.parametrize("n", [32, 33, 40, 64])
def test_wide_encode_decode_round_trip(n):
    from splitp_b200 import engine
    rng = random.Random(n)
    pats = ["".join(rng.choice("ACGT") for _ in range(n)) for _ in range(200)]
    pats += ["A" * n, "T" * n, "A" * (n - 1) + "C", "C" + "A" * (n - 1), "T" * 32 + "A" * (n - 32), "A" * (n - 32) + "T" * 32]
    keys, m = engine.encode_patterns(pats)
    assert m == n and keys.dtype == np.uint64 and keys.shape == (len(pats), 2)
    assert [_as_int(k) for k in keys] == [_reference_key(p) for p in pats]
    assert engine.decode_keys(keys, n) == pats
    if n == 64:  # the all-T pattern of 64 taxa is the all-ones key (the EMPTY marker of the hashed wide table)
        assert keys[pats.index("T" * 64)].tolist() == [2 ** 64 - 1, 2 ** 64 - 1]


def test_narrow_keys_unchanged_at_31_taxa():
    from splitp_b200 import engine
    pats = ["T" * 31, "ACGT" * 7 + "ACG"]
    keys, n = engine.encode_patterns(pats)
    assert n == 31 and keys.shape == (2,) and keys.dtype == np.uint64
    assert [int(k) for k in keys] == [_reference_key(p) for p in pats]


@pytest.mark.parametrize("bad", ["N", "a", "-", "U"])
def test_wide_encode_rejects_non_acgt(bad):
    from splitp_b200 import engine
    pats = ["ACGT" * 10, "ACGT" * 9 + "AC" + bad + "T"]
    with pytest.raises(KeyError) as err:
        engine.encode_patterns(pats)
    assert err.value.args[0] == bad
    with pytest.raises(KeyError):
        engine.encode_patterns(["A" * 40, "A" * 39])  # patterns of unequal length


def test_more_than_64_taxa_raises():
    from splitp_b200 import engine
    with pytest.raises(NotImplementedError, match="64 taxa"):
        engine.encode_patterns(["A" * 65])
