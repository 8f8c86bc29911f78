"""Replay buffer semantics (main.py:21-53) - against the reference's own CircularArray when it is importable."""
import json
import os
import random

import numpy as np
import pytest

from othellozero_b200.buffer import CircularArray, RecordBuffer
from tools import ref_loader


def _model(max_, items):
    """The rule stated independently: a list that grows to max_, then overflow item k replaces slot k mod max_."""
    out, k = [], 0
    for it in items:
        if len(out) < max_:
            out.append(it)
        else:
            out[k % max_] = it
            k += 1
    return out


@pytest.mark.parametrize("max_,count", [(5, 3), (5, 5), (5, 17), (1, 4), (8, 64)])
def test_circular_array_overwrites_oldest(max_, count):
    ca = CircularArray(max_)
    ca.extend(range(count))
    assert list(ca) == _model(max_, range(count)) and len(ca) == min(max_, count)
    ca.append("x")
    assert list(ca) == _model(max_, list(range(count)) + ["x"])
    assert ca[0] == list(ca)[0] and repr(ca) == f"CircularArray({len(ca)})"
    random.Random(0).shuffle(ca)                      # main.py:99 shuffles the buffer in place
    assert sorted(map(str, ca)) == sorted(map(str, _model(max_, list(range(count)) + ["x"])))


def test_circular_array_equals_reference():
    """list() and str() after each extend of a seeded sequence, as stored in tests/golden/reference_checks.json
    (tools/gen_reference_checks.py); where the reference is importable its own CircularArray must match them too."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")) as f:
        stored = json.load(f)["circular_array"]
    main = ref_loader.load_main() if ref_loader.available() else None
    for case in stored:
        arrays = [CircularArray(case["max"])] + ([main.CircularArray(case["max"])] if main else [])
        items = []
        for step in case["steps"]:
            items += step["chunk"]
            assert step["list"] == _model(case["max"], items)
            for a in arrays:
                a.extend(step["chunk"])
                assert list(a) == step["list"] and len(a) == len(step["list"]) and str(a) == step["str"]


def test_record_buffer_matches_circular_array():
    rb, ca = RecordBuffer(8 * 10), CircularArray(10)
    rng = np.random.default_rng(0)
    for _ in range(12):
        rows = rng.integers(0, 2**62, size=(int(rng.integers(0, 25)), 3), dtype=np.uint64)
        rb.extend(rows)
        ca.extend([tuple(int(x) for x in r) for r in rows])
        assert [tuple(int(x) for x in r) for r in rb.positions()] == list(ca)
        assert len(rb) == 8 * len(ca)
