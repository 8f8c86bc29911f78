"""Example stream (SURVEY 8f rank 1) against the REFERENCE: `selfplay.records_to_examples*` must reproduce
training.execute_episode's list (training.py:58-72: 8 symmetries per move in the order of :13-23, one-hot policies,
z, dtypes) element for element.  The committed digests (tests/golden/examples.json) were produced by running the
reference's own execute_episode (tools/gen_golden.py examples); one of those streams is stored in full
(tests/golden/examples_reference_stream.npz, its bytes checked against the reference's digest) for the element-wise
comparison."""
import os

import numpy as np

import oracle
import prior_fns
from example_digest import examples_digest, oracle_episode_as_records
from othellozero_b200 import selfplay

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _oracle_records(g):
    predict = None if g["prior"] == "hash" else prior_fns.sha_prior
    out = oracle.execute_episode(g["n"], g["sims"], c=1.0, temperature=g["T"], e_greedy=g["e_greedy"], predict=predict,
                                 seed=g["seed"], game_id=g["game_id"])
    assert [a for a in out["moves"]] == g["moves"]
    return oracle_episode_as_records(out, g["n"])


def test_example_stream_digests(golden_examples):
    for g in golden_examples:
        rec = _oracle_records(g)
        n = g["n"]
        aliased = selfplay.records_to_examples(rec, 0, n, reference_aliasing=True)
        snap = selfplay.records_to_examples(rec, 0, n)
        batch = selfplay.records_to_examples_batch(rec, n)[0]
        assert len(aliased) == len(snap) == len(batch) == g["n_examples"]
        assert examples_digest(aliased) == g["sha256_reference_stream"]     # the reference's stream, byte for byte
        assert examples_digest(snap) == g["sha256_snapshot_stream"]        # same stream with true per-move boards
        assert examples_digest(batch) == g["sha256_snapshot_stream"]
        assert all(type(z) is int for _, _, z in aliased + snap + batch)


def test_example_stream_elementwise_vs_live_reference(golden_examples):
    g = golden_examples[1]  # 6x6, T = 0, e_greedy 0.7: every draw site is exercised
    with np.load(os.path.join(GOLDEN, "examples_reference_stream.npz")) as f:
        ref = [(b, p, int(z)) for b, p, z in zip(f["board"], f["policy"], f["z"])]
    assert examples_digest(ref) == g["sha256_reference_stream"]  # the stored stream is the reference's, byte for byte
    rec = _oracle_records(g)
    ours = selfplay.records_to_examples(rec, 0, g["n"], reference_aliasing=True)
    assert len(ours) == len(ref)
    for (b1, p1, z1), (b2, p2, z2) in zip(ours, ref):
        assert b1.dtype == b2.dtype == bool and b1.shape == b2.shape and np.array_equal(b1, b2)
        assert p1.dtype == p2.dtype == np.float64 and np.array_equal(p1, p2)
        assert z1 == z2 and type(z1) is type(z2) is int
    # the per-move snapshots differ from the aliased stream only in the boards
    snap = selfplay.records_to_examples(rec, 0, g["n"])
    assert all(np.array_equal(a[1], b[1]) and a[2] == b[2] for a, b in zip(snap, ref))
    assert not np.array_equal(snap[0][0], ref[0][0])  # the first move's true board is not the final position
