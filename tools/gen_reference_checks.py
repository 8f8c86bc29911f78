"""Write tests/golden/reference_checks.json: the values that test_oracle_vs_reference.py and
test_buffer_cpu.py::test_circular_array_equals_reference compare with, so that those tests run where the original
project (OthelloZero) is not installed.

The original's sources are not part of this repository, so these values come from its restatements: the oracle
(oracle/oz_oracle.c, pinned to the original by the other golden vectors) and othellozero_b200.buffer.CircularArray.
The turn logic below is the original's (a side without a legal move passes; the game ends when neither side can
move), checked against every move of tests/golden/rules.json, which the original produced.  Wherever the original
is importable (tools/ref_loader.py), the tests recompute the same values with it and require them to equal these.

    python tools/gen_reference_checks.py
"""
from __future__ import annotations

import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import oracle  # noqa: E402
import prior_fns  # noqa: E402
from othellozero_b200.buffer import CircularArray  # noqa: E402


def _side_to_move(board, mover):
    """After `mover` played: the other side if it can move, else `mover` if it can, else None (game over)."""
    for ch in (1 - mover, mover):
        if oracle.valid_actions(board, ch):
            return ch
    return None


def rules_random_game(n):
    """The positions of test_rules_random_game's game (random.Random(n) over the mover's legal actions) with both
    sides' legal actions and the board after each of them."""
    rng = random.Random(n)
    board, ch, out = oracle.initial_board(n), 0, []
    while ch is not None:
        rec = {"b": "%016x" % oracle.board_to_bits(board)[0], "w": "%016x" % oracle.board_to_bits(board)[1]}
        for side in (0, 1):
            rec[f"moves{side}"] = [[r, c, *("%016x" % x for x in oracle.board_to_bits(oracle.flip_board(board, side, r, c)))]
                                   for r, c in oracle.valid_actions(board, side)]
        out.append(rec)
        acts = oracle.valid_actions(board, ch)
        r, c = acts[rng.randrange(len(acts))]
        board = oracle.flip_board(board, ch, r, c)
        ch = _side_to_move(board, ch)
    return out


def search_nondyadic(n=6, sims=60):
    """Root statistics after `sims` simulations from the initial position with prior_fns.sha_prior, c = 1."""
    m = oracle.Mcts(n, 1.0, prior_fns.sha_prior)
    st = oracle.initial_board(n)
    for _ in range(sims):
        m.simulate(st, 0)
    ns, v = m.visits(st)
    q, p, _ = m.node_stats(st)
    acts = oracle.valid_actions(st, 0)
    return {"n": n, "sims": sims, "ns": int(ns), "actions": [list(a) for a in acts], "n_sa": [int(v[a]) for a in acts],
            "q": [float(q[a]) for a in acts], "p": [float(p[a]) for a in acts], "net_calls": m.net_calls}


def circular_array():
    """list() and str() after each extend of test_circular_array_equals_reference's seeded sequence."""
    rng, out = random.Random(3), []
    for max_ in (1, 4, 7):
        a, steps = CircularArray(max_), []
        for _ in range(40):
            chunk = [rng.random() for _ in range(rng.randrange(0, 6))]
            a.extend(chunk)
            steps.append({"chunk": chunk, "list": list(a), "str": str(a)})
        out.append({"max": max_, "steps": steps})
    return out


def main():
    data = {"rules_random_game": {str(n): rules_random_game(n) for n in (6, 8)},
            "search_nondyadic": search_nondyadic(), "circular_array": circular_array()}
    with open(os.path.join(ROOT, "tests", "golden", "reference_checks.json"), "w") as f:
        json.dump(data, f, separators=(",", ":"))


if __name__ == "__main__":
    main()
