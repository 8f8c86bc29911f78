"""Standard search values without a GPU: the header constants, argument checks in Python, the C-ABI and the CLI, the
standard-values oracle's source diff, and its semantics on positions taken from seeded random games: a game-ending
winning move is worth +1 to its edge (-1 under the reference's values, SURVEY A.3's probe), a value crossing a pass keeps
its sign, and with leaf solving every child of a root with at most K+1 empties is worth the sign of its exact margin."""
import difflib
import os
import re

import numpy as np
import pytest

import oracle
import oracle_scoring
import oracle_solver
import oracle_standard
import oracle_values

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASES = [(r, s) for r in ("reference", "standard") for s in ("reference", "standard")]


def _base_oracle(rules, scoring):
    if scoring == "standard":
        return oracle_scoring.load(rules)
    return oracle if rules == "reference" else oracle_standard.load()


def _canon(board, player):
    return board if player == 0 else board[..., ::-1]


# ---- constants and argument checks ------------------------------------------------------------------------------------
def test_header_constants_match_lib():
    from othellozero_b200 import _lib
    h = open(os.path.join(ROOT, "include", "oz_b200.h")).read()
    defs = dict(re.findall(r"#define (OZ_VALUES_\w+|OZ_SOLVE_LEAVES_MAX)\s+(\d+)", h))
    assert int(defs["OZ_VALUES_REFERENCE"]) == _lib.VALUES.index("reference") == 0
    assert int(defs["OZ_VALUES_STANDARD"]) == _lib.VALUES.index("standard") == 1
    assert int(defs["OZ_SOLVE_LEAVES_MAX"]) == _lib.SOLVE_LEAVES_MAX == 12
    assert "int oz_search_set_values(oz_engine* e, int32_t values, int32_t solve_leaves);" in h
    assert "int oz_search_solve_counters(oz_engine* e, uint64_t* out2);" in h


def test_values_arg_validation():
    from othellozero_b200 import _lib
    assert _lib.values_arg() == 0 and _lib.values_arg("standard") == 1
    assert _lib.values_arg("standard", 12, "standard") == 1 and _lib.values_arg("standard", 0, "reference") == 1
    for args in [("x",), ("standard", 13, "standard"), ("standard", -1, "standard"), ("standard", 4, "reference"),
                 ("reference", 4, "standard"), ("standard", 4.0, "standard"), ("standard", True, "standard")]:
        with pytest.raises(ValueError):
            _lib.values_arg(*args)


def test_python_entry_points_reject_bad_values_before_the_device():
    from othellozero_b200 import arena, engine, selfplay
    from othellozero_b200.mcts import HashPriorNet
    with pytest.raises(ValueError):
        engine.Engine(8, values="x")
    with pytest.raises(ValueError):
        engine.Engine(8, values="standard", solve_leaves=6)               # reference scoring
    with pytest.raises(ValueError):
        selfplay.execute_episodes(1, 6, HashPriorNet(), 1.0, 4, 1.0, 1.0, values="reference", solve_leaves=4,
                                  scoring="standard")
    with pytest.raises(ValueError):
        selfplay.make_b200_worker(values="standard", solve_leaves=13, scoring="standard")
    with pytest.raises(ValueError):
        arena.pit(6, HashPriorNet(), HashPriorNet(), 4, values=("standard", "bogus"))
    with pytest.raises(ValueError):
        arena.evaluate_neural_network(6, 2, HashPriorNet(), 4, 1.0, values="standard", solve_leaves=3)


def test_abi_set_values_null_engine_fails_before_cuda():
    from othellozero_b200 import _lib
    L = _lib.load()
    assert L.oz_search_set_values(None, 1, 0) == _lib.OZ_ERR_INVALID and "null" in L.oz_last_error().decode()
    assert L.oz_search_solve_counters(None, None) == _lib.OZ_ERR_INVALID


def test_iteration_cli_takes_values_and_solve_leaves(monkeypatch):
    from othellozero_b200 import iteration
    cfg = iteration.IterationConfig()
    assert cfg.values == "reference" and cfg.solve_leaves == 0
    for bad in (["--values", "x"], ["--solve-leaves", "13", "--values", "standard", "--scoring", "standard"],
                ["--solve-leaves", "4"], ["--solve-leaves", "4", "--values", "standard"],
                ["--solve-leaves", "4", "--scoring", "standard"]):
        with pytest.raises(SystemExit):
            iteration.main(bad)
    seen = {}

    class Stop(Exception):
        pass

    def fake_trainer(c):
        seen["cfg"] = c
        raise Stop

    monkeypatch.setattr(iteration, "Trainer", fake_trainer)
    for k in (0, 8, 12):
        with pytest.raises(Stop):
            iteration.main(["--rules", "standard", "--scoring", "standard", "--values", "standard", "--solve-leaves",
                            str(k), "--solve-empties", "10"])
        c = seen["cfg"]
        assert (c.values, c.solve_leaves, c.solve_empties, c.scoring) == ("standard", k, 10, "standard")
    with pytest.raises(Stop):
        iteration.main(["--values", "standard"])
    assert seen["cfg"].values == "standard" and seen["cfg"].solve_leaves == 0


def test_cli_help_keeps_the_two_solver_flags_apart(capsys):
    from othellozero_b200 import iteration
    with pytest.raises(SystemExit):
        iteration.main(["--help"])
    out = " ".join(capsys.readouterr().out.split())
    assert "--solve-empties" in out and "--solve-leaves" in out and "training targets" in out and "search: new leaves" in out


# ---- the oracle's source ----------------------------------------------------------------------------------------------
def _changed_lines(a, b):
    out = []
    for line in difflib.unified_diff(a.splitlines(), b.splitlines(), lineterm="", n=0):
        if line.startswith(("+++", "---", "@@")):
            continue
        out.append(line)
    return out


@pytest.mark.parametrize("rules,scoring", BASES)
def test_values_oracle_source_differs_from_its_base_by_exactly_the_patch(rules, scoring):
    base = oracle_values.base_source(rules, scoring)
    if scoring == "standard":
        assert base == oracle_scoring.source(rules)
    else:
        ref = open(os.path.join(ROOT, "oracle", "oz_oracle.c")).read()
        assert base == (oracle_standard.source() if rules == "standard" else ref)
    k0 = oracle_values.source(rules, scoring, 0)
    removed = [l[1:] for l in _changed_lines(base, k0) if l.startswith("-")]
    added = [l[1:] for l in _changed_lines(base, k0) if l.startswith("+")]
    assert removed == [oracle_values.SWAP_ANCHOR.rstrip("\n")]
    assert added == (oracle_values.SWAP + oracle_values.NEGATE).rstrip("\n").split("\n")
    if scoring == "standard":
        k = oracle_values.source(rules, scoring, 8)
        assert k.endswith(oracle_solver.SOLVER)
        body = k[: -len(oracle_solver.SOLVER)]
        # two insertions into the K = 0 variant, nothing else
        for ins in (oracle_values.DECL, oracle_values.leaf(8)):
            assert body.count(ins) == 1
            body = body.replace(ins, "")
        assert body == k0
    else:
        with pytest.raises(ValueError):
            oracle_values.source(rules, scoring, 8)


# ---- the oracle's semantics ---------------------------------------------------------------------------------------------
def _positions(O, n, seed, want, count, games=4000):
    """Positions of seeded random games (the oracle's playouts) that satisfy want(board, player) -> value or None."""
    out = []
    for g in range(games):
        full = O.playout(n, seed, g)
        for k in range(len(full["moves"])):
            st = O.playout(n, seed, g, max_moves=k)
            w = want(O, st["board"], st["player"])
            if w is not None:
                out.append((st["board"], st["player"], w))
                break
        if len(out) == count:
            return out
    raise AssertionError("not enough positions")


def _q(m, board, player, sq):
    q, _, tag = m.node_stats(_canon(board, player))
    r, c = divmod(sq, board.shape[0])
    return q[r, c], tag[r, c]


@pytest.mark.parametrize("rules,scoring", BASES)
def test_game_ending_winning_move_is_worth_plus_one(rules, scoring):
    """SURVEY A.3's probe: a single legal move that ends the game with the mover ahead backs up -1 under the reference's
    values; under standard values it is worth +1 (and a losing one -1)."""
    n = 4
    R = _base_oracle(rules, scoring)
    V = oracle_values.load(rules, scoring, 0)
    V.build()

    def want(O, b, p):
        acts = O.valid_actions(b, p)
        if len(acts) != 1:
            return None
        child = O.flip_board(b, p, *acts[0])
        if not O.has_finished(child):
            return None
        ch, _ = O.winner(child)
        return (acts[0][0] * n + acts[0][1], ch)

    seen = set()
    for board, player, (sq, ch) in _positions(R, n, 3, want, 12):
        if ch == 2:
            continue
        mover_won = ch == player
        outs = {}
        for name, O in (("reference", R), ("standard", V)):
            m = O.Mcts(n)
            for _ in range(2):
                m.simulate(board, player)
            outs[name] = _q(m, board, player, sq)
        assert outs["standard"] == ((1.0 if mover_won else -1.0), 1)
        assert outs["reference"] == ((-1.0 if mover_won else 1.0), 1)
        seen.add(mover_won)
    assert True in seen


@pytest.mark.parametrize("rules,scoring", BASES)
def test_value_crossing_a_pass_keeps_its_sign(rules, scoring):
    R = _base_oracle(rules, scoring)
    V = oracle_values.load(rules, scoring, 0)
    for n in (4, 6):
        def want(O, b, p):
            acts = O.valid_actions(b, p)
            if len(acts) != 1:
                return None
            child = O.flip_board(b, p, *acts[0])
            if O.has_finished(child) or O.valid_actions(child, 1 - p):
                return None
            return acts[0][0] * n + acts[0][1]

        for board, player, sq in _positions(R, n, 5, want, 4):
            r, c = divmod(sq, n)
            child = _canon(R.flip_board(board, player, r, c), player)    # the mover keeps the move: ch0 = mover
            v = float(np.float32(R.hash_prior(child)[1]))
            got = {}
            for name, O in (("reference", R), ("standard", V)):
                m = O.Mcts(n)
                for _ in range(2):
                    m.simulate(board, player)
                got[name] = _q(m, board, player, sq)
            assert got["standard"] == (v, 2) and got["reference"] == (-v, 2)


@pytest.mark.parametrize("rules", ["reference", "standard"])
@pytest.mark.parametrize("n,k", [(4, 4), (4, 8), (6, 6)])
def test_solved_children_are_worth_the_sign_of_their_exact_margin(rules, n, k):
    V = oracle_values.load(rules, "standard", k)
    S = oracle_solver.load(rules)
    R = oracle_scoring.load(rules)

    def want(O, b, p):
        empties = n * n - int(b.sum())
        return empties if 2 <= empties <= k + 1 and O.valid_actions(b, p) else None

    checked = 0
    for board, player, _ in _positions(R, n, 11 + k, want, 6):
        m = V.Mcts(n)
        for _ in range(40):
            m.simulate(board, player)
        assert m.nodes == 1                                    # the root is expanded; every child below it is solved
        ns, counts = m.visits(_canon(board, player))
        assert ns == 39
        for sq, margin in S.solve_move_margins(board, player).items():
            r, c = divmod(sq, 8)
            if counts[r, c]:
                q, tag = _q(m, board, player, r * n + c)
                assert (q, tag) == (float(np.sign(margin)), 1), (sq, margin)
                checked += 1
    assert checked >= 6
