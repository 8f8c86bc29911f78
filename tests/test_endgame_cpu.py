"""The exact endgame solver without a GPU: the oracle solver (known 4x4 answer, its source, alpha-beta against unpruned
minimax, finished positions), perfect_play_winner, per-position winners through packed rows and training examples,
--solve-empties, and the C-ABI's argument checks that fail before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

import oracle_solver
from endgame_util import empties, kinds, playout_positions

RULES = ["reference", "standard"]


@pytest.mark.parametrize("rules", RULES)
def test_oracle_solver_4x4_initial_position(rules):
    O = oracle_solver.load(rules)
    b = O.initial_board(4)
    assert O.solve_margin(b, 0) == -8 and O.solve_minimax(b, 0) == -8
    moves = O.solve_move_margins(b, 0)
    assert len(moves) == 4 and set(moves.values()) == {-8}


@pytest.mark.parametrize("rules", RULES)
def test_oracle_solver_source_is_base_plus_appended_text(rules):
    base, src = oracle_solver.base_source(rules), oracle_solver.source(rules)
    assert src.startswith(base) and src[len(base):] == oracle_solver.SOLVER
    assert "orc_solve_margin" not in base and "orc_solve_minimax" not in base


@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("n", [4, 6, 8])
def test_oracle_alphabeta_equals_minimax(rules, n):
    O = oracle_solver.load(rules)
    pos = playout_positions(O, n, 120, 8, seed=100 + n)
    k = kinds(O, pos, n)
    assert k["finished"] > 0 and k["root_pass"] + k["inner_pass"] > 0, k
    for own, opp, _ in pos:
        b = O.bits_to_board(int(own), int(opp), n)
        assert O.solve_margin(b, 0) == O.solve_minimax(b, 0), (own, opp)


@pytest.mark.parametrize("rules", RULES)
def test_oracle_finished_positions_are_their_disc_difference(rules):
    O = oracle_solver.load(rules)
    for n in (4, 6, 8):
        for g in range(20):
            st = O.playout(n, 5, g)
            assert st["finished"]
            k0, k1 = int(st["board"][:, :, 0].sum()), int(st["board"][:, :, 1].sum())
            assert O.solve_margin(st["board"], 0) == k0 - k1 and O.solve_margin(st["board"], 1) == k1 - k0


def test_perfect_play_winner_table():
    from othellozero_b200 import engine
    from othellozero_b200._lib import WINNER_DRAW
    margin = np.array([5, 5, -3, -3, 0, 0])
    player = np.array([0, 1, 0, 1, 0, 1])
    assert engine.perfect_play_winner(margin, player).tolist() == [0, 1, 1, 0, 0, 0]
    assert engine.perfect_play_winner(margin, player, "reference").tolist() == [0, 1, 1, 0, 0, 0]
    assert engine.perfect_play_winner(margin, player, "standard").tolist() == [0, 1, 1, 0, WINNER_DRAW, WINNER_DRAW]
    assert engine.perfect_play_winner(np.array([64, -64]), np.array([1, 1]), "standard").tolist() == [1, 0]
    with pytest.raises(ValueError):
        engine.perfect_play_winner(margin, player, "tournament")


def _record(n=6, k=5):
    rng = np.random.default_rng(11)
    return {"n_moves": np.array([k, k], dtype=np.int32), "winner": np.array([0, 1], dtype=np.int32),
            "black": rng.integers(0, 2 ** 36, (2, 64), dtype=np.uint64),
            "white": rng.integers(0, 2 ** 36, (2, 64), dtype=np.uint64),
            "action": rng.integers(0, n, (2, 64)).astype(np.uint8) * 9,
            "player": (np.arange(64)[None, :] % 2).repeat(2, 0).astype(np.uint8)}


def _winners(rec):
    w = np.repeat(rec["winner"][:, None], 64, axis=1).astype(np.int32)
    w[0, 3:5] = 1      # game 0 (BLACK won): its last two positions are WHITE wins under perfect play
    w[1, 4] = 2        # game 1: a draw at its last position
    return w


def test_packed_rows_carry_per_position_winners():
    from othellozero_b200 import dist, iteration
    rec = _record()
    assert np.array_equal(dist.pack_records(rec, None), dist.pack_records(rec))
    rows = dist.pack_records(rec, _winners(rec))
    plain = dist.pack_records(rec)
    assert np.array_equal(rows[:, :2], plain[:, :2])
    assert ((rows[:, 2] >> np.uint64(16)) & np.uint64(0xFF)).tolist() == [0, 0, 0, 1, 1] + [1, 1, 1, 1, 2]
    *_, z = iteration.unpack_rows(rows)
    # players alternate 0, 1, 0, 1, 0: z = +1 where the (per-position) winner moved, 0 on the draw
    assert z.tolist() == [1, -1, 1, 1, -1] + [-1, 1, -1, 1, 0]
    *_, z0 = iteration.unpack_rows(plain)
    assert z0.tolist() == [1, -1, 1, -1, 1] + [-1, 1, -1, 1, -1]


def test_examples_batch_takes_per_position_winners():
    from othellozero_b200 import selfplay
    n, rec = 6, _record()
    plain = selfplay.records_to_examples_batch(rec, n)
    same = selfplay.records_to_examples_batch(rec, n, winners=None)
    for a, b in zip(plain, same):
        for (b1, p1, z1), (b2, p2, z2) in zip(a, b):
            assert np.array_equal(b1, b2) and np.array_equal(p1, p2) and z1 == z2
    solved = selfplay.records_to_examples_batch(rec, n, winners=_winners(rec))
    assert [z for _, _, z in solved[0][::8]] == [1, -1, 1, 1, -1]
    assert [z for _, _, z in solved[1][::8]] == [-1, 1, -1, 1, 0]
    for a, b in zip(plain, solved):
        for (b1, p1, _), (b2, p2, _) in zip(a, b):
            assert np.array_equal(b1, b2) and np.array_equal(p1, p2)


def test_solvable_positions_counts_empties():
    from othellozero_b200 import selfplay
    rec = _record(6)
    mask = selfplay.solvable_positions(rec, 6, 20)
    for g in range(2):
        for p in range(64):
            e = empties(rec["black"][g, p], rec["white"][g, p], 6) if p < 5 else None
            assert mask[g, p] == (p < 5 and e <= 20)


def test_execute_episodes_rejects_solving_with_reference_aliasing():
    from othellozero_b200 import mcts, selfplay
    with pytest.raises(ValueError):
        selfplay.execute_episodes(1, 6, mcts.HashPriorNet(), 1.0, 4, 1.0, 1.0, reference_aliasing=True, solve_empties=6)


def test_iteration_cli_takes_solve_empties(monkeypatch):
    from othellozero_b200 import iteration
    assert iteration.IterationConfig().solve_empties == 0
    for bad in ("-1", "21", "x"):
        with pytest.raises(SystemExit):
            iteration.main(["--solve-empties", bad])
    seen = {}

    class Stop(Exception):
        pass

    def fake_trainer(cfg):
        seen["cfg"] = cfg
        raise Stop

    monkeypatch.setattr(iteration, "Trainer", fake_trainer)
    for k in (0, 12, 20):
        with pytest.raises(Stop):
            iteration.main(["--solve-empties", str(k)])
        assert seen["cfg"].solve_empties == k


def test_abi_solver_argument_errors_fail_before_cuda():
    from othellozero_b200 import _lib, engine
    L = _lib.load()
    assert _lib.SOLVE_MAX_EMPTIES == 20 and _lib.SOLVE_NONE == -128
    own, opp = np.array([0x0000000810000000], np.uint64), np.array([0x0000001008000000], np.uint64)
    margin, nodes = np.zeros(1, np.int8), np.zeros(1, np.uint64)
    rows = np.zeros((1, 64), np.int8)
    u64p, i8p = _lib.u64p, _lib.i8p

    def host(bs=8, me=20, o=own, p=opp, m=margin, n=1):
        return L.oz_endgame_solve_host(0, bs, _lib.ptr(o, u64p), _lib.ptr(p, u64p), n, me, _lib.ptr(m, i8p),
                                       _lib.ptr(rows, i8p), _lib.ptr(nodes, u64p))

    def dev(bs=8, me=20, o=own, p=opp, m=margin, n=1):
        vp = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        return L.oz_endgame_solve_dev(bs, vp(o), vp(p), n, me, vp(m), None, None, None)

    for call in (host, dev):
        assert call(bs=0x200 | 8) == _lib.OZ_ERR_INVALID
        assert call(bs=5) == _lib.OZ_ERR_INVALID
        assert call(me=21) == _lib.OZ_ERR_INVALID and "max_empties" in L.oz_last_error().decode()
        assert call(me=-1) == _lib.OZ_ERR_INVALID
        assert call(o=None) == _lib.OZ_ERR_INVALID and "null" in L.oz_last_error().decode()
        assert call(p=None) == _lib.OZ_ERR_INVALID
        assert call(m=None) == _lib.OZ_ERR_INVALID
        assert call(n=-1) == _lib.OZ_ERR_INVALID
        assert call(o=None, p=None, m=None, n=0) == _lib.OZ_OK   # nothing to do
    # _host checks the content of every position before launching: the first bad one is named (4x4: at most 16 empties)
    two = lambda a, b: np.array([a, b], np.uint64)
    m2 = np.zeros(2, np.int8)
    b4, w4 = 0x20400, 0x40200                                             # the 4x4 initial position
    assert host(bs=4, o=two(b4, 1), p=two(w4, 1), m=m2, n=2) == _lib.OZ_ERR_INVALID
    assert "position 1" in L.oz_last_error().decode() and "overlap" in L.oz_last_error().decode()
    assert host(bs=4, o=two(b4, b4 | 1 << 4), p=two(w4, w4), m=m2, n=2) == _lib.OZ_ERR_INVALID
    assert "position 1" in L.oz_last_error().decode() and "outside" in L.oz_last_error().decode()
    assert host(me=16) == _lib.OZ_ERR_INVALID and "position 0: 60 empties" in L.oz_last_error().decode()
    with pytest.raises(AssertionError):
        engine.solve_endgame(own, opp, max_empties=21)
    with pytest.raises(ValueError):
        engine.solve_endgame(own, opp, rules="tournament")
