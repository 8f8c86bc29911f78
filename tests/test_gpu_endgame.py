"""The exact endgame solver on the device: the known 4x4 answer, exact parity with the oracle solver under both rule sets
(value and per-move margins), the per-move rows, one-ply self-consistency at 14 empties, independence from batching,
the device-pointer entry point, perfect-play winners of self-play records, and the iteration driver's --solve-empties."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_solver
from endgame_util import empties, kinds, oracle_margins, playout_positions

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RULES = ["reference", "standard"]
NONE = -128


@pytest.fixture(scope="module")
def E():
    from othellozero_b200 import engine
    return engine


def _solve(E, pos, n, rules, per_move=False, max_empties=20):
    own = np.array([o for o, _, _ in pos], dtype=np.uint64)
    opp = np.array([p for _, p, _ in pos], dtype=np.uint64)
    return E.solve_endgame(own, opp, n, max_empties=max_empties, per_move=per_move, rules=rules)


@pytest.mark.parametrize("rules", RULES)
def test_4x4_initial_position_is_minus_8(E, rules):
    black, white = 0x20400, 0x40200
    for per_move in (False, True):
        out = E.solve_endgame([black], [white], 4, per_move=per_move, rules=rules)
        assert out["margin"].tolist() == [-8] and out["nodes"][0] > 0
        if per_move:
            row = out["move_margin"][0]
            legal = int(E.legal_moves([black], [white], 4)[0])
            assert sorted(np.flatnonzero(row != NONE).tolist()) == [s for s in range(64) if legal >> s & 1]
            assert set(row[row != NONE].tolist()) == {-8} and (row != NONE).sum() == 4


@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("n,count,top", [(4, 300, 12), (6, 300, 12), (8, 300, 12)])
def test_margins_equal_oracle_solver(E, rules, n, count, top):
    O = oracle_solver.load(rules)
    pos = playout_positions(O, n, count, 10, seed=17 * n + len(rules))
    pos += playout_positions(O, n, 6, top, seed=29 * n, min_empties=11)   # a few at 11-12 empties
    assert max(empties(o, p, n) for o, p, _ in pos) >= 11 or n == 4
    k = kinds(O, pos, n)
    assert k["finished"] > 0 and k["root_pass"] > 0 and k["inner_pass"] > 0, k
    ref, ref_rows = oracle_margins(O, pos, n, per_move=True)
    val = _solve(E, pos, n, rules)
    mov = _solve(E, pos, n, rules, per_move=True)
    assert np.array_equal(val["margin"].astype(np.int64), ref)
    assert np.array_equal(mov["margin"].astype(np.int64), ref)
    assert np.array_equal(mov["move_margin"].astype(np.int64), ref_rows)
    # value mode is the max of the row wherever the mover has a move; every other square is OZ_SOLVE_NONE
    own = np.array([o for o, _, _ in pos], np.uint64)
    opp = np.array([p for _, p, _ in pos], np.uint64)
    legal = E.legal_moves(own, opp, n)
    for i in range(len(pos)):
        row = mov["move_margin"][i]
        on = np.array([(int(legal[i]) >> s) & 1 for s in range(64)], bool)
        assert (row[~on] == NONE).all() and (row[on] != NONE).all()
        if on.any():
            assert int(val["margin"][i]) == int(row[on].max())


@pytest.mark.parametrize("rules", RULES)
def test_14_empties_one_ply_consistency(E, rules):
    # 14 empties: the oracle is slow there.  (15-16 empties: a single position can take 1e7-6e7 nodes with the static
    # ordering, seconds to minutes for the one thread that searches it, too long for a test.)
    n = 8
    pp = E.perft_playouts(128, n, seed=9, max_moves=46, rules=rules)
    own = np.where(pp["player"] == 0, pp["black"], pp["white"])
    opp = np.where(pp["player"] == 0, pp["white"], pp["black"])
    e = np.array([empties(o, p, n) for o, p in zip(own, opp)])
    legal = E.legal_moves(own, opp, n)
    pick = np.flatnonzero((e == 14) & (legal != 0))[:24]
    assert pick.size == 24
    own, opp, legal = own[pick], opp[pick], legal[pick]
    root = E.solve_endgame(own, opp, n, max_empties=14, per_move=True, rules=rules)
    par, sq = [], []
    for i in range(pick.size):
        for s in range(64):
            if int(legal[i]) >> s & 1:
                par.append(i)
                sq.append(s)
    par, sq = np.array(par), np.array(sq, np.int32)
    co, cp, fl, _ = E.apply_moves(own[par], opp[par], sq, n, rules=rules)
    child = E.solve_endgame(co, cp, n, max_empties=14, rules=rules)["margin"].astype(np.int64)
    v = np.where(fl & 1, -child, child)                      # MOVE_SWAPPED: the child is the opponent's margin
    assert np.array_equal(root["move_margin"][par, sq].astype(np.int64), v)
    best = np.full(pick.size, -1000)
    np.maximum.at(best, par, v)
    assert np.array_equal(root["margin"].astype(np.int64), best)


@pytest.mark.parametrize("rules", RULES)
def test_results_do_not_depend_on_batching(E, rules):
    n = 8
    pp = E.perft_playouts(400_000, n, seed=21, max_moves=54, rules=rules)
    own = np.where(pp["player"] == 0, pp["black"], pp["white"])
    opp = np.where(pp["player"] == 0, pp["white"], pp["black"])
    occ = np.unpackbits((own | opp).view(np.uint8).reshape(-1, 8), axis=1).sum(axis=1)
    keep = np.flatnonzero(64 - occ <= 6)
    assert keep.size >= 100_000
    own, opp = own[keep], opp[keep]
    big = E.solve_endgame(own, opp, n, max_empties=6, per_move=True, rules=rules)
    rng = np.random.default_rng(5)
    sample = rng.choice(keep.size, 200, replace=False)
    for i in sample[:40]:
        alone = E.solve_endgame(own[i:i + 1], opp[i:i + 1], n, max_empties=6, per_move=True, rules=rules)
        assert alone["margin"][0] == big["margin"][i] and alone["nodes"][0] == big["nodes"][i]
        assert np.array_equal(alone["move_margin"][0], big["move_margin"][i])
    value = E.solve_endgame(own, opp, n, max_empties=6, rules=rules)
    assert np.array_equal(value["margin"], big["margin"])
    O = oracle_solver.load(rules)
    ref = oracle_margins(O, [(own[i], opp[i], 0) for i in sample], n)
    assert np.array_equal(big["margin"][sample].astype(np.int64), ref)


def test_dev_entry_point_marks_over_limit_positions_and_ignores_scoring(E):
    import ctypes as C
    import torch
    from othellozero_b200 import _lib
    L = _lib.load()
    n, rules = 6, "standard"
    O = oracle_solver.load(rules)
    pos = playout_positions(O, n, 200, 9, seed=3)
    pos += playout_positions(O, n, 40, 14, seed=4, min_empties=10)       # 10-14 empties: over the limit of 9
    own = np.array([o for o, _, _ in pos], np.uint64)
    opp = np.array([p for _, p, _ in pos], np.uint64)
    e = np.array([empties(o, p, n) for o, p in zip(own, opp)])
    ref = E.solve_endgame(own[e <= 9], opp[e <= 9], n, max_empties=9, per_move=True, rules=rules)
    dev = torch.device("cuda", 0)
    d_own = torch.from_numpy(own.view(np.int64)).to(dev)
    d_opp = torch.from_numpy(opp.view(np.int64)).to(dev)
    for flags in (_lib.RULES_STANDARD, _lib.RULES_STANDARD | _lib.SCORING_STANDARD):
        margin = torch.zeros(len(pos), dtype=torch.int8, device=dev)
        rows = torch.zeros((len(pos), 64), dtype=torch.int8, device=dev)
        nodes = torch.zeros(len(pos), dtype=torch.int64, device=dev)
        st = torch.cuda.current_stream(dev)
        rc = L.oz_endgame_solve_dev(n | flags, C.c_void_p(d_own.data_ptr()), C.c_void_p(d_opp.data_ptr()), len(pos), 9,
                                    C.c_void_p(margin.data_ptr()), C.c_void_p(rows.data_ptr()),
                                    C.c_void_p(nodes.data_ptr()), C.c_void_p(st.cuda_stream))
        _lib.check(rc)
        st.synchronize()
        m, r, nd = margin.cpu().numpy(), rows.cpu().numpy(), nodes.cpu().numpy()
        assert (m[e > 9] == NONE).all() and (r[e > 9] == NONE).all() and (nd[e > 9] == 0).all()
        assert np.array_equal(m[e <= 9], ref["margin"]) and np.array_equal(r[e <= 9], ref["move_margin"])
        assert np.array_equal(nd[e <= 9].view(np.uint64), ref["nodes"])


@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("scoring", ["reference", "standard"])
def test_selfplay_record_winners_are_perfect_play(E, rules, scoring):
    from othellozero_b200 import mcts, selfplay
    n, K = 6, 8
    sp = selfplay.SelfPlay(n, mcts.HashPriorNet(), 1.0, max_games=48, num_simulations=8, seed=7, rules=rules,
                           scoring=scoring)
    rec = sp.play(48, 1.0, 0.9)
    sp.close()
    winners = selfplay.solve_record_winners(rec, n, K, rules, scoring)
    mask = selfplay.solvable_positions(rec, n, K)
    game = np.repeat(rec["winner"][:, None], 64, axis=1)
    assert mask.sum() > 100 and np.array_equal(winners[~mask], game[~mask])
    O = oracle_solver.load(rules)
    g, p = np.nonzero(mask)
    player = rec["player"][g, p].astype(np.int64)
    own = np.where(player == 0, rec["black"][g, p], rec["white"][g, p])
    opp = np.where(player == 0, rec["white"][g, p], rec["black"][g, p])
    ref = oracle_margins(O, list(zip(own, opp, player)), n)
    assert np.array_equal(winners[g, p], E.perfect_play_winner(ref, player, scoring))
    assert (winners[g, p] != game[g, p]).any()          # e_greedy = 0.9: some game outcomes are not perfect play


def test_iteration_driver_solve_empties():
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "4", "--arena-threshold", "3",
           "--arena-simulations", "8", "--iterations", "1", "--solve-empties", "8"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = lines[0]
    assert d["config"]["solve_empties"] == 8 and d["phases"]["solve_s"] > 0
    assert 0 < d["solved_positions"] <= d["positions_gathered"]
    assert 0 <= d["solve_relabelled"] <= d["solved_positions"]
