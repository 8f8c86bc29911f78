"""Oracle against the reference's rules and search.  The expected values are stored in
tests/golden/reference_checks.json (tools/gen_reference_checks.py); where the reference itself is importable
(tools/ref_loader.py) they are recomputed with it and must equal the stored ones."""
import json
import os
import random

import numpy as np
import pytest

import oracle
import prior_fns
from tools import ref_loader


@pytest.fixture(scope="module")
def stored():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")) as f:
        return json.load(f)


def _board(rec, n):
    return oracle.bits_to_board(int(rec["b"], 16), int(rec["w"], 16), n)


def _reference_rules_game(R, n):
    """The same records as tools/gen_reference_checks.rules_random_game, computed by the reference's OthelloGame."""
    Game, Player = R.Othello.OthelloGame, R.Othello.OthelloPlayer
    rng = random.Random(n)
    g = Game(n)
    out = []
    while not g.has_finished():
        board = g.board(R.Othello.BoardView.TWO_CHANNELS)
        b, w = oracle.board_to_bits(board)
        rec = {"b": "%016x" % b, "w": "%016x" % w}
        for ch, pl in ((0, Player.BLACK), (1, Player.WHITE)):
            moves = []
            for r, c in (tuple(int(x) for x in a) for a in Game.get_player_valid_actions(board, pl)):
                nb = np.copy(board)
                Game.flip_board_squares(nb, pl, r, c)
                moves.append([r, c, *("%016x" % x for x in oracle.board_to_bits(nb))])
            rec[f"moves{ch}"] = moves
        out.append(rec)
        acts = list(g.get_valid_actions())
        a = acts[rng.randrange(len(acts))]
        g.play(int(a[0]), int(a[1]))
    return out


@pytest.mark.parametrize("n", [6, 8])
def test_rules_random_game(stored, n):
    recs = stored["rules_random_game"][str(n)]
    for rec in recs:
        board = _board(rec, n)
        for ch in (0, 1):
            want = rec[f"moves{ch}"]
            assert oracle.valid_actions(board, ch) == [(r, c) for r, c, _, _ in want]
            for r, c, fb, fw in want:
                assert np.array_equal(oracle.flip_board(board, ch, r, c), _board({"b": fb, "w": fw}, n))
    if ref_loader.available():
        assert _reference_rules_game(ref_loader.load(), n) == recs


def test_search_visits_nondyadic_prior(stored):
    """Non-dyadic float32 priors: exercises numpy's pairwise np.sum order and f32/f64 Q updates."""
    want = stored["search_nondyadic"]
    n, sims = want["n"], want["sims"]
    m = oracle.Mcts(n, 1.0, prior_fns.sha_prior)
    st = oracle.initial_board(n)
    for _ in range(sims):
        m.simulate(st, 0)
    ns, v = m.visits(st)
    q, p, _ = m.node_stats(st)
    acts = [tuple(a) for a in want["actions"]]
    assert ns == want["ns"] and oracle.valid_actions(st, 0) == acts
    assert [int(v[a]) for a in acts] == want["n_sa"]
    assert [float(q[a]) for a in acts] == want["q"] and [float(p[a]) for a in acts] == want["p"]
    assert m.net_calls == want["net_calls"]
    if ref_loader.available():
        R = ref_loader.load()
        net = ref_loader.StubNet(prior_fns.sha_prior)
        mcts = R.othelo_mcts.OthelloMCTS(n, net, 1)
        rst = R.Othello.OthelloGame(n).board(R.Othello.BoardView.TWO_CHANNELS)
        for _ in range(sims):
            mcts.simulate(rst, R.Othello.OthelloPlayer.BLACK)
        h = R.MCTS.hash_ndarray(rst)
        assert mcts.N(rst) == want["ns"] and sorted(tuple(int(x) for x in a) for a in mcts.get_state_actions(rst)) == sorted(acts)
        assert [mcts.N(rst, a) for a in acts] == want["n_sa"]
        assert [float(mcts._Qsa[h][a]) for a in acts] == want["q"] and [float(mcts._Psa[h][a]) for a in acts] == want["p"]
        assert net.calls == want["net_calls"]
