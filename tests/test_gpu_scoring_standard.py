"""Standard scoring on the device (a finished game with equal disc counts is a draw, worth 0 in the search, winner code 2 in
self-play): the search and self-play against the draw-scoring oracles under both rule sets, bit for bit, virtual-loss
waves, the arena, the game classes and the iteration driver.  Draws are rare from the initial position, so most roots
and starts are positions a few plies before the end of seeded random games that ended drawn."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
import oracle_scoring
import oracle_standard
import prior_fns
from gpu_util import canon_board, sq8, visits_to_grid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STD = "standard"
RULES = ["reference", "standard"]


@pytest.fixture(scope="module")
def E():
    from othellozero_b200 import engine
    return engine


def _base_oracle(rules):
    """The oracle under `rules` with reference scoring."""
    return oracle if rules == "reference" else oracle_standard.load()


def _near_draw_starts(rules, n, count, seed, back=(4, 10)):
    """Positions `back` plies (drawn per game) before the end of engine-RNG random playouts under `rules` that ended
    drawn -> list of (black, white, player, board)."""
    D = oracle_scoring.load(rules)
    rng = np.random.default_rng(seed)
    out, g = [], 0
    while len(out) < count:
        full = D.playout(n, seed, g)
        g += 1
        assert g < 20000
        if not full["finished"] or D.winner(full["board"])[0] != 2:
            continue
        k = len(full["moves"]) - int(rng.integers(back[0], back[1] + 1))
        if k < 0:
            continue
        st = D.playout(n, seed, g - 1, max_moves=k)
        assert not st["finished"]
        out.append((st["black"], st["white"], st["player"], st["board"]))
    return out


def _bits(q):
    return np.asarray(q, dtype=np.float64).view(np.int64)


# ---- 1. sequential search against the draw-scoring oracle ----------------------------------------------------------------
@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("prior", ["hash", "host"])
def test_sequential_search_equals_draw_scoring_oracle(E, rules, prior):
    n, sims = 8, 160
    D = oracle_scoring.load(rules)
    R = _base_oracle(rules)
    changed = terminal = 0
    for black, white, player, board in _near_draw_starts(rules, n, 5, seed=21 if prior == "hash" else 22):
        if prior == "hash":
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HASH, rules=rules, scoring=STD)
            m, r = D.Mcts(n), R.Mcts(n)
        else:
            def predict_batch(own, opp):
                outs = [prior_fns.sha_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
                return np.stack([o[0].ravel() for o in outs]), np.array([o[1] for o in outs], dtype=np.float32)
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HOST, rules=rules, scoring=STD)
            m, r = D.Mcts(n, predict=prior_fns.sha_prior), R.Mcts(n, predict=prior_fns.sha_prior)
        e.reset(1, [black], [white], [player])
        e.search(sims, predict_batch if prior == "host" else None)
        v, ns = e.visits()
        q, p, tag = e.root_stats(0)
        c = e.counters()
        e.close()
        terminal += c["terminal_visits"]
        for _ in range(sims):
            m.simulate(board, player)
            r.simulate(board, player)
        canon = board if player == 0 else board[..., ::-1]
        rns, rv = m.visits(canon)
        assert int(ns[0]) == rns and visits_to_grid(v[0], n).tolist() == rv.reshape(-1).tolist(), hex(black)
        assert c["nodes"] == m.nodes
        rq, rp, rtag = m.node_stats(canon)
        for rr in range(n):
            for cc in range(n):
                if rtag[rr, cc] >= 0:
                    s = rr * 8 + cc
                    assert _bits(q[s]) == _bits(rq[rr, cc]) and p[s] == rp[rr, cc] and tag[s] == rtag[rr, cc], (hex(black), s)
        # the same search under reference scoring: the drawn terminals it visited are valued differently there
        _, qv = r.visits(canon)
        qq = r.node_stats(canon)[0]
        changed += (qv.tolist() != rv.tolist()) or not np.array_equal(_bits(qq), _bits(rq))
    assert terminal > 0
    assert changed > 0            # the oracle's search reached drawn terminals, and the feature changes results


# ---- 2. self-play with the hash prior against the oracle ----------------------------------------------------------------
@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("n,sims,T,eg", [(4, 12, 1.0, 0.8), (4, 6, 0.0, 0.9), (6, 16, 1.0, 0.9), (6, 8, 0.0, 0.9),
                                         (8, 20, 1.0, 0.9), (8, 8, 0.0, 0.9)])
def test_selfplay_hash_prior_equals_draw_scoring_oracle(E, rules, n, sims, T, eg):
    D = oracle_scoring.load(rules)
    near = _near_draw_starts(rules, n, 12, seed=30 + n, back=(1, 4))
    starts = [(s["black"], s["white"], s["player"], s["board"]) for s in (D.playout(n, 4, g, max_moves=g % 3)
                                                                       for g in range(4))] + near
    G, slots = len(starts), 5                                    # more games than slots: the device queue is used
    black = [s[0] for s in starts]; white = [s[1] for s in starts]; player = [s[2] for s in starts]
    ids = [700 + g for g in range(G)]
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=13, log_visits=True, rules=rules, scoring=STD)
    e.selfplay_begin(G, sims, T, eg, -1, black, white, player, ids)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    e.close()
    for g in range(G):
        ref = D.execute_episode(n, sims, temperature=T, e_greedy=eg, seed=13, game_id=ids[g], start_board=starts[g][3],
                                start_player=player[g], log_visits=True)
        k = int(out["n_moves"][g])
        assert [int(a) for a in out["action"][g][:k]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert [int(x) for x in out["black"][g][:k]] == ref["black"] and [int(x) for x in out["white"][g][:k]] == ref["white"]
        assert int(out["winner"][g]) == ref["winner"], g
        for p in range(k):
            assert visits_to_grid(out["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    assert (out["winner"] == 2).sum() >= 2
    assert set(int(w) for w in out["winner"]) <= {0, 1, 2}


# ---- 3. self-play with the network against the oracle fed the device priors --------------------------------------------
@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("n", [6, 8])
def test_selfplay_network_equals_draw_scoring_oracle_fed_device_priors(E, rules, n):
    from othellozero_b200 import net as oznet
    D = oracle_scoring.load(rules)
    C, sims, slots = 128, 24, 4
    blob = oznet.init_weights(n, C, seed=8, randomize_bn=True)
    starts = _near_draw_starts(rules, n, 8, seed=50 + n, back=(1, 6))
    black = np.array([s[0] for s in starts], dtype=np.uint64)
    white = np.array([s[1] for s in starts], dtype=np.uint64)
    player = np.array([s[2] for s in starts], dtype=np.int32)
    games = len(starts)
    ids = np.arange(40, 40 + games, dtype=np.uint64)
    e = E.Engine(n, slots, sims * 12 + 64, E.PRIOR_NET, seed=2, log_visits=True, eval_cache_log2=14, rules=rules,
                 scoring=STD)
    e.load_weights(blob, C)
    e.selfplay_begin(games, sims, 1.0, 0.9, -1, black, white, player, ids)
    assert e.selfplay_run(-1) == 0
    rec = e.selfplay_records()
    e.close()
    f = E.Engine(n, 4, 2, E.PRIOR_NET)
    f.load_weights(blob, C)
    cache = {}

    def predict(board):
        o, p = oznet.boards_to_bits(board)
        key = (int(o[0]), int(p[0]))
        if key not in cache:
            pi, _, v = f.net_forward(o, p, want_logits=False)
            cache[key] = (pi[0].reshape(n, n).copy(), np.float32(v[0]))
        return cache[key]

    for g in range(games):
        ref = D.execute_episode(n, sims, temperature=1.0, e_greedy=0.9, predict=predict, seed=2, game_id=int(ids[g]),
                                start_board=starts[g][3], start_player=int(player[g]), log_visits=True)
        k = int(rec["n_moves"][g])
        assert k == len(ref["moves"])
        assert [int(a) for a in rec["action"][g][:k]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert int(rec["winner"][g]) == ref["winner"], g
        for p in range(k):
            assert visits_to_grid(rec["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    f.close()


# ---- 4. virtual-loss waves ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rules", RULES)
def test_wave_search_standard_scoring(E, rules):
    sims, V = 203, 4
    roots = _near_draw_starts(rules, 8, 3, seed=9)
    outs = []
    for _ in range(2):
        e = E.Engine(8, 3, sims + 16, E.PRIOR_HASH, vl_width=V, rules=rules, scoring=STD)
        e.reset(3, [r[0] for r in roots], [r[1] for r in roots], [r[2] for r in roots])
        e.search(sims)
        v, ns = e.visits()
        assert (ns == sims - 1).all() and (v.sum(axis=1) == ns).all()   # visits conserved, no virtual loss left
        e.search(50)
        v2, ns2 = e.visits()
        assert (ns2 == sims + 49).all() and (v2.sum(axis=1) == ns2).all()
        assert e.counters()["terminal_visits"] > 0
        outs.append(v2.copy())
        e.close()
    assert np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("rules", RULES)
def test_wave_selfplay_standard_scoring_is_deterministic_and_cache_independent(E, rules):
    from othellozero_b200 import net as oznet
    n, C, sims, V = 6, 128, 16, 4
    blob = oznet.init_weights(n, C, seed=4, randomize_bn=True)
    starts = _near_draw_starts(rules, n, 16, seed=61, back=(1, 6))
    black = np.array([s[0] for s in starts], dtype=np.uint64)
    white = np.array([s[1] for s in starts], dtype=np.uint64)
    player = np.array([s[2] for s in starts], dtype=np.int32)
    outs = []
    for cache in (14, 14, 0):
        e = E.Engine(n, 8, sims * 40 + 64, E.PRIOR_NET, seed=3, vl_width=V, eval_cache_log2=cache, rules=rules,
                     scoring=STD)
        e.load_weights(blob, C)
        e.selfplay_begin(len(starts), sims, 1.0, 0.9, -1, black, white, player, np.arange(len(starts), dtype=np.uint64))
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        e.close()
    for o in outs[1:]:
        for k in ("action", "n_moves", "winner", "black", "white"):
            assert np.array_equal(outs[0][k], o[k]), k
    assert set(int(w) for w in outs[0]["winner"]) <= {0, 1, 2}


# ---- 5. the arena ----------------------------------------------------------------------------------------------------------
def _popcount(x):
    return bin(int(x)).count("1")


@pytest.mark.parametrize("rules", RULES)
def test_arena_reports_draws(E, rules):
    from othellozero_b200 import arena
    from othellozero_b200.mcts import HashPriorNet
    n, G = 4, 96
    outs = {}
    for scoring in ("reference", STD):
        outs[scoring] = arena.pit(n, HashPriorNet(), arena.RANDOM_AGENT, 8, n_games=G, rng=np.random.default_rng(5),
                                  rules=rules, scoring=scoring)
    out = outs[STD]
    cb = np.array([_popcount(b) for b in out["black"]])
    cw = np.array([_popcount(w) for w in out["white"]])
    D = oracle_scoring.load(rules)
    for g in range(G):                                             # every game ran to its end
        assert D.has_finished(oracle.bits_to_board(int(out["black"][g]), int(out["white"][g]), n))
    assert np.array_equal(out["draws"], cb == cw) and out["draws"].sum() >= 2
    assert np.array_equal(out["winner"], np.where(cb > cw, 0, np.where(cb < cw, 1, 2)))
    ref = outs["reference"]
    rb = np.array([_popcount(b) for b in ref["black"]])
    rw = np.array([_popcount(w) for w in ref["white"]])
    assert np.array_equal(ref["winner"], np.where(rb >= rw, 0, 1)) and np.array_equal(ref["draws"], rb == rw)
    duels = arena.duels_between_neural_networks(G, n, HashPriorNet(), HashPriorNet(), 1.0, 4,
                                                rng=np.random.default_rng(6), rules=rules, scoring=STD)
    assert set(duels) <= {0, 1, 2}
    wins = arena.evaluate_neural_network(n, 40, HashPriorNet(), 6, 1.0, rng=np.random.default_rng(1), rules=rules,
                                         scoring=STD, repeats=2)
    assert all(0 <= w <= 40 for w in wins)


def test_arena_moves_replay_under_standard_scoring(E, monkeypatch):
    """pit() with standard scoring plays legal moves under its rule set: every applied move reproduces the oracle's."""
    from othellozero_b200 import arena
    from othellozero_b200 import engine as eng
    from othellozero_b200.mcts import HashPriorNet
    n = 6
    real = eng.apply_moves
    seen = []

    def spy(own, opp, sq, board_size=8, device=0, rules="reference"):
        out = real(own, opp, sq, board_size, device, rules=rules)
        seen.append((np.array(own), np.array(opp), np.array(sq), out))
        return out

    monkeypatch.setattr(arena._e, "apply_moves", spy)
    S = oracle_standard.load()
    arena.pit(n, HashPriorNet(), HashPriorNet(), 6, n_games=6, rng=np.random.default_rng(2), rules=STD, scoring=STD)
    assert seen
    for own, opp, sq, (o2, p2, fl, nl) in seen:
        for i in range(own.size):
            r, c = divmod(int(sq[i]), 8)
            b = S.flip_board(oracle.bits_to_board(int(own[i]), int(opp[i]), n), 0, r, c)
            mover = int(p2[i]) if int(fl[i]) & 1 else int(o2[i])
            assert oracle.board_to_bits(b)[0] == mover


# ---- 6. the game classes -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rules", RULES)
def test_game_class_agrees_with_oracle_on_a_drawn_game(E, rules):
    from othellozero_b200.othello import BoardView, OthelloGame, OthelloPlayer, game_class
    D = oracle_scoring.load(rules)
    n = 6
    cls = game_class(rules, STD)
    g = 0
    while True:
        full = D.playout(n, 77, g)
        if full["finished"] and D.winner(full["board"])[0] == 2:
            break
        g += 1
    game = cls(n)
    for a in full["moves"]:
        assert not game.has_finished()
        game.play(a // n, a % n)
    assert game.has_finished()
    board = game.board(BoardView.TWO_CHANNELS)
    assert np.array_equal(board.astype(np.uint8), full["board"])
    ch, pts = D.winner(full["board"])
    assert ch == 2 and game.get_winning_player() == (None, pts) and cls.get_board_winning_player(board) == (None, pts)
    assert cls.getGameEnded(board) == 1e-4
    assert OthelloGame.getGameEnded(board) == OthelloPlayer.BLACK.value
    assert OthelloGame.get_board_winning_player(board) == (OthelloPlayer.BLACK, pts)
    # not a draw: the winner as before
    won = oracle.bits_to_board(0xF0F, 0x30000, n).astype(bool)
    assert cls.get_board_winning_player(won) == OthelloGame.get_board_winning_player(won) == (OthelloPlayer.BLACK, 8)


# ---- 7. the iteration driver -------------------------------------------------------------------------------------------
def test_iteration_driver_standard_rules_and_scoring():
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "6", "--arena-threshold", "4",
           "--arena-simulations", "8", "--iterations", "2", "--rules", "standard", "--scoring", "standard"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2
    for i, d in enumerate(lines, start=1):
        assert d["config"]["rules"] == "standard" and d["config"]["scoring"] == "standard" and d["iteration"] == i
        assert d["positions_gathered"] >= 12 * 20 and d["selfplay_sims"] == 10 * d["positions_gathered"]
        assert 0 <= d["arena_draws"] and d["arena_new_wins"] + d["arena_draws"] <= 6
        assert d["promoted"] == (d["arena_new_wins"] >= 4)
        assert np.isfinite(np.array(d["train_history"])).all()
