"""Standard search values on the device (a child's value is negated only when the move swapped the side to move), with
and without leaf solving: the search and self-play against the standard-values oracles (tests/oracle_values.py) bit for
bit, Q bit patterns included, under both rule sets and both scorings; virtual-loss waves; the game queue; the evaluation
cache; the error paths; the arena; and the iteration driver.  Roots and starts are positions of seeded random games a few
plies before their end (values only) or a few empties above K (leaf solving), so that passes, finished games and solved
leaves occur inside the searched trees; the tests check that they do."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
import oracle_scoring
import oracle_values
import prior_fns
from gpu_util import canon_board, sq8, visits_to_grid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STD = "standard"
BASES = [(r, s) for r in ("reference", "standard") for s in ("reference", "standard")]
K_OF = {4: 4, 6: 6, 8: 8}


@pytest.fixture(scope="module")
def E():
    from othellozero_b200 import engine
    return engine


def _pass_within(O, board, player, plies):
    """Whether some line of at most `plies` moves from (board, player) contains a pass with the game going on."""
    if plies == 0:
        return False
    for r, c in O.valid_actions(board, player):
        child = O.flip_board(board, player, r, c)
        if O.valid_actions(child, 1 - player):
            if _pass_within(O, child, 1 - player, plies - 1):
                return True
        elif O.valid_actions(child, player):
            return True
    return False


def _starts(rules, n, count, seed, empties=None, back=(2, 8), need_pass=False):
    """Positions of engine-RNG random playouts under `rules`: `back` plies (drawn per game) before the end, or, with
    empties=(lo, hi), the first position of the game with at most hi empties if it has at least lo.  need_pass: only
    positions with a pass within two plies.  -> list of (black, white, player, board)."""
    O = oracle_scoring.load(rules)           # the rules are the same under either scoring
    rng = np.random.default_rng(seed)
    out, g = [], 0
    while len(out) < count:
        full = O.playout(n, seed, g)
        g += 1
        assert g < 20000
        if empties is None:
            k = len(full["moves"]) - int(rng.integers(back[0], back[1] + 1))
        else:
            k = next((i for i in range(len(full["moves"]) + 1)
                      if n * n - int(O.playout(n, seed, g - 1, max_moves=i)["board"].sum()) <= empties[1]), None)
            if k is None:
                continue
        if k < 0:
            continue
        st = O.playout(n, seed, g - 1, max_moves=k)
        if st["finished"] or not O.valid_actions(st["board"], st["player"]):
            continue
        if empties is not None and n * n - int(st["board"].sum()) < empties[0]:
            continue
        if need_pass and not _pass_within(O, st["board"], st["player"], 2):
            continue
        out.append((st["black"], st["white"], st["player"], st["board"]))
    return out


def _passes_below(E, starts, n, rules, plies=3):
    """Moves within `plies` of the starts after which the opponent must pass (the game going on), by the rules API."""
    own = np.array([s[1] if s[2] else s[0] for s in starts], np.uint64)
    opp = np.array([s[0] if s[2] else s[1] for s in starts], np.uint64)
    passes = 0
    for _ in range(plies):
        legal = E.legal_moves(own, opp, n)
        o, p, sq = [], [], []
        for i in range(own.size):
            x = int(legal[i])
            while x:
                b = (x & -x).bit_length() - 1
                x &= x - 1
                o.append(own[i]); p.append(opp[i]); sq.append(b)
        if not sq:
            break
        o2, p2, fl, _ = E.apply_moves(np.array(o, np.uint64), np.array(p, np.uint64), np.array(sq, np.int32), n,
                                      rules=rules)
        passes += int(((fl & 2) != 0).sum())
        live = (fl & 4) == 0
        own, opp = o2[live], p2[live]
    return passes


def _bits(q):
    return np.asarray(q, dtype=np.float64).view(np.int64)


def _search_case(E, rules, scoring, k, prior, n, sims, starts):
    V = oracle_values.load(rules, scoring, k)
    R = oracle_values.load(rules, scoring, 0) if k else None
    solved = terminal = changed = 0
    for black, white, player, board in starts:
        if prior == "hash":
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HASH, rules=rules, scoring=scoring, values=STD, solve_leaves=k)
            m = V.Mcts(n)
            predict_batch = None
        else:
            def predict_batch(own, opp):
                outs = [prior_fns.sha_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
                return np.stack([o[0].ravel() for o in outs]), np.array([o[1] for o in outs], dtype=np.float32)
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HOST, rules=rules, scoring=scoring, values=STD, solve_leaves=k)
            m = V.Mcts(n, predict=prior_fns.sha_prior)
        e.reset(1, [black], [white], [player])
        e.search(sims, predict_batch)
        v, ns = e.visits()
        q, p, tag = e.root_stats(0)
        c, sc = e.counters(), e.solve_counters()
        e.close()
        terminal += c["terminal_visits"]
        solved += sc["solved_leaves"]
        assert sc["solved_leaves"] <= c["terminal_visits"] and (sc["solver_nodes"] > sc["solved_leaves"]) == bool(sc["solved_leaves"])
        for _ in range(sims):
            m.simulate(board, player)
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
        if R is not None:   # leaf solving changes the search
            r = R.Mcts(n, predict=None if prior == "hash" else prior_fns.sha_prior)
            for _ in range(sims):
                r.simulate(board, player)
            changed += r.visits(canon)[1].tolist() != rv.tolist()
    return solved, terminal, changed


# ---- 1. sequential search against the standard-values oracle ---------------------------------------------------------
@pytest.mark.parametrize("rules,scoring", BASES)
@pytest.mark.parametrize("prior", ["hash", "host"])
@pytest.mark.parametrize("n", [4, 6, 8])
def test_search_standard_values_equals_oracle(E, rules, scoring, prior, n):
    sims = {4: 40, 6: 100, 8: 160}[n]
    starts = _starts(rules, n, 4, seed=100 + n + (prior == "host"), back=(3, 10), need_pass=True)
    _, terminal, _ = _search_case(E, rules, scoring, 0, prior, n, sims, starts)
    assert terminal > 0
    assert _passes_below(E, starts, n, rules) > 0


@pytest.mark.parametrize("rules", ["reference", "standard"])
@pytest.mark.parametrize("prior", ["hash", "host"])
@pytest.mark.parametrize("n,k", [(4, 4), (6, 4), (6, 6), (8, 4), (8, 6), (8, 8)])
def test_search_with_solved_leaves_equals_oracle(E, rules, prior, n, k):
    sims = {4: 40, 6: 100, 8: 160}[n]
    starts = _starts(rules, n, 3, seed=200 + 10 * n + k, empties=(k + 2, k + 5))
    solved, _, changed = _search_case(E, rules, STD, k, prior, n, sims, starts)
    assert solved > 0 and changed > 0


# ---- 2. self-play against the oracle's episode driver --------------------------------------------------------------------
@pytest.mark.parametrize("solve", [False, True])
@pytest.mark.parametrize("n,sims,T,eg", [(4, 12, 1.0, 0.8), (4, 6, 0.0, 0.9), (6, 16, 1.0, 0.9), (6, 8, 0.0, 0.9),
                                         (8, 20, 1.0, 0.9), (8, 8, 0.0, 0.9)])
def test_selfplay_hash_prior_equals_oracle(E, solve, n, sims, T, eg):
    rules, scoring, k = ("standard", STD, K_OF[n]) if solve else ("reference", "reference", 0)
    V = oracle_values.load(rules, scoring, k)
    starts = _starts(rules, n, 10, seed=30 + n, back=(4, 16))
    G, slots = len(starts), 4                                    # more games than slots: the device queue is used
    black = [s[0] for s in starts]; white = [s[1] for s in starts]; player = [s[2] for s in starts]
    ids = [900 + g for g in range(G)]
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=13, log_visits=True, rules=rules, scoring=scoring,
                 values=STD, solve_leaves=k)
    e.selfplay_begin(G, sims, T, eg, -1, black, white, player, ids)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    sc = e.solve_counters()
    e.close()
    assert (sc["solved_leaves"] > 0) == solve
    for g in range(G):
        ref = V.execute_episode(n, sims, temperature=T, e_greedy=eg, seed=13, game_id=ids[g], start_board=starts[g][3],
                                start_player=player[g], log_visits=True)
        kk = int(out["n_moves"][g])
        assert [int(a) for a in out["action"][g][:kk]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert [int(x) for x in out["black"][g][:kk]] == ref["black"] and [int(x) for x in out["white"][g][:kk]] == ref["white"]
        assert int(out["winner"][g]) == ref["winner"], g
        for p in range(kk):
            assert visits_to_grid(out["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)


def _net_predict(E, n, blob, C):
    from othellozero_b200 import net as oznet
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
    return f, predict


@pytest.mark.parametrize("solve", [False, True])
@pytest.mark.parametrize("n", [6, 8])
def test_selfplay_network_equals_oracle_fed_device_priors(E, solve, n):
    from othellozero_b200 import net as oznet
    rules, scoring, k = ("standard", STD, K_OF[n]) if solve else ("standard", "reference", 0)
    V = oracle_values.load(rules, scoring, k)
    C, sims, slots = 128, 24, 4
    blob = oznet.init_weights(n, C, seed=8, randomize_bn=True)
    starts = _starts(rules, n, 8, seed=50 + n, back=(4, 14))
    black = np.array([s[0] for s in starts], dtype=np.uint64)
    white = np.array([s[1] for s in starts], dtype=np.uint64)
    player = np.array([s[2] for s in starts], dtype=np.int32)
    games = len(starts)
    ids = np.arange(40, 40 + games, dtype=np.uint64)
    e = E.Engine(n, slots, sims * 12 + 64, E.PRIOR_NET, seed=2, log_visits=True, eval_cache_log2=14, rules=rules,
                 scoring=scoring, values=STD, solve_leaves=k)
    e.load_weights(blob, C)
    e.selfplay_begin(games, sims, 1.0, 0.9, -1, black, white, player, ids)
    assert e.selfplay_run(-1) == 0
    rec = e.selfplay_records()
    assert (e.solve_counters()["solved_leaves"] > 0) == solve
    e.close()
    f, predict = _net_predict(E, n, blob, C)
    for g in range(games):
        ref = V.execute_episode(n, sims, temperature=1.0, e_greedy=0.9, predict=predict, seed=2, game_id=int(ids[g]),
                                start_board=starts[g][3], start_player=int(player[g]), log_visits=True)
        kk = int(rec["n_moves"][g])
        assert [int(a) for a in rec["action"][g][:kk]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert int(rec["winner"][g]) == ref["winner"], g
        for p in range(kk):
            assert visits_to_grid(rec["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    f.close()


# ---- 3. virtual-loss waves ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 8])
def test_wave_search_conserves_visits_and_ignores_the_prior_source(E, k):
    sims, V, n = 203, 4, 8
    roots = _starts(STD, n, 3, seed=9 + k, empties=(k + 3, k + 8))

    def host_hash(own, opp):   # the closed-form hash prior, evaluated on the host
        outs = [oracle.hash_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
        return np.stack([np.asarray(o[0], np.float32).ravel() for o in outs]), np.array([o[1] for o in outs], np.float32)

    outs = []
    for mode in (E.PRIOR_HASH, E.PRIOR_HASH, E.PRIOR_HOST):
        e = E.Engine(n, 3, sims + 16, mode, vl_width=V, rules=STD, scoring=STD, values=STD, solve_leaves=k)
        e.reset(3, [r[0] for r in roots], [r[1] for r in roots], [r[2] for r in roots])
        cb = host_hash if mode == E.PRIOR_HOST else None
        e.search(sims, cb)
        v, ns = e.visits()
        assert (ns == sims - 1).all() and (v.sum(axis=1) == ns).all()   # visits conserved, no virtual loss left
        e.search(50, cb)
        v2, ns2 = e.visits()
        assert (ns2 == sims + 49).all() and (v2.sum(axis=1) == ns2).all()
        assert e.counters()["terminal_visits"] > 0
        assert (e.solve_counters()["solved_leaves"] > 0) == (k > 0)
        outs.append(v2.copy())
        e.close()
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


def _net_selfplay(E, n, C, blob, starts, sims, slots, k, cache, vl=1):
    black = np.array([s[0] for s in starts], dtype=np.uint64)
    white = np.array([s[1] for s in starts], dtype=np.uint64)
    player = np.array([s[2] for s in starts], dtype=np.int32)
    e = E.Engine(n, slots, sims * 40 + 64, E.PRIOR_NET, seed=3, vl_width=vl, eval_cache_log2=cache, rules=STD,
                 scoring=STD, values=STD, solve_leaves=k)
    e.load_weights(blob, C)
    e.selfplay_begin(len(starts), sims, 1.0, 0.9, -1, black, white, player, np.arange(len(starts), dtype=np.uint64))
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    e.close()
    return out


@pytest.mark.parametrize("vl", [1, 4])
def test_selfplay_is_deterministic_cache_and_queue_independent(E, vl):
    from othellozero_b200 import net as oznet
    n, C, sims, k = 6, 128, 16, 6
    blob = oznet.init_weights(n, C, seed=4, randomize_bn=True)
    starts = _starts(STD, n, 12, seed=61, back=(4, 14))
    outs = [_net_selfplay(E, n, C, blob, starts, sims, 5, k, cache, vl) for cache in (14, 14, 0)]
    if vl == 1:   # the game queue: 12 games through 5 slots equal 12 games in 12 slots
        outs.append(_net_selfplay(E, n, C, blob, starts, sims, 12, k, 14, vl))
    ref = outs[0]
    for o in outs[1:]:
        assert np.array_equal(ref["n_moves"], o["n_moves"]) and np.array_equal(ref["winner"], o["winner"])
        for g, m in enumerate(ref["n_moves"]):   # entries past a game's end (row n_moves holds the final position)
            m = int(m)
            assert np.array_equal(ref["action"][g][:m], o["action"][g][:m]), g
            for key in ("black", "white"):
                assert np.array_equal(ref[key][g][:m + 1], o[key][g][:m + 1]), (key, g)
    assert set(int(w) for w in ref["winner"]) <= {0, 1, 2}


# ---- 4. error paths -------------------------------------------------------------------------------------------------------
def test_set_values_errors_and_latching(E):
    from othellozero_b200 import _lib
    L = _lib.load()
    e = E.Engine(6, 2, 256, E.PRIOR_HASH, scoring="reference")
    h = e._h
    assert L.oz_search_set_values(h, 2, 0) == _lib.OZ_ERR_INVALID
    assert L.oz_search_set_values(h, 1, 13) == _lib.OZ_ERR_INVALID and "solve_leaves" in L.oz_last_error().decode()
    assert L.oz_search_set_values(h, 1, -1) == _lib.OZ_ERR_INVALID
    assert L.oz_search_set_values(h, 1, 4) == _lib.OZ_ERR_INVALID and "scoring" in L.oz_last_error().decode()
    assert L.oz_search_set_values(h, 0, 0) == 0 and L.oz_search_set_values(h, 1, 0) == 0
    e.close()
    f = E.Engine(6, 2, 256, E.PRIOR_HASH, scoring=STD)
    assert L.oz_search_set_values(f._h, 0, 4) == _lib.OZ_ERR_INVALID
    # latched by the next reset: requested after a reset, the search still runs with the values of that reset
    start = _starts(STD, 6, 2, seed=77, empties=(8, 10))
    f.reset(2, [s[0] for s in start], [s[1] for s in start], [s[2] for s in start])
    assert L.oz_search_set_values(f._h, 1, 6) == 0
    f.search(60)
    assert f.solve_counters() == {"solved_leaves": 0, "solver_nodes": 0}
    f.reset(2, [s[0] for s in start], [s[1] for s in start], [s[2] for s in start])
    f.search(60)
    assert f.solve_counters()["solved_leaves"] > 0
    f.close()


# ---- 5. the arena ---------------------------------------------------------------------------------------------------------
def test_arena_with_standard_values(E):
    from othellozero_b200 import arena
    from othellozero_b200.mcts import HashPriorNet
    n, G = 6, 48
    out = arena.pit(n, HashPriorNet(), HashPriorNet(), 16, n_games=G, rng=np.random.default_rng(5), rules=STD,
                    scoring=STD, values=(STD, "reference"), solve_leaves=(6, 0))
    assert out["winner"].shape == (G,) and set(int(w) for w in out["winner"]) <= {0, 1, 2}
    again = arena.pit(n, HashPriorNet(), HashPriorNet(), 16, n_games=G, rng=np.random.default_rng(5), rules=STD,
                      scoring=STD, values=(STD, "reference"), solve_leaves=(6, 0))
    assert np.array_equal(out["winner"], again["winner"]) and np.array_equal(out["black"], again["black"])
    ref = arena.pit(n, HashPriorNet(), HashPriorNet(), 16, n_games=G, rng=np.random.default_rng(5), rules=STD,
                    scoring=STD)
    assert not np.array_equal(ref["black"], out["black"])          # the searches play differently
    duels = arena.duels_between_neural_networks(8, n, HashPriorNet(), HashPriorNet(), 1.0, 8,
                                                rng=np.random.default_rng(6), rules=STD, scoring=STD, values=STD,
                                                solve_leaves=8)
    assert set(duels) <= {0, 1, 2}
    wins = arena.evaluate_neural_network(n, 10, HashPriorNet(), 8, 1.0, rng=np.random.default_rng(1), values=STD)
    assert 0 <= wins <= 10


# ---- 6. the iteration driver ----------------------------------------------------------------------------------------------
def test_iteration_driver_standard_values_and_solved_leaves():
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "6", "--arena-threshold", "4",
           "--arena-simulations", "8", "--iterations", "1", "--rules", "standard", "--scoring", "standard",
           "--values", "standard", "--solve-leaves", "8"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = lines[0]
    assert d["config"]["values"] == "standard" and d["config"]["solve_leaves"] == 8 and d["iteration"] == 1
    assert d["positions_gathered"] >= 12 * 20 and d["selfplay_sims"] == 10 * d["positions_gathered"]
    assert d["arena_new_wins"] + d["arena_draws"] <= 6
