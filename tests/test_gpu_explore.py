"""Root exploration on the device: Dirichlet noise on each root's priors (once per node) and self-play opening moves drawn
in proportion to the root visit counts, against the exploring oracles (tests/oracle_explore.py) bit for bit - root
priors, Q bit patterns and visit counts of the search, records, winners and visit logs of self-play - over the
reference base and the standard rules/scoring/values base; noise applied once; independence from the game queue, the
evaluation cache and leaf solving; virtual-loss waves; game diversity from the initial position; error paths and
latching; the Python entry points and the iteration driver."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
import oracle_explore
import prior_fns
from gpu_util import canon_board, sq8, visits_to_grid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STD = "standard"
BASES = {"reference": ("reference", "reference", "reference"), "standard": (STD, STD, STD)}


@pytest.fixture(scope="module")
def E():
    from othellozero_b200 import engine
    return engine


def _oracle(base):
    X = oracle_explore.load(*BASES[base])
    X.build()
    return X


def _kw(base):
    r, s, v = BASES[base]
    return dict(rules=r, scoring=s, values=v)


def _starts(n, count, seed, plies=(2, 12)):
    """Positions of engine-RNG random playouts `plies` moves in, side to move able to move (reference rules: the
    standard base only needs positions, which both rule sets share this early)."""
    rng = np.random.default_rng(seed)
    out, g = [], 0
    while len(out) < count:
        st = oracle.playout(n, seed, g, max_moves=int(rng.integers(plies[0], plies[1] + 1)))
        g += 1
        if st["finished"] or not oracle.valid_actions(st["board"], st["player"]):
            continue
        out.append((st["black"], st["white"], st["player"], st["board"]))
    return out


def _bits(q):
    return np.asarray(q, dtype=np.float64).view(np.int64)


def _host_predict(n):
    def predict_batch(own, opp):
        outs = [prior_fns.sha_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
        return np.stack([o[0].ravel() for o in outs]), np.array([o[1] for o in outs], dtype=np.float32)
    return predict_batch


def _compare_root(e, m, board, player, n, tag=""):
    v, ns = e.visits()
    q, p, t = e.root_stats(0)
    canon = board if player == 0 else board[..., ::-1]
    rns, rv = m.visits(canon)
    assert int(ns[0]) == rns and visits_to_grid(v[0], n).tolist() == rv.reshape(-1).tolist(), tag
    rq, rp, rt = m.node_stats(canon)
    for r in range(n):
        for c in range(n):
            s = r * 8 + c
            assert p[s] == rp[r, c], (tag, s)           # the (noised) priors of every square
            if rt[r, c] >= 0:
                assert _bits(q[s]) == _bits(rq[r, c]) and t[s] == rt[r, c], (tag, s)
    return rp


# ---- 1. the search API against the exploring oracle, bit for bit -------------------------------------------------------
@pytest.mark.parametrize("base", ["reference", "standard"])
@pytest.mark.parametrize("prior", ["hash", "host"])
@pytest.mark.parametrize("n", [6, 8])
@pytest.mark.parametrize("alpha", [0.3, 2.5])
def test_search_root_noise_equals_oracle(E, base, prior, n, alpha):
    X = _oracle(base)
    sims, eps, seed = {6: 80, 8: 120}[n], 0.25, 7
    X.set_explore(alpha, eps, 0)
    mode = E.PRIOR_HASH if prior == "hash" else E.PRIOR_HOST
    cb = _host_predict(n) if prior == "host" else None
    changed = 0
    for i, (black, white, player, board) in enumerate(_starts(n, 3, seed=20 + n)):
        gid = 100 + i
        e = E.Engine(n, 1, 4 * sims, mode, seed=seed, dirichlet_alpha=alpha, dirichlet_fraction=eps, **_kw(base))
        e.reset(1, [black], [white], [player], [gid])
        e.search(sims, cb)
        m = X.Mcts(n, predict=None if prior == "hash" else prior_fns.sha_prior)
        X.mcts_explore_key(m, seed, gid)
        for _ in range(sims):
            m.simulate(board, player)
        rp = _compare_root(e, m, board, player, n, (base, prior, i))
        e.close()
        # the noise moved the priors away from the network's
        X.set_explore(0.0, 0.0, 0)
        m0 = X.Mcts(n, predict=None if prior == "hash" else prior_fns.sha_prior)
        m0.simulate(board, player)
        X.set_explore(alpha, eps, 0)
        canon = board if player == 0 else board[..., ::-1]
        changed += not np.array_equal(m0.node_stats(canon)[1], rp)
        assert abs(rp.sum() - 1.0) < 1e-12
    X.set_explore(0.0, 0.0, 0)
    assert changed == 3


# ---- 2. noise only once ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prior", ["hash", "host"])
def test_noise_is_applied_once_per_node(E, prior):
    n, alpha, eps, seed = 8, 0.5, 0.4, 3
    X = _oracle("reference")
    X.set_explore(alpha, eps, 0)
    mode = E.PRIOR_HASH if prior == "hash" else E.PRIOR_HOST
    cb = _host_predict(n) if prior == "host" else None
    pred = None if prior == "hash" else prior_fns.sha_prior
    black, white, player, board = _starts(n, 1, seed=5)[0]
    # (a) begin twice on one root equals one search of the sum
    e = E.Engine(n, 1, 1024, mode, seed=seed, dirichlet_alpha=alpha, dirichlet_fraction=eps)
    e.reset(1, [black], [white], [player], [9])
    e.search(40, cb)
    e.search(35, cb)
    m = X.Mcts(n, predict=pred)
    X.mcts_explore_key(m, seed, 9)
    for _ in range(75):
        m.simulate(board, player)
    _compare_root(e, m, board, player, n, "twice")
    # (b) set_roots to a child and back: the child is noised when it becomes a root, the old root is not noised again
    r, c = oracle.valid_actions(board, player)[0]
    child = oracle.flip_board(board, player, r, c)
    cplayer = 1 - player if oracle.valid_actions(child, 1 - player) else player
    cb_, cw_ = oracle.board_to_bits(child)
    e.set_roots([cb_], [cw_], [cplayer])
    e.search(30, cb)
    for _ in range(30):
        m.simulate(child, cplayer)
    _compare_root(e, m, child, cplayer, n, "child")
    e.set_roots([black], [white], [player])
    e.search(30, cb)
    for _ in range(30):
        m.simulate(board, player)
    _compare_root(e, m, board, player, n, "back")
    e.close()
    X.set_explore(0.0, 0.0, 0)


# ---- 3. self-play against the oracle's episode driver --------------------------------------------------------------------
MODES = {"noise": (0.3, 0.25, 0), "sampled": (0.0, 0.25, 12), "both": (1.5, 0.4, 20)}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("base", ["reference", "standard"])
@pytest.mark.parametrize("n,sims,T,eg", [(6, 16, 1.0, 0.9), (6, 8, 0.0, 1.0), (8, 16, 1.0, 1.0), (8, 8, 0.0, 0.9)])
def test_selfplay_hash_prior_equals_oracle(E, mode, base, n, sims, T, eg):
    alpha, eps, M = MODES[mode]
    X = _oracle(base)
    X.set_explore(alpha, eps, M)
    G, slots, seed = 10, 4, 13       # more games than slots: the device queue is used
    starts = _starts(n, G - 4, seed=40 + n, plies=(1, 8))
    black = [s[0] for s in starts] + [None] * 4
    ids = [700 + g for g in range(G)]
    ib, iw = oracle.board_to_bits(oracle.initial_board(n))
    bl = [b if b is not None else ib for b in black]
    wh = [s[1] for s in starts] + [iw] * 4
    pl = [s[2] for s in starts] + [0] * 4
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=seed, log_visits=True, dirichlet_alpha=alpha,
                 dirichlet_fraction=eps, sample_moves=M, **_kw(base))
    e.selfplay_begin(G, sims, T, eg, -1, bl, wh, pl, ids)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    e.close()
    boards = [s[3] for s in starts] + [oracle.initial_board(n)] * 4
    for g in range(G):
        ref = X.execute_episode(n, sims, temperature=T, e_greedy=eg, seed=seed, game_id=ids[g], start_board=boards[g],
                                start_player=pl[g], log_visits=True)
        kk = int(out["n_moves"][g])
        assert [int(a) for a in out["action"][g][:kk]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert [int(x) for x in out["black"][g][:kk]] == ref["black"] and [int(x) for x in out["white"][g][:kk]] == ref["white"]
        assert int(out["winner"][g]) == ref["winner"], g
        for p in range(kk):
            assert visits_to_grid(out["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    X.set_explore(0.0, 0.0, 0)
    # the same games without exploration play differently
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=seed, **_kw(base))
    e.selfplay_begin(G, sims, T, eg, -1, bl, wh, pl, ids)
    assert e.selfplay_run(-1) == 0
    plain = e.selfplay_records()
    e.close()
    assert not np.array_equal(plain["action"], out["action"])


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


@pytest.mark.parametrize("n", [6, 8])
def test_selfplay_network_equals_oracle_fed_device_priors(E, n):
    from othellozero_b200 import net as oznet
    base = "standard" if n == 8 else "reference"
    alpha, eps, M = 0.5, 0.25, 10
    X = _oracle(base)
    C, sims, slots, seed = 128, 24, 4, 2
    blob = oznet.init_weights(n, C, seed=8, randomize_bn=True)
    games = 8
    ids = np.arange(40, 40 + games, dtype=np.uint64)
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_NET, seed=seed, log_visits=True, eval_cache_log2=14,
                 dirichlet_alpha=alpha, dirichlet_fraction=eps, sample_moves=M, **_kw(base))
    e.load_weights(blob, C)
    e.selfplay_begin(games, sims, 1.0, 0.9, -1, None, None, None, ids)
    assert e.selfplay_run(-1) == 0
    rec = e.selfplay_records()
    e.close()
    f, predict = _net_predict(E, n, blob, C)
    X.set_explore(alpha, eps, M)
    for g in range(games):
        ref = X.execute_episode(n, sims, temperature=1.0, e_greedy=0.9, predict=predict, seed=seed, game_id=int(ids[g]),
                                log_visits=True)
        kk = int(rec["n_moves"][g])
        assert [int(a) for a in rec["action"][g][:kk]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert int(rec["winner"][g]) == ref["winner"], g
        for p in range(kk):
            assert visits_to_grid(rec["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    X.set_explore(0.0, 0.0, 0)
    f.close()


# ---- 4. independence from the queue, the evaluation cache and leaf solving -----------------------------------------------
def _same_records(a, b):
    assert np.array_equal(a["n_moves"], b["n_moves"]) and np.array_equal(a["winner"], b["winner"])
    for g, m in enumerate(a["n_moves"]):
        m = int(m)
        assert np.array_equal(a["action"][g][:m], b["action"][g][:m]), g
        for key in ("black", "white"):
            assert np.array_equal(a[key][g][:m + 1], b[key][g][:m + 1]), (key, g)


def test_hash_selfplay_queue_independent(E):
    # 8192 games from the initial position with e_greedy = 1 through 2048 slots or all at once: the same games
    n, sims, G = 6, 8, 8192
    outs = {}
    for key, slots in (("q", 2048), ("all", G)):
        e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=21, dirichlet_alpha=0.3, sample_moves=4)
        e.selfplay_begin(G, sims, 1.0, 1.0)
        assert e.selfplay_run(-1) == 0
        outs[key] = e.selfplay_records()
        e.close()
    _same_records(outs["q"], outs["all"])
    assert len({bytes(outs["q"]["action"][g][:int(outs["q"]["n_moves"][g])]) for g in range(G)}) > 1


def test_root_noise_diversifies_games_from_the_initial_position(E):
    # 4096 games from the initial position with e_greedy = 1 (no random moves): without exploration they are one game,
    # with root noise nearly every game is its own
    n, sims, G = 8, 16, 4096
    distinct = {}
    for alpha in (0.0, 0.3):
        e = E.Engine(n, G, sims * 61 + 64, E.PRIOR_HASH, seed=21, dirichlet_alpha=alpha)
        e.selfplay_begin(G, sims, 1.0, 1.0)
        assert e.selfplay_run(-1) == 0
        rec = e.selfplay_records()
        e.close()
        distinct[alpha] = len({bytes(rec["action"][g][:int(rec["n_moves"][g])]) for g in range(G)})
    assert distinct[0.0] == 1
    assert distinct[0.3] > 0.9 * G, distinct


@pytest.mark.parametrize("k", [0, 6])
def test_net_selfplay_cache_queue_and_solver_independent(E, k):
    from othellozero_b200 import net as oznet
    n, C, sims, G = 6, 128, 16, 24
    blob = oznet.init_weights(n, C, seed=4, randomize_bn=True)
    kw = dict(rules=STD, scoring=STD, values=STD, solve_leaves=k) if k else {}

    def run(slots, cache):
        e = E.Engine(n, slots, sims * 40 + 64, E.PRIOR_NET, seed=3, eval_cache_log2=cache, dirichlet_alpha=0.3,
                     dirichlet_fraction=0.25, sample_moves=8, **kw)
        e.load_weights(blob, C)
        e.selfplay_begin(G, sims, 1.0, 1.0, -1, None, None, None, np.arange(G, dtype=np.uint64))
        assert e.selfplay_run(-1) == 0
        out = e.selfplay_records()
        if k:
            assert e.solve_counters()["solved_leaves"] > 0
        e.close()
        return out
    ref = run(5, 14)
    for slots, cache in ((5, 14), (5, 0), (G, 14), (G, 0)):
        _same_records(ref, run(slots, cache))
    assert len({bytes(ref["action"][g][:int(ref["n_moves"][g])]) for g in range(G)}) == G


# ---- 5. virtual-loss waves ---------------------------------------------------------------------------------------------
def test_wave_search_with_noise_is_deterministic_and_conserves_visits(E):
    sims, V, n = 203, 4, 8
    roots = _starts(n, 3, seed=9)

    def host_hash(own, opp):
        outs = [oracle.hash_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
        return np.stack([np.asarray(o[0], np.float32).ravel() for o in outs]), np.array([o[1] for o in outs], np.float32)

    outs = []
    for mode in (E.PRIOR_HASH, E.PRIOR_HASH, E.PRIOR_HOST):
        e = E.Engine(n, 3, sims + 16, mode, vl_width=V, dirichlet_alpha=0.3, dirichlet_fraction=0.25)
        e.reset(3, [r[0] for r in roots], [r[1] for r in roots], [r[2] for r in roots])
        cb = host_hash if mode == E.PRIOR_HOST else None
        e.search(sims, cb)
        v, ns = e.visits()
        assert (ns == sims - 1).all() and (v.sum(axis=1) == ns).all()
        e.search(50, cb)
        v2, ns2 = e.visits()
        assert (ns2 == sims + 49).all() and (v2.sum(axis=1) == ns2).all()
        outs.append((v2.copy(), e.root_stats(0)[1].copy()))
        e.close()
    assert all(np.array_equal(outs[0][0], o[0]) and np.array_equal(outs[0][1], o[1]) for o in outs[1:])
    e = E.Engine(n, 3, sims + 16, E.PRIOR_HASH, vl_width=V)
    e.reset(3, [r[0] for r in roots], [r[1] for r in roots], [r[2] for r in roots])
    e.search(sims + 50)
    assert not np.array_equal(e.root_stats(0)[1], outs[0][1])   # the noise is in the wave search's root priors
    e.close()


# ---- 6. errors and latching --------------------------------------------------------------------------------------------
def test_set_exploration_errors_and_latching(E):
    from othellozero_b200 import _lib
    L = _lib.load()
    n = 6
    e = E.Engine(n, 1, 512, E.PRIOR_HASH, seed=1)
    h = e._h
    for a, f, m in ((-0.1, 0.25, 0), (float("nan"), 0.25, 0), (float("inf"), 0.25, 0), (0.3, 1.01, 0), (0.3, -0.5, 0),
                    (0.3, float("nan"), 0), (0.3, 0.25, 65), (0.3, 0.25, -1)):
        assert L.oz_search_set_exploration(h, a, f, m) == _lib.OZ_ERR_INVALID, (a, f, m)
    assert L.oz_search_set_exploration(None, 0.3, 0.25, 0) == _lib.OZ_ERR_INVALID
    assert L.oz_search_set_exploration(h, 0.3, 0.25, 99) == _lib.OZ_ERR_INVALID
    assert "sample_moves" in L.oz_last_error().decode()
    black, white, player, board = _starts(n, 1, seed=3)[0]
    X = _oracle("reference")
    # requested after a reset: the search still runs without noise, the next reset latches it
    e.reset(1, [black], [white], [player], [4])
    assert L.oz_search_set_exploration(h, 0.3, 0.5, 0) == 0
    e.search(40)
    X.set_explore(0.0, 0.0, 0)
    m = X.Mcts(n)
    for _ in range(40):
        m.simulate(board, player)
    _compare_root(e, m, board, player, n, "not latched")
    e.reset(1, [black], [white], [player], [4])
    e.search(40)
    X.set_explore(0.3, 0.5, 0)
    m = X.Mcts(n)
    X.mcts_explore_key(m, 1, 4)
    for _ in range(40):
        m.simulate(board, player)
    _compare_root(e, m, board, player, n, "latched")
    X.set_explore(0.0, 0.0, 0)
    # sample_moves alone does not change the search API
    assert L.oz_search_set_exploration(h, 0.0, 0.25, 30) == 0
    e.reset(1, [black], [white], [player], [4])
    e.search(40)
    m = X.Mcts(n)
    for _ in range(40):
        m.simulate(board, player)
    _compare_root(e, m, board, player, n, "sample_moves only")
    e.close()
    with pytest.raises(ValueError):
        E.Engine(n, 1, 64, E.PRIOR_HASH, dirichlet_alpha=-1.0)


# ---- 7. the Python entry points and the iteration driver ---------------------------------------------------------------
def test_python_entry_points(E):
    from othellozero_b200 import selfplay
    from othellozero_b200.mcts import HashPriorNet, OthelloMCTS
    n = 6
    kw = dict(seed=5, game_ids=np.arange(16, dtype=np.uint64))
    a = selfplay.execute_episodes(16, n, HashPriorNet(), 1.0, 10, 1.0, 1.0, dirichlet_alpha=0.3, sample_moves=6, **kw)
    b = selfplay.execute_episodes(16, n, HashPriorNet(), 1.0, 10, 1.0, 1.0, dirichlet_alpha=0.3, sample_moves=6, **kw)
    c = selfplay.execute_episodes(16, n, HashPriorNet(), 1.0, 10, 1.0, 1.0, **kw)
    key = [[int(np.argmax(p)) for _, p, _ in ex] for ex in a]
    assert key == [[int(np.argmax(p)) for _, p, _ in ex] for ex in b]
    assert key != [[int(np.argmax(p)) for _, p, _ in ex] for ex in c]
    assert len({tuple(k) for k in key}) > 1 and len({tuple([int(np.argmax(p)) for _, p, _ in ex]) for ex in c}) == 1
    W = selfplay.make_b200_worker(seed=5, dirichlet_alpha=0.3, sample_moves=6)
    w = W()
    assert w.explore_kw == dict(dirichlet_alpha=0.3, dirichlet_fraction=0.25, sample_moves=6)
    # OthelloMCTS: with an explicit (seed, game id) the root's priors carry the noise of (seed, game id, root), the
    # oracle's too; by default every instance has a stream of its own, so two instances noise the same root differently
    X = _oracle("reference")
    X.set_explore(0.3, 0.25, 0)
    board = oracle.initial_board(n)
    from othellozero_b200.othello import OthelloPlayer

    def root_priors(**kw):
        mc = OthelloMCTS(n, HashPriorNet(), 1.0, dirichlet_alpha=0.3, **kw)
        mc.simulate(board, OthelloPlayer.BLACK, num_simulations=30)
        return mc, mc._eng.root_stats(0)[1].copy()

    mc, p_fixed = root_priors(seed=11, game_id=3)
    m = X.Mcts(n)
    X.mcts_explore_key(m, 11, 3)
    for _ in range(30):
        m.simulate(board, 0)
    _compare_root(mc._eng, m, board, 0, n, "OthelloMCTS")
    assert np.array_equal(root_priors(seed=11, game_id=3)[1], p_fixed)
    (a, pa), (b, pb) = root_priors(), root_priors()
    assert a.seed == b.seed and a.game_id != b.game_id
    assert not np.array_equal(pa, pb) and not np.array_equal(pa, p_fixed)
    X.set_explore(0.0, 0.0, 0)


# ---- 8. roots with more than 32 legal moves: the second half of every warp-wide step ---------------------------------
WIDE = (0x2881040210fc2402, 0x404e022460024a00)   # black to move, 34 legal moves (8x8)


def test_roots_with_more_than_32_moves_equal_oracle(E):
    n, own, opp = 8, WIDE[0], WIDE[1]
    board = oracle.bits_to_board(own, opp, n)
    legal = [r * 8 + c for r, c in oracle.valid_actions(board, 0)]
    assert len(legal) == 34
    X = _oracle("reference")
    # the search: noise drawn by lanes l and l + 32
    X.set_explore(0.3, 0.25, 0)
    e = E.Engine(n, 1, 2048, E.PRIOR_HASH, seed=4, dirichlet_alpha=0.3, dirichlet_fraction=0.25)
    e.reset(1, [own], [opp], [0], [5])
    e.search(400)
    m = X.Mcts(n)
    X.mcts_explore_key(m, 4, 5)
    for _ in range(400):
        m.simulate(board, 0)
    _compare_root(e, m, board, 0, n, "wide search")
    e.close()
    # self-play: the first move sampled from 34 visit counts (the second prefix-sum half and the second ballot)
    G, sims = 64, 60
    X.set_explore(0.3, 0.25, 1)
    ids = list(range(300, 300 + G))
    e = E.Engine(n, 16, sims * 4 + 64, E.PRIOR_HASH, seed=4, log_visits=True, dirichlet_alpha=0.3,
                 dirichlet_fraction=0.25, sample_moves=1)
    e.selfplay_begin(G, sims, 1.0, 1.0, 1, [own] * G, [opp] * G, [0] * G, ids)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    e.close()
    slots = []
    for g in range(G):
        ref = X.execute_episode(n, sims, temperature=1.0, e_greedy=1.0, seed=4, game_id=ids[g], start_board=board,
                                start_player=0, max_moves=1, log_visits=True)
        assert int(out["n_moves"][g]) == 1 and int(out["action"][g][0]) == sq8(ref["moves"][0], n), g
        assert visits_to_grid(out["visits"][g][0], n).tolist() == ref["visits"][0].tolist(), g
        slots.append(legal.index(int(out["action"][g][0])))
    X.set_explore(0.0, 0.0, 0)
    assert max(slots) >= 32, slots          # some draw landed past the first 32 children


def _driver(*flags):
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "6", "--arena-threshold", "4",
           "--arena-simulations", "8", "--iterations", "1", "--e-greedy", "1.0", *flags]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and lines[0]["iteration"] == 1
    return lines[0]


def test_iteration_driver_forwards_exploration_to_selfplay():
    # e_greedy = 1: without exploration the 12 episodes are one game; each flag reaches self-play on its own
    assert _driver()["selfplay_distinct_games"] == 1
    d = _driver("--dirichlet-alpha", "0.3")
    assert d["config"]["dirichlet_alpha"] == 0.3 and d["selfplay_distinct_games"] > 1
    assert d["positions_gathered"] >= 12 * 20 and d["selfplay_sims"] == 10 * d["positions_gathered"]
    assert _driver("--dirichlet-alpha", "0.3", "--dirichlet-fraction", "0")["selfplay_distinct_games"] == 1
    assert _driver("--sample-moves", "8")["selfplay_distinct_games"] > 1
