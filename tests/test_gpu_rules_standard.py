"""Standard Othello rules on the device: the rules kernels against the host bitboard forms, a level-by-level perft through
the batched rules API, perft playouts, the search and self-play against the oracle's standard-rule restatement, virtual
loss waves, the arena, the OthelloGame façade and the iteration driver.  The two rule sets first differ at ply 7, so
every comparison reaches it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
import oracle_standard
import prior_fns
from gpu_util import canon_board, sq8, visits_to_grid
from rules_util import golden_positions, host_play, lib, random_positions, standard_playout_positions

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STD = "standard"
S = oracle_standard.load()   # the oracle under standard rules (same API as `oracle`)


@pytest.fixture(scope="module")
def E():
    from othellozero_b200 import engine
    return engine


@pytest.fixture(scope="module")
def L():
    return lib()


def _popcount(x):
    return bin(int(x)).count("1")


def _replay_records(L, rec, n):
    """Every recorded move is legal under the host standard rules and leads to the next recorded position."""
    for g in range(len(rec["n_moves"])):
        k = int(rec["n_moves"][g])
        b, w, pl = int(rec["black"][g][0]), int(rec["white"][g][0]), int(rec["player"][g][0])
        for p in range(k):
            assert (b, w, pl) == (int(rec["black"][g][p]), int(rec["white"][g][p]), int(rec["player"][g][p])), (g, p)
            own, opp = (b, w) if pl == 0 else (w, b)
            sq = int(rec["action"][g][p])
            assert (L.bbr_legal(own, opp, n) >> sq) & 1, (g, p)
            o2, p2, fl, _ = host_play(L, sq, own, opp, n)
            pl = 1 - pl if fl & 1 else pl
            b, w = (o2, p2) if pl == 0 else (p2, o2)
        if k < 64:
            assert (b, w) == (int(rec["black"][g][k]), int(rec["white"][g][k])), g


# ---- 1. stateless rules ---------------------------------------------------------------------------------------------
def test_apply_moves_equals_host_standard_forms(E, L):
    cases = [(n, o, p) for n, o, p in golden_positions()]
    for n in (4, 6, 8):
        owns, opps = random_positions(4000, n, seed=40 + n)
        cases += [(n, o, p) for o, p in zip(owns, opps)]
        cases += [(n, o, p) for o, p in standard_playout_positions(L, n, games=20, seed=n)]
    for n in (4, 6, 8):
        sel = [(o, p) for m, o, p in cases if m == n]
        own = np.array([o for o, _ in sel], dtype=np.uint64)
        opp = np.array([p for _, p in sel], dtype=np.uint64)
        lr = E.legal_moves(own, opp, n)
        assert np.array_equal(lr, E.legal_moves(own, opp, n, rules=STD))
        assert [int(x) for x in lr] == [L.bbr_legal(o, p, n) for o, p in sel]
        rows, sqs = [], []
        for i, m in enumerate(int(x) for x in lr):
            for s in range(64):
                if (m >> s) & 1:
                    rows.append(i); sqs.append(s)
        rows = np.array(rows)
        o2, p2, fl, nl = E.apply_moves(own[rows], opp[rows], np.array(sqs, dtype=np.int32), n, rules=STD)
        differ = 0
        for j, (i, s) in enumerate(zip(rows, sqs)):
            want = host_play(L, s, int(own[i]), int(opp[i]), n)
            assert (int(o2[j]), int(p2[j]), int(fl[j]), int(nl[j])) == want, (n, hex(int(own[i])), hex(int(opp[i])), s)
            differ += host_play(L, s, int(own[i]), int(opp[i]), n, standard=False) != want
        assert differ > 0 if n >= 6 else differ == 0
        _, _, bad, _ = E.apply_moves(own[:1], opp[:1], np.array([-1], dtype=np.int32), n, rules=STD)
        assert int(bad[0]) == 0x80000000


# ---- 2. perft through the batched rules API ----------------------------------------------------------------------------
@pytest.mark.parametrize("n,want", [(8, [4, 12, 56, 244, 1396, 8200, 55092, 390216]),
                                    (6, [4, 12, 56, 244, 1364, 7604, 47740, 308716])])
def test_device_perft_level_by_level(E, n, want):
    b, w = oracle.board_to_bits(oracle.initial_board(n))
    own, opp = np.array([b], dtype=np.uint64), np.array([w], dtype=np.uint64)
    legal = E.legal_moves(own, opp, n, rules=STD)
    done = 0                                                    # finished games are leaves at every later depth
    got = []
    for _ in range(len(want)):
        rows = np.repeat(np.arange(own.size), [_popcount(x) for x in legal])
        bits = np.unpackbits(legal.astype("<u8").view(np.uint8).reshape(-1, 8), axis=1, bitorder="little")
        sqs = np.nonzero(bits)[1].astype(np.int32)              # row-major over (position, square) == rows' order
        own, opp, fl, legal = E.apply_moves(own[rows], opp[rows], sqs, n, rules=STD)
        assert not (fl & 0x80000000).any()
        fin = (fl & 4) != 0
        done += int(fin.sum())
        own, opp, legal = own[~fin], opp[~fin], legal[~fin]
        got.append(int(own.size) + done)
    assert got == want


# ---- 3. perft playouts -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [6, 8])
def test_perft_playouts_replay_under_host_standard_rules(E, L, n):
    G = 3000
    out = E.perft_playouts(G, n, seed=11, want_moves=True, rules=STD)
    ref = E.perft_playouts(G, n, seed=11, want_moves=True)
    differ = sum(not np.array_equal(out["moves"][g], ref["moves"][g]) for g in range(G))
    assert differ > G // 2
    b0, w0 = oracle.board_to_bits(oracle.initial_board(n))
    for g in range(0, G, 3):
        own, opp, player, passes = b0, w0, 0, 0
        plies = int(out["plies"][g])
        for p in range(plies):
            own, opp, fl, legal = host_play(L, int(out["moves"][g][p]), own, opp, n)
            player ^= fl & 1
            passes += (fl >> 1) & 1
        assert all(int(x) == 0xFF for x in out["moves"][g][plies:])
        black, white = (own, opp) if player == 0 else (opp, own)
        assert (int(out["black"][g]), int(out["white"][g])) == (black, white), g
        assert legal == 0 and bool(out["finished"][g]) and int(out["passes"][g]) == passes
        assert int(out["player"][g]) == 1 - player                # a finished game reports the opponent of the last mover


# ---- 4. sequential search against the oracle -------------------------------------------------------------------------
def _quirk_roots(L, n, count, seed):
    """Positions at ply >= 7 of standard-rule random games where some legal move flips differently under the quirk."""
    roots = []
    rng = np.random.default_rng(seed)
    while len(roots) < count:
        b, w = oracle.board_to_bits(oracle.initial_board(n))
        own, opp, player, ply = b, w, 0, 0
        legal = L.bbr_legal(own, opp, n)
        while legal:
            moves = [s for s in range(64) if (legal >> s) & 1]
            if ply >= 7 and any(host_play(L, s, own, opp, n) != host_play(L, s, own, opp, n, False) for s in moves):
                roots.append(((own, opp) if player == 0 else (opp, own)) + (player,))
                break
            own, opp, fl, legal = host_play(L, int(rng.choice(moves)), own, opp, n)
            player ^= fl & 1
            ply += 1
    return roots


@pytest.mark.parametrize("prior", ["hash", "host"])
def test_sequential_search_equals_oracle(E, L, prior):
    n, sims = 8, 160
    for black, white, player in _quirk_roots(L, n, 4, seed=5 if prior == "hash" else 6):
        board = oracle.bits_to_board(black, white, n)
        if prior == "hash":
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HASH, rules=STD)
            m = S.Mcts(n)
        else:
            def predict_batch(own, opp):
                outs = [prior_fns.sha_prior(canon_board(o, p, n)) for o, p in zip(own, opp)]
                return np.stack([o[0].ravel() for o in outs]), np.array([o[1] for o in outs], dtype=np.float32)
            e = E.Engine(n, 1, 4 * sims, E.PRIOR_HOST, rules=STD)
            m = S.Mcts(n, predict=prior_fns.sha_prior)
        e.reset(1, [black], [white], [player])
        e.search(sims, predict_batch if prior == "host" else None)
        v, ns = e.visits()
        q, p, tag = e.root_stats(0)
        nodes = e.counters()["nodes"]
        e.close()
        for _ in range(sims):
            m.simulate(board, player)
        canon = board if player == 0 else board[..., ::-1]
        rns, rv = m.visits(canon)
        assert int(ns[0]) == rns and visits_to_grid(v[0], n).tolist() == rv.reshape(-1).tolist(), hex(black)
        assert nodes == m.nodes
        rq, rp, rtag = m.node_stats(canon)
        for r in range(n):
            for c in range(n):
                if rtag[r, c] >= 0:
                    assert q[r * 8 + c] == rq[r, c] and p[r * 8 + c] == rp[r, c] and tag[r * 8 + c] == rtag[r, c]


# ---- 5. self-play against the oracle ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,sims,T,eg", [(6, 25, 1.0, 0.9), (6, 8, 0.0, 1.0), (8, 20, 1.0, 0.9), (8, 6, 0.0, 0.9)])
def test_selfplay_hash_prior_equals_oracle(E, n, sims, T, eg):
    G, slots = 14, 5                                              # more games than slots: the device queue is used
    starts = [S.playout(n, 4, g, max_moves=g % 3) for g in range(G)]
    black = [s["black"] for s in starts]; white = [s["white"] for s in starts]; player = [s["player"] for s in starts]
    ids = [900 + g for g in range(G)]
    e = E.Engine(n, slots, sims * n * n + 64, E.PRIOR_HASH, seed=13, log_visits=True, rules=STD)
    e.selfplay_begin(G, sims, T, eg, -1, black, white, player, ids)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    e.close()
    differ = 0
    for g in range(G):
        ref = S.execute_episode(n, sims, temperature=T, e_greedy=eg, seed=13, game_id=ids[g],
                                start_board=starts[g]["board"], start_player=player[g], log_visits=True)
        k = int(out["n_moves"][g])
        assert [int(a) for a in out["action"][g][:k]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        assert [int(x) for x in out["black"][g][:k]] == ref["black"] and [int(x) for x in out["white"][g][:k]] == ref["white"]
        assert int(out["winner"][g]) == ref["winner"]
        for p in range(k):
            assert visits_to_grid(out["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
        quirk = oracle.execute_episode(n, sims, temperature=T, e_greedy=eg, seed=13, game_id=ids[g],
                                       start_board=starts[g]["board"], start_player=player[g])
        differ += quirk["moves"] != ref["moves"]
    assert differ > G // 2


def test_selfplay_network_equals_oracle_fed_device_priors(E):
    from othellozero_b200 import net as oznet
    n, C, sims, games, slots, max_moves = 6, 128, 30, 10, 4, 14
    blob = oznet.init_weights(n, C, seed=8, randomize_bn=True)
    st = E.perft_playouts(games, n, seed=3, max_moves=7, rules=STD)
    black, white, player = st["black"], st["white"], st["player"].astype(np.int32)
    ids = np.arange(40, 40 + games, dtype=np.uint64)
    e = E.Engine(n, slots, sims * 40 + 64, E.PRIOR_NET, seed=2, log_visits=True, eval_cache_log2=14, rules=STD)
    e.load_weights(blob, C)
    e.selfplay_begin(games, sims, 1.0, 0.9, max_moves, black, white, player, ids)
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
        ref = S.execute_episode(n, sims, temperature=1.0, e_greedy=0.9, predict=predict, seed=2, game_id=int(ids[g]),
                                start_board=oracle.bits_to_board(int(black[g]), int(white[g]), n),
                                start_player=int(player[g]), max_moves=max_moves, log_visits=True)
        k = int(rec["n_moves"][g])
        assert k == len(ref["moves"])
        assert [int(a) for a in rec["action"][g][:k]] == [sq8(a, n) for a in ref["moves"]], f"game {g}"
        for p in range(k):
            assert visits_to_grid(rec["visits"][g][p], n).tolist() == ref["visits"][p].tolist(), (g, p)
    f.close()


# ---- 6. virtual-loss waves -------------------------------------------------------------------------------------------
def test_wave_search_standard_rules(E, L):
    sims, V = 203, 4
    roots = _quirk_roots(L, 8, 3, seed=9)
    outs = []
    for _ in range(2):
        e = E.Engine(8, 3, sims + 16, E.PRIOR_HASH, vl_width=V, rules=STD)
        e.reset(3, [r[0] for r in roots], [r[1] for r in roots], [r[2] for r in roots])
        e.search(sims)
        v, ns = e.visits()
        assert (ns == sims - 1).all() and (v.sum(axis=1) == ns).all()   # visits conserved, no virtual loss left
        e.search(50)
        v2, ns2 = e.visits()
        assert (ns2 == sims + 49).all() and (v2.sum(axis=1) == ns2).all()
        outs.append(v2.copy())
        e.close()
    assert np.array_equal(outs[0], outs[1])


def test_wave_selfplay_standard_rules_replays(E, L):
    n, sims, G, V = 8, 32, 64, 4
    outs = []
    for _ in range(2):
        e = E.Engine(n, G, sims * 61 + 64, E.PRIOR_HASH, seed=3, vl_width=V, rules=STD)
        e.selfplay_begin(G, sims, 1.0, 0.9)
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        e.close()
    for k in ("action", "n_moves", "winner"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    _replay_records(L, outs[0], n)


# ---- 7. façade drivers: self-play jobs and the arena -----------------------------------------------------------------
def test_selfplay_job_and_arena_replay_under_standard_rules(E, L):
    from othellozero_b200 import arena, selfplay
    from othellozero_b200.mcts import HashPriorNet
    n = 6
    sp = selfplay.SelfPlay(n, HashPriorNet(), max_games=8, num_simulations=12, seed=4, rules=STD)
    rec = sp.play(20, 1.0, 0.9, game_ids=np.arange(20, dtype=np.uint64))
    sp.close()
    _replay_records(L, rec, n)
    ex = selfplay.execute_episodes(3, n, HashPriorNet(), 1.0, 8, 1.0, 0.9, seed=1, rules=STD)
    assert len(ex) == 3 and all(len(x) > 0 for x in ex)

    rng = np.random.default_rng(0)
    G = 24
    out = arena.pit(n, HashPriorNet(), arena.RANDOM_AGENT, 10, n_games=G, rng=rng, rules=STD)
    assert out["plies"].min() > 7
    fb, fw = out["black"], out["white"]                          # every game ran to its end
    assert all(L.bbr_legal(int(b), int(w), n) == 0 and L.bbr_legal(int(w), int(b), n) == 0 for b, w in zip(fb, fw))
    wins = arena.evaluate_neural_network(n, 6, HashPriorNet(), 6, 1.0, rules=STD, rng=np.random.default_rng(1))
    assert 0 <= wins <= 6
    with pytest.raises(ValueError):
        arena.pit(n, HashPriorNet(), arena.RANDOM_AGENT, 4, n_games=2, rules="quirk")


def test_arena_moves_replay_under_standard_rules(E, L, monkeypatch):
    """Every move pit() applies is legal under the host standard rules and yields the position the host computes."""
    from othellozero_b200 import arena
    from othellozero_b200 import engine as eng
    from othellozero_b200.mcts import HashPriorNet
    n = 8
    real = eng.apply_moves
    seen = []

    def spy(own, opp, sq, board_size=8, device=0, rules="reference"):
        out = real(own, opp, sq, board_size, device, rules=rules)
        seen.append((np.array(own), np.array(opp), np.array(sq), out, rules))
        return out

    monkeypatch.setattr(arena._e, "apply_moves", spy)
    arena.pit(n, HashPriorNet(), HashPriorNet(), 6, n_games=6, rng=np.random.default_rng(2), rules=STD)
    assert seen and all(r == STD for *_, r in seen)
    for own, opp, sq, (o2, p2, fl, nl), _ in seen:
        for i in range(own.size):
            assert (L.bbr_legal(int(own[i]), int(opp[i]), n) >> int(sq[i])) & 1
            assert host_play(L, int(sq[i]), int(own[i]), int(opp[i]), n) == (int(o2[i]), int(p2[i]), int(fl[i]), int(nl[i]))


# ---- 8. the OthelloGame façade ---------------------------------------------------------------------------------------
def test_standard_othello_game_agrees_with_oracle(E):
    from othellozero_b200.othello import BoardView, OthelloGame, OthelloPlayer, StandardOthelloGame
    n = 8
    rng = np.random.default_rng(12)
    differ = 0
    for g in range(4):
        game = StandardOthelloGame(n)
        ref = oracle.initial_board(n)
        ch = 0
        while not game.has_finished():
            acts = oracle.valid_actions(ref, ch)
            r, c = acts[int(rng.integers(len(acts)))]
            player = game.current_player
            assert player is (OthelloPlayer.BLACK if ch == 0 else OthelloPlayer.WHITE)
            two = np.array(game.board(BoardView.TWO_CHANNELS), copy=True)
            fl = S.flip_squares(ref, ch, r, c)
            got = set(StandardOthelloGame.get_action_flip_squares(two, player, r, c))
            assert got == {(i, j) for i in range(n) for j in range(n) if fl[i, j]}
            differ += got != set(OthelloGame.get_action_flip_squares(two, player, r, c))
            nb, np_ = StandardOthelloGame.getNextState(two, player, (r, c))
            fb = np.array(two, copy=True)
            StandardOthelloGame.flip_board_squares(fb, player, r, c)
            game.play(r, c)
            ref = S.flip_board(ref, ch, r, c)
            nxt = 1 - ch
            if not oracle.valid_actions(ref, nxt):
                nxt = ch if oracle.valid_actions(ref, ch) else nxt
            ch = nxt
            assert np.array_equal(game.board(BoardView.TWO_CHANNELS).astype(np.uint8), ref)
            assert np.array_equal(nb.astype(np.uint8), ref) and np.array_equal(fb.astype(np.uint8), ref)
            assert np_ is game.current_player
        assert oracle.has_finished(ref)
    assert differ > 0
    # the reference class in the same process still plays the reference's flip rule; row 0 = . W W W B W W B
    board = oracle.bits_to_board(0x10 | (1 << 7), 0x2 | 0x4 | 0x8 | 0x20 | 0x40, n).astype(bool)
    got_ref = set(OthelloGame.get_action_flip_squares(board, OthelloPlayer.BLACK, 0, 0))
    got_std = set(StandardOthelloGame.get_action_flip_squares(board, OthelloPlayer.BLACK, 0, 0))
    assert got_std == {(0, 1), (0, 2), (0, 3)} and got_ref == {(0, 1), (0, 2), (0, 3), (0, 5), (0, 6)}
    assert OthelloGame.rules == "reference" and StandardOthelloGame.rules == STD


# ---- 9. the iteration driver -------------------------------------------------------------------------------------------
def test_iteration_driver_standard_rules():
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "6", "--arena-threshold", "4",
           "--arena-simulations", "8", "--iterations", "2", "--rules", "standard"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2
    for i, d in enumerate(lines, start=1):
        assert d["config"]["rules"] == "standard" and d["iteration"] == i
        assert d["positions_gathered"] >= 12 * 20 and d["selfplay_sims"] == 10 * d["positions_gathered"]
        assert np.isfinite(np.array(d["train_history"])).all()
