"""K7-K10 (bf16 tcgen05 OthelloNNet tower) against the PyTorch fp32 restatement (oracle/net_torch.py).
Tolerance (north_star): 1e-2 absolute on policy logits and on the value."""
import numpy as np
import pytest

import oracle
from oracle import net_torch

pytestmark = pytest.mark.gpu

TOL = 1e-2


def _positions(n, count, seed):
    """Canonical positions sampled from random playouts at assorted depths."""
    own, opp = [], []
    for g in range(count):
        po = oracle.playout(n, seed, g, max_moves=g % (n * n - 6))
        b, w, p = po["black"], po["white"], po["player"]
        own.append(w if p else b)
        opp.append(b if p else w)
    return np.array(own, dtype=np.uint64), np.array(opp, dtype=np.uint64)


@pytest.fixture(params=["table", "table-wino", "gemm"])
def conv2_mode(request, monkeypatch):
    """conv2 runs either as the conv1∘conv2 partial-product table gather (default) or as the tcgen05 implicit GEMM, and
    with the table conv3 runs either as the direct implicit GEMM (default) or as the opt-in 1-D Winograd F(2,3) SM-pair kernel;
    the modes are read from OZ_NET_CONV2 / OZ_NET_CONV3 when an engine is created."""
    monkeypatch.setenv("OZ_NET_CONV2", "gemm" if request.param == "gemm" else "table")
    monkeypatch.setenv("OZ_NET_CONV3", "wino" if request.param == "table-wino" else "direct")
    return request.param


def _check(n, C, B, max_games, seed, randomize_bn=True, conv2_mode="table"):
    import torch
    from othellozero_b200 import engine, net
    blob = net.init_weights(n, C, seed=seed, randomize_bn=randomize_bn)
    assert blob.size == net_torch.blob_floats(n, C)
    e = engine.Engine(n, max_games=max_games, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    e.load_weights(blob, C)
    own, opp = _positions(n, B, seed)
    pi, lg, v = e.net_forward(own, opp)
    x = net_torch.boards_from_bits(own, opp, n)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    rpi, rlg, rv, hidden = net_torch.forward(blob, x, n, C, device=dev, return_hidden=True)
    # layer-by-layer first: localises a failure
    rows = [n * n, n * n, (n - 2) ** 2, (n - 4) ** 2, 1, 1]
    chans = [C, C, C, C, 1024, 512]
    first = {"table": 1, "table-wino": 2, "gemm": 0}[conv2_mode]
    for li in range(first):
        with pytest.raises(RuntimeError):
            e.activation(li, B, rows[li], chans[li])   # conv1's (and, with Winograd conv3, conv2's) output is never materialised
    for li in range(first, 6):
        got = e.activation(li, B, rows[li], chans[li])
        ref = hidden[li]
        scale = max(1.0, float(np.abs(ref).max()))
        err = float(np.abs(got - ref).max())
        assert err <= 0.03 * scale, f"layer {li}: max abs err {err} (scale {scale})"
    assert np.abs(lg - rlg).max() <= TOL, f"logits err {np.abs(lg - rlg).max()}"
    assert np.abs(v - rv).max() <= TOL, f"value err {np.abs(v - rv).max()}"
    assert np.abs(pi - rpi).max() <= TOL
    assert np.allclose(pi.sum(axis=1), 1.0, atol=1e-4)
    e.close()
    return lg, v


def test_net_8x8_c512_ragged_batch(conv2_mode):
    # 301 boards: not a multiple of any tile's boards-per-tile (2, 3, 8, 128)
    _check(8, 512, 301, 512, seed=1, conv2_mode=conv2_mode)


def test_net_8x8_keras_default_init(conv2_mode):
    _check(8, 512, 64, 64, seed=2, randomize_bn=False, conv2_mode=conv2_mode)


def test_net_6x6_c512(conv2_mode):
    _check(6, 512, 130, 256, seed=3, conv2_mode=conv2_mode)


def test_net_small_channels_single_board(conv2_mode):
    _check(8, 128, 1, 8, seed=4, conv2_mode=conv2_mode)


@pytest.mark.parametrize("C", [256, 384, 640, 768, 896, 1024])
def test_net_other_channel_counts(C, conv2_mode):
    _check(8, C, 37, 64, seed=12, conv2_mode=conv2_mode)


def test_conv2_table_vs_gemm_agree(monkeypatch):
    """The two conv2 formulations differ only in where the nine tap sums are rounded to bf16."""
    from othellozero_b200 import engine, net
    n, C = 8, 512
    blob = net.init_weights(n, C, seed=21, randomize_bn=True)
    own, opp = _positions(n, 150, 21)
    outs = []
    monkeypatch.setenv("OZ_NET_CONV3", "direct")   # keeps conv2's output materialised
    for mode in ("table", "gemm"):
        monkeypatch.setenv("OZ_NET_CONV2", mode)
        e = engine.Engine(n, max_games=256, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
        e.load_weights(blob, C)
        pi, lg, v = e.net_forward(own, opp)
        a2 = e.activation(1, 150, 64, C)
        outs.append((lg, v, a2))
        e.close()
    scale = max(1.0, float(np.abs(outs[1][2]).max()))
    assert np.abs(outs[0][2] - outs[1][2]).max() <= 0.02 * scale
    assert np.abs(outs[0][0] - outs[1][0]).max() <= TOL and np.abs(outs[0][1] - outs[1][1]).max() <= TOL


def test_fused_tail_matches_split_launches(monkeypatch):
    """fc2 + heads as ONE kernel (opt-in OZ_NET_TAIL=fused, oz_tail_kernel: f2 stays in shared memory as the heads' A operand)
    against the default two generic launches: the accumulation orders are the same, so logits, probabilities, value and the f2 layer
    must be BIT-identical - including batches that leave the last 128-row tile ragged and batches with more tiles than SMs
    (a CTA then walks several tiles and every barrier of the kernel changes phase)."""
    from othellozero_b200 import engine, net
    for n, C, B, seed in ((8, 512, 301, 31), (6, 128, 148 * 128 + 200, 32), (8, 128, 1, 33)):
        blob = net.init_weights(n, C, seed=seed, randomize_bn=True)
        own, opp = _positions(n, min(B, 600), seed)
        own, opp = np.resize(own, B), np.resize(opp, B)
        outs = []
        for mode in ("split", "fused"):
            monkeypatch.setenv("OZ_NET_TAIL", mode)
            e = engine.Engine(n, max_games=B + 5, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
            e.load_weights(blob, C)
            pi, lg, v = e.net_forward(own, opp)
            outs.append((pi, lg, v, e.activation(5, B, 1, 512)))
            e.close()
        for a, b, name in zip(outs[0], outs[1], ("pi", "logits", "v", "f2")):
            assert np.array_equal(a, b), f"{name} differs between the fused and the split tail (n={n}, C={C}, B={B})"


def test_conv3_wino_vs_direct_agree(monkeypatch):
    """conv3 as 1-D Winograd F(2,3) (transformed bf16 inputs/filters, fp32 accumulate) against the direct implicit GEMM:
    same layer output up to bf16 rounding of the transforms, same logits/value within the north-star tolerance."""
    from othellozero_b200 import engine, net
    for n, B in ((8, 150), (6, 77)):
        C = 512
        blob = net.init_weights(n, C, seed=22, randomize_bn=True)
        own, opp = _positions(n, B, 22)
        outs = []
        for mode in ("wino", "direct"):
            monkeypatch.setenv("OZ_NET_CONV2", "table")
            monkeypatch.setenv("OZ_NET_CONV3", mode)
            e = engine.Engine(n, max_games=256, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
            e.load_weights(blob, C)
            pi, lg, v = e.net_forward(own, opp)
            a3 = e.activation(2, B, (n - 2) ** 2, C)
            outs.append((lg, v, a3))
            e.close()
        scale = max(1.0, float(np.abs(outs[1][2]).max()))
        assert np.abs(outs[0][2] - outs[1][2]).max() <= 0.02 * scale
        assert np.abs(outs[0][0] - outs[1][0]).max() <= TOL and np.abs(outs[0][1] - outs[1][1]).max() <= TOL


def test_net_is_row_independent(conv2_mode):
    """A board's output must not depend on its position in the batch or on its neighbours."""
    from othellozero_b200 import engine, net
    n, C = 8, 128
    blob = net.init_weights(n, C, seed=5, randomize_bn=True)
    e = engine.Engine(n, max_games=256, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    e.load_weights(blob, C)
    own, opp = _positions(n, 200, 9)
    pi, lg, v = e.net_forward(own, opp)
    perm = np.random.default_rng(0).permutation(200)
    pi2, lg2, v2 = e.net_forward(own[perm], opp[perm])
    assert np.array_equal(lg[perm], lg2) and np.array_equal(v[perm], v2)
    pi3, lg3, v3 = e.net_forward(own[:7], opp[:7])
    assert np.array_equal(lg[:7], lg3)
    e.close()


def test_predict_contract():
    """NNetWrapper.predict: (N,N,2) board -> (pi (N,N) float32 probabilities, v float32)."""
    from othellozero_b200 import net
    nn = net.B200NNet((8, 8), num_channels_1=128, max_batch=8, seed=6)
    board = oracle.initial_board(8).astype(bool)
    pi, v = nn.predict(board)
    assert pi.shape == (8, 8) and pi.dtype == np.float32 and abs(float(pi.sum()) - 1.0) < 1e-4
    assert -1.0 <= float(v) <= 1.0
    x = board[None].astype(np.float32)
    rpi, _, rv = net_torch.forward(nn.blob, x, 8, 128)
    assert np.abs(pi.ravel() - rpi[0]).max() <= TOL and abs(float(v) - float(rv[0])) <= TOL


def test_selfplay_with_net_matches_oracle_search():
    """End to end: device self-play with the device net == oracle search fed the SAME (device) priors."""
    from othellozero_b200 import engine, net
    n, C, sims = 6, 128, 16
    blob = net.init_weights(n, C, seed=7, randomize_bn=True)
    e = engine.Engine(n, max_games=4, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, log_visits=True)
    e.load_weights(blob, C)
    e.selfplay_begin(4, sims, 1.0, 1.0)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()
    pe = engine.Engine(n, max_games=64, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    pe.load_weights(blob, C)

    def predict(board):
        own, opp = net.boards_to_bits(board)
        pi, _, v = pe.net_forward(own, opp, want_logits=False)
        return pi[0].reshape(n, n), v[0]

    ref = oracle.execute_episode(n, sims, predict=predict, log_visits=True)
    k = int(out["n_moves"][0])
    assert [int(a) for a in out["action"][0][:k]] == [(a // n) * 8 + a % n for a in ref["moves"]]
    assert int(out["winner"][0]) == ref["winner"]
    assert e.counters()["nodes"] == 4 * ref["net_calls"]
    e.close(); pe.close()


def test_eval_cache_is_results_preserving():
    """Cross-game evaluation cache: identical positions are evaluated once; records must not change."""
    from othellozero_b200 import engine, net
    n, C, sims, G = 6, 128, 16, 96
    blob = net.init_weights(n, C, seed=11, randomize_bn=True)
    ids = np.arange(G, dtype=np.uint64) + 7000
    outs, ctr = [], []
    for lg in (0, 16):
        e = engine.Engine(n, max_games=G, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, seed=5,
                          log_visits=True, eval_cache_log2=lg)
        e.load_weights(blob, C)
        e.selfplay_begin(G, sims, 1.0, 0.8, -1, None, None, None, ids)   # all games start at the initial position
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        ctr.append(e.counters())
        e.close()
    a, b = outs
    for k in ("black", "white", "action", "player", "n_moves", "winner", "visits"):
        assert np.array_equal(a[k], b[k]), k
    assert ctr[0]["cache_hits"] == 0 and ctr[0]["cache_aliases"] == 0
    assert ctr[1]["cache_hits"] + ctr[1]["cache_aliases"] > 0
    assert ctr[0]["nodes"] == ctr[1]["nodes"] and ctr[0]["sims"] == ctr[1]["sims"]


def test_config0_6x6_25sims_c512_episode():
    """BASELINE configs[0]: 6x6, 25 sims/move, random-init OthelloNNet (C=512), one self-play game; the oracle search
    fed the same device priors must replay it move for move."""
    from othellozero_b200 import engine, net
    n, C, sims = 6, 512, 25
    blob = net.init_weights(n, C, seed=0)
    e = engine.Engine(n, max_games=1, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, log_visits=True)
    e.load_weights(blob, C)
    e.selfplay_begin(1, sims, 1.0, 1.0)
    assert e.selfplay_run(-1) == 0
    out = e.selfplay_records()

    def predict(board):
        own, opp = net.boards_to_bits(board)
        pi, _, v = e.net_forward(own, opp, want_logits=False)
        return pi[0].reshape(n, n), v[0]

    ref = oracle.execute_episode(n, sims, predict=predict, log_visits=True)
    k = int(out["n_moves"][0])
    assert [int(a) for a in out["action"][0][:k]] == [(a // n) * 8 + a % n for a in ref["moves"]]
    for p in range(k):
        got = [int(out["visits"][0][p][r * 8 + c]) for r in range(n) for c in range(n)]
        assert got == ref["visits"][p].tolist()
    assert int(out["winner"][0]) == ref["winner"]
    e.close()


def test_sim_budget_is_results_preserving(monkeypatch):
    """The tree kernel yields after OZ_TREE_SIM_BUDGET evaluator-free simulations per launch (terminal visits, cache
    hits); where a game pauses must not change anything it plays or counts."""
    from othellozero_b200 import engine, net
    n, C, sims, G = 6, 128, 20, 48
    blob = net.init_weights(n, C, seed=13, randomize_bn=True)
    ids = np.arange(G, dtype=np.uint64) + 500
    outs, steps = [], []
    for budget in ("0", "1", "8"):
        monkeypatch.setenv("OZ_TREE_SIM_BUDGET", budget)
        e = engine.Engine(n, max_games=G, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, seed=9, log_visits=True,
                          eval_cache_log2=14)
        e.load_weights(blob, C)
        e.selfplay_begin(G, sims, 1.0, 0.9, -1, None, None, None, ids)
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        c = e.counters()
        steps.append((c["sims"], c["nodes"], c["terminal_visits"], c["moves"]))
        e.close()
    for o in outs[1:]:
        for k in ("black", "white", "action", "player", "n_moves", "winner", "visits"):
            assert np.array_equal(outs[0][k], o[k]), k
    assert steps[0] == steps[1] == steps[2]
    assert steps[0][2] > 0   # the endgames did visit terminal edges


def test_game_queue_with_network_matches_one_batch():
    """Queued self-play with the real evaluator (leaf batches mix games of different ages, evaluation cache on):
    every game equals the same game played with all games resident at once."""
    from othellozero_b200 import engine, net
    n, C, sims, total, slots = 6, 128, 10, 40, 8
    blob = net.init_weights(n, C, seed=31, randomize_bn=True)
    ids = np.arange(100, 100 + total, dtype=np.uint64)
    outs = []
    for mg, cache in ((slots, 16), (total, 0)):
        e = engine.Engine(n, max_games=mg, nodes_per_game=sims * 36 + 64, prior_mode=engine.PRIOR_NET,
                          eval_cache_log2=cache, log_visits=True)
        e.load_weights(blob, C)
        e.selfplay_begin(total, sims, 1.0, 0.85, game_ids=ids)
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        e.close()
    a, b = outs
    assert np.array_equal(a["n_moves"], b["n_moves"]) and np.array_equal(a["winner"], b["winner"])
    for g in range(total):
        k = int(a["n_moves"][g])
        assert np.array_equal(a["action"][g][:k], b["action"][g][:k])
        assert np.array_equal(a["visits"][g][:k], b["visits"][g][:k])


@pytest.mark.parametrize("n", [6, 8])
def test_device_tower_reproduces_delta_network_known_answer(n, conv2_mode):
    """The hand-derived whole-network answer of tests/kat_net.py (HWIO cross-correlation, 'same' padding, (h,w,c) flatten,
    Dense (in,out), BN folding) on the CUDA tower itself - not only through the fp32 restatement."""
    import kat_net
    from othellozero_b200 import engine
    C = 128
    blob, boards, exp = kat_net.delta_network(n, C, bn5=(2.0, 0.1, 0.5, 4.0 - 1e-3))
    own = np.array([sum(1 << (r * 8 + c) for r in range(n) for c in range(n) if boards[b, r, c, 0]) for b in range(2)], dtype=np.uint64)
    opp = np.array([sum(1 << (r * 8 + c) for r in range(n) for c in range(n) if boards[b, r, c, 1]) for b in range(2)], dtype=np.uint64)
    e = engine.Engine(n, max_games=4, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    e.load_weights(blob, C)
    pi, lg, v = e.net_forward(own, opp)
    e.close()
    assert np.abs(lg - exp["logits"]).max() <= TOL, np.abs(lg - exp["logits"]).max()
    assert np.abs(v - exp["v"]).max() <= TOL and np.abs(pi - exp["pi"]).max() <= TOL
    assert abs(float(lg[0].max() - lg[1].max())) > 1.0      # board 0 hits the fc1 tap, the transposed board 1 misses it
