"""FP8 network evaluation (DESIGN.md 13) on the device.

The device FP8 tower is checked against the host emulation (tests/fp8_emul.py), layer by layer.  The emulation is fed
the device's scales and, for each layer, the device's own input to that layer.  It reproduces every rounding, so each
layer can differ only through the order of the fp32 sums.  That flips an e4m3 or bf16 rounding only for a value within
an fp32 ulp or so of a rounding boundary, and the flip moves the value by one step.  So each layer must agree code for
code, except for a tiny fraction of small differences (_code_mismatch).

End to end, flips cascade: one act2 flip moves thousands of act3 pre-activations a little, and some of those cross a
boundary in turn.  So the end-to-end comparison is made with the fp32 oracle instead: the device's error must match the
emulation's own error on the same weights.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from oracle import net_torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fp8_emul  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _positions(n, count, seed):
    own, opp = [], []
    for g in range(count):
        po = oracle.playout(n, seed, g, max_moves=g % (n * n - 6))
        b, w, p = po["black"], po["white"], po["player"]
        own.append(w if p else b)
        opp.append(b if p else w)
    return np.array(own, dtype=np.uint64), np.array(opp, dtype=np.uint64)


def _fp8_engine(n, C, blob, max_games=64, **kw):
    from othellozero_b200 import engine
    e = engine.Engine(n, max_games=max_games, nodes_per_game=2, prior_mode=engine.PRIOR_NET, **kw)
    e.load_weights(blob, C, "fp8")
    return e


def _code_mismatch(a, b):
    """(fraction of differing elements, True iff every difference is small) for activations in e4m3 units.

    A difference is small if the two values are adjacent e4m3 codes, or if they differ by at most 1 in scaled units,
    which is 1/448 of the layer's calibrated maximum.  The second case covers values near zero.  A flip upstream moves a
    pre-activation by a small absolute amount.  Near zero the e4m3 grid is finer than that amount, so the value can move
    by several codes while the change stays small in absolute terms."""
    diff = a != b
    if not diff.any():
        return 0.0, True
    import torch
    ca = torch.as_tensor(a[diff]).to(torch.float8_e4m3fn).view(torch.uint8).numpy().astype(int)
    cb = torch.as_tensor(b[diff]).to(torch.float8_e4m3fn).view(torch.uint8).numpy().astype(int)
    small = (np.abs(ca - cb) <= 1) | (np.abs(a[diff] - b[diff]) <= 1.0)
    return float(diff.mean()), bool(small.all())


@pytest.mark.parametrize("randomize_bn", [False, True])
@pytest.mark.parametrize("n,C", [(6, 256), (6, 512), (8, 256), (8, 512), (6, 768), (8, 1024)])
def test_fp8_tower_matches_emulation(n, C, randomize_bn):
    from othellozero_b200 import net
    blob = net.init_weights(n, C, seed=3, randomize_bn=randomize_bn)
    B = 48
    own, opp = _positions(n, B, seed=5)
    e = _fp8_engine(n, C, blob)
    pi, lg, v = e.net_forward(own, opp)
    sc = e.fp8_scales()
    hid = [e.activation(l, B, r, C) for l, r in ((1, n * n), (2, (n - 2) ** 2), (3, (n - 4) ** 2))]
    e.close()
    # weight scales are a pure function of the fp32 weights: bit-equal to the host's
    for k, ref in fp8_emul.weight_scales(blob, n, C).items():
        assert np.array_equal(sc[k], ref), k
    assert np.all(sc["act"] > 0)
    epi, elg, ev, ehid = fp8_emul.forward(blob, own, opp, n, C, scales=sc)
    # layer by layer: act2 from the boards; act3 / act4 from the device's act2 / act3; the outputs from the device's act4
    checks = [("act2", hid[0], ehid["act2"])]
    for i, (src, dst) in enumerate((("act2", "act3"), ("act3", "act4"))):
        checks.append((dst, hid[i + 1], fp8_emul.forward(blob, own, opp, n, C, scales=sc, inject={src: hid[i]})[3][dst]))
    for name, a, b in checks:
        frac, small = _code_mismatch(a, b)
        print(f"  {name}: {frac:.2e} of elements differ, max |diff| {np.abs(a - b).max():.3g} (e4m3 units)")
        assert small and frac < 1e-3, (name, frac, np.abs(a - b).max())
    _, ilg, iv, _ = fp8_emul.forward(blob, own, opp, n, C, scales=sc, inject={"act4": hid[2]})
    opi, olg, ov = net_torch.forward(blob, net_torch.boards_from_bits(own, opp, n), n, C)
    err_emul = max(np.abs(elg - olg).max(), np.abs(ev - ov).max())
    err_dev = max(np.abs(lg - olg).max(), np.abs(v - ov).max())
    d_tail = max(np.abs(lg - ilg).max(), np.abs(v - iv).max())
    d = max(np.abs(lg - elg).max(), np.abs(v - ev).max())
    print(f"n={n} C={C} bn={randomize_bn}: FP8 vs fp32 oracle {err_dev:.3g} (emulation {err_emul:.3g}); "
          f"fc1..heads vs emulation {d_tail:.3g}; end to end vs emulation {d:.3g}; policy {np.abs(pi - opi).max():.3g}")
    assert d_tail <= 0.05 * err_emul + 1e-4
    assert err_dev <= 1.25 * err_emul + 1e-3
    assert np.allclose(pi.sum(axis=1), 1.0, atol=1e-5)


M64 = (1 << 64) - 1
CAL_SEED, CAL_GAMES = 0xCA11B7A7E, 256       # oz_net.cu: CAL_SEED, CAL_GAMES
CAL_POSITIONS = {6: 8175, 8: 15358}          # DESIGN.md 13


def _sm64(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    z = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def _calibration_positions(n):
    """The calibration set restated on the host: every position (mover's frame) of CAL_GAMES random games under the
    reference rules; move p of game g is legal move number ((sm64(key + p) >> 32) * count) >> 32, ascending by bit, with
    key = sm64(sm64(CAL_SEED) + g).  Moves are played by the device rules API (passes are automatic)."""
    from othellozero_b200 import engine
    q = (n - 2) // 2
    white = (1 << (q * 8 + q)) | (1 << ((q + 1) * 8 + q + 1))
    black = (1 << (q * 8 + q + 1)) | (1 << ((q + 1) * 8 + q))
    keys = [_sm64((_sm64(CAL_SEED) + g) & M64) for g in range(CAL_GAMES)]
    own = np.full(CAL_GAMES, black, dtype=np.uint64)
    opp = np.full(CAL_GAMES, white, dtype=np.uint64)
    legal = engine.legal_moves(own, opp, n)
    got_own, got_opp = [], []
    ply = 0
    while (legal != 0).any():
        idx = np.nonzero(legal != 0)[0]
        got_own.append(own[idx].copy())
        got_opp.append(opp[idx].copy())
        sq = []
        for g in idx:
            bits = [b for b in range(64) if int(legal[g]) >> b & 1]
            k = ((_sm64((keys[g] + ply) & M64) >> 32) * len(bits)) >> 32
            sq.append(bits[k])
        o2, p2, _, nl = engine.apply_moves(own[idx], opp[idx], np.array(sq, np.int32), n)
        own[idx], opp[idx], legal[idx] = o2, p2, nl
        ply += 1
    return np.concatenate(got_own), np.concatenate(got_opp)


@pytest.mark.parametrize("n", [6, 8])
def test_fp8_activation_scales_are_the_calibration_maxima(n):
    """sa_l = amax_l / 448 exactly, amax_l being the largest bf16 act2 / act3 / act4 of the documented calibration set
    through the bf16 tower of the same weights (an engine of 8 rows, so the calibration runs in many chunks)."""
    from othellozero_b200 import engine, net
    C = 256
    own, opp = _calibration_positions(n)
    assert own.size == CAL_POSITIONS[n]
    blob = net.init_weights(n, C, seed=12, randomize_bn=True)
    f = _fp8_engine(n, C, blob, max_games=8)
    sa = f.fp8_scales()["act"]
    f.close()
    e = engine.Engine(n, max_games=4096, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    e.load_weights(blob, C)
    amax = np.zeros(3, dtype=np.float32)
    for i in range(0, own.size, 4096):
        k = min(4096, own.size - i)
        e.net_forward(own[i:i + k], opp[i:i + k], want_logits=False)
        for l, rows in enumerate((n * n, (n - 2) ** 2, (n - 4) ** 2)):
            amax[l] = max(amax[l], e.activation(l + 1, k, rows, C).max())
    e.close()
    assert np.all(amax > 0)
    assert np.array_equal(sa, amax / np.float32(448.0)), (sa, amax)


def test_fp8_emulation_without_quantisation_is_the_oracle():
    from othellozero_b200 import net
    n, C = 6, 256
    blob = net.init_weights(n, C, seed=4, randomize_bn=True)
    own, opp = _positions(n, 16, seed=2)
    _, elg, ev, _ = fp8_emul.forward(blob, own, opp, n, C, quantize=False)
    _, olg, ov = net_torch.forward(blob, net_torch.boards_from_bits(own, opp, n), n, C)
    assert np.abs(elg - olg).max() < 1e-4 and np.abs(ev - ov).max() < 1e-4


def test_fp8_is_independent_of_the_batch():
    from othellozero_b200 import net
    n, C = 8, 256
    blob = net.init_weights(n, C, seed=8, randomize_bn=True)
    own, opp = _positions(n, 40, seed=9)
    small = _fp8_engine(n, C, blob, max_games=8)
    big = _fp8_engine(n, C, blob, max_games=4096)
    s1, s2 = small.fp8_scales(), big.fp8_scales()
    for k in s1:
        assert np.array_equal(s1[k], s2[k]), k
    pi_b, lg_b, v_b = big.net_forward(own, opp)
    rows = [small.net_forward(own[i:i + 8], opp[i:i + 8]) for i in range(0, 40, 8)]
    assert np.array_equal(np.concatenate([r[1] for r in rows]), lg_b)
    assert np.array_equal(np.concatenate([r[2] for r in rows]), v_b)
    one = [big.net_forward(own[i:i + 1], opp[i:i + 1]) for i in (0, 17, 39)]   # row independence
    for (p1, l1, v1), i in zip(one, (0, 17, 39)):
        assert np.array_equal(l1[0], lg_b[i]) and v1[0] == v_b[i]
    small.close(); big.close()


def test_fp8_scales_follow_the_weights_only():
    from othellozero_b200 import engine, net
    n, C = 6, 256
    blob = net.init_weights(n, C, seed=1, randomize_bn=True)
    ref = _fp8_engine(n, C, blob)
    s0 = ref.fp8_scales()
    std = _fp8_engine(n, C, blob, rules="standard")
    for k in s0:
        assert np.array_equal(s0[k], std.fp8_scales()[k]), k
    ref.load_weights(blob, C, "fp8")  # reload: same scales
    for k in s0:
        assert np.array_equal(s0[k], ref.fp8_scales()[k]), k
    ref.load_weights(net.init_weights(n, C, seed=2, randomize_bn=True), C, "fp8")
    s1 = ref.fp8_scales()
    assert not np.array_equal(s0["act"], s1["act"]) and not np.array_equal(s0["conv3"], s1["conv3"])
    ref.close(); std.close()


def test_fp8_eval_cache_is_results_preserving():
    from othellozero_b200 import engine, net
    n, C, sims, G = 6, 256, 16, 96
    blob = net.init_weights(n, C, seed=11, randomize_bn=True)
    ids = np.arange(G, dtype=np.uint64) + 7000
    outs, ctr = [], []
    for lg in (0, 16):
        e = engine.Engine(n, max_games=G, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, seed=5,
                          log_visits=True, eval_cache_log2=lg)
        e.load_weights(blob, C, "fp8")
        e.selfplay_begin(G, sims, 1.0, 0.8, -1, None, None, None, ids)
        assert e.selfplay_run(-1) == 0
        outs.append(e.selfplay_records())
        ctr.append(e.counters())
        e.close()
    a, b = outs
    for k in ("black", "white", "action", "player", "n_moves", "winner", "visits"):
        assert np.array_equal(a[k], b[k]), k
    assert ctr[1]["cache_hits"] + ctr[1]["cache_aliases"] > 0


def test_fp8_selfplay_matches_oracle_search_and_queue():
    from othellozero_b200 import engine, net
    n, C, sims = 6, 256, 16
    blob = net.init_weights(n, C, seed=7, randomize_bn=True)
    ids = np.arange(6, dtype=np.uint64)
    e = engine.Engine(n, max_games=2, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, log_visits=True)
    e.load_weights(blob, C, "fp8")
    e.selfplay_begin(6, sims, 1.0, 1.0, -1, None, None, None, ids)   # 6 games through 2 slots: the game queue
    assert e.selfplay_run(-1) == 0
    queued = e.selfplay_records()
    sep = []
    for g in range(6):
        e2 = engine.Engine(n, max_games=1, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, log_visits=True)
        e2.load_weights(blob, C, "fp8")
        e2.selfplay_begin(1, sims, 1.0, 1.0, -1, None, None, None, ids[g:g + 1])
        assert e2.selfplay_run(-1) == 0
        sep.append(e2.selfplay_records())
        e2.close()
    for g in range(6):
        k = int(queued["n_moves"][g])
        assert k == int(sep[g]["n_moves"][0])
        assert np.array_equal(queued["action"][g][:k], sep[g]["action"][0][:k])
        assert np.array_equal(queued["visits"][g][:k], sep[g]["visits"][0][:k])
    pe = _fp8_engine(n, C, blob)

    def predict(board):
        own, opp = net.boards_to_bits(board)
        pi, _, v = pe.net_forward(own, opp, want_logits=False)
        return pi[0].reshape(n, n), v[0]

    e1 = engine.Engine(n, max_games=1, nodes_per_game=sims * 40, prior_mode=engine.PRIOR_NET, log_visits=True)
    e1.load_weights(blob, C, "fp8")
    e1.selfplay_begin(1, sims, 1.0, 1.0)
    assert e1.selfplay_run(-1) == 0
    out = e1.selfplay_records()
    ref = oracle.execute_episode(n, sims, predict=predict, log_visits=True)
    k = int(out["n_moves"][0])
    assert [int(a) for a in out["action"][0][:k]] == [(a // n) * 8 + a % n for a in ref["moves"]]
    assert int(out["winner"][0]) == ref["winner"]
    if "visits" in ref:
        for i in range(k):
            vis = np.zeros(64, dtype=np.int64)
            for a, c in enumerate(ref["visits"][i]):
                vis[(a // n) * 8 + a % n] = c
            assert np.array_equal(out["visits"][0][i].astype(np.int64), vis), i
    e.close(); e1.close(); pe.close()


def test_fp8_errors():
    from othellozero_b200 import engine, net
    from othellozero_b200._lib import OzError
    n, C = 6, 256
    blob = net.init_weights(n, C, seed=0)
    e = engine.Engine(n, max_games=4, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    e.load_weights(blob, C)
    with pytest.raises(OzError, match="FP8"):
        e.fp8_scales()
    with pytest.raises(OzError, match="precision cannot change"):
        e.load_weights(blob, C, "fp8")
    e.close()
    f = _fp8_engine(n, C, blob, max_games=4)
    with pytest.raises(OzError, match="precision cannot change"):
        f.load_weights(blob, C, "bf16")
    f.close()
    g = engine.Engine(n, max_games=4, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    with pytest.raises(AssertionError, match="multiple of 256"):
        g.load_weights(net.init_weights(n, 128, seed=0), 128, "fp8")
    g.close()


@pytest.mark.parametrize("var,val,msg", [("OZ_NET_CONV2", "gemm", "OZ_NET_CONV2=gemm"),
                                         ("OZ_NET_CONV3", "wino", "OZ_NET_CONV3=wino"),
                                         ("OZ_NET_NO_2SM", "1", "OZ_NET_NO_2SM=1")])
def test_fp8_unsupported_modes_fail(var, val, msg):
    # a fresh process: OZ_NET_NO_2SM is read once per process
    code = ("from othellozero_b200 import engine, net\n"
            "from othellozero_b200._lib import OzError\n"
            "e = engine.Engine(6, max_games=4, nodes_per_game=2, prior_mode=engine.PRIOR_NET)\n"
            "try:\n"
            "    e.load_weights(net.init_weights(6, 256, seed=0), 256, 'fp8')\n"
            "    print('LOADED')\n"
            "except OzError as exc:\n"
            "    print('ERR', exc)\n")
    env = dict(os.environ, **{var: val})
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    assert "ERR" in out.stdout and msg in out.stdout, out.stdout


def test_fp8_fused_tail_matches_split_launches(monkeypatch):
    from othellozero_b200 import net
    n, C = 8, 256
    blob = net.init_weights(n, C, seed=6, randomize_bn=True)
    own, opp = _positions(n, 24, seed=4)
    a = _fp8_engine(n, C, blob)
    ref = a.net_forward(own, opp)
    a.close()
    monkeypatch.setenv("OZ_NET_TAIL", "fused")
    b = _fp8_engine(n, C, blob)
    got = b.net_forward(own, opp)
    b.close()
    assert np.array_equal(ref[1], got[1]) and np.array_equal(ref[2], got[2])


def test_fp8_arena_and_iteration_end_to_end(tmp_path):
    from othellozero_b200 import arena, net
    n, C = 6, 256
    blob = net.init_weights(n, C, seed=2)
    f8 = net.B200NNet((n, n), C, max_batch=8, blob=blob, precision="fp8")
    b16 = net.B200NNet((n, n), C, max_batch=8, blob=blob)
    assert f8.copy().precision == "fp8"
    out = arena.pit(n, f8, b16, 8, n_games=8, rng=np.random.default_rng(0))
    assert len(out["winner"]) == 8
    r = subprocess.run([sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "256",
                        "--episodes", "4", "--num-simulations", "4", "--epochs", "1", "--arena-games", "2",
                        "--arena-simulations", "4", "--max-concurrent", "8", "--precision", "fp8"],
                       cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["config"]["precision"] == "fp8" and line["selfplay_sims"] > 0
