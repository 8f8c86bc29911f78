"""Standard scoring (a finished game with equal disc counts is a draw) without a GPU: the C-ABI's checks of the scoring
flag, board_arg, the draw-scoring oracles' sources and their draw semantics, and the host-side consumers of winner code 2
(training examples, packed rows, the training step, the iteration helpers, the game classes' scoring attribute)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
import oracle_scoring
import oracle_standard

SCORING_STANDARD = 0x400


def test_abi_scoring_flag_validation():
    import torch
    from othellozero_b200 import _lib
    L = _lib.load()
    assert _lib.SCORING_STANDARD == SCORING_STANDARD
    own, opp = np.array([0x0000000810000000], dtype=np.uint64), np.array([0x0000001008000000], dtype=np.uint64)
    sq = np.array([19], dtype=np.int32)
    o2, p2, nl = np.zeros(1, np.uint64), np.zeros(1, np.uint64), np.zeros(1, np.uint64)
    fl = np.zeros(1, np.uint32)
    p64, p32, pi32 = _lib.u64p, _lib.u32p, _lib.i32p

    def apply(bs):
        return L.oz_rules_apply_host(0, bs, _lib.ptr(own, p64), _lib.ptr(opp, p64), _lib.ptr(sq, pi32), _lib.ptr(o2, p64),
                                     _lib.ptr(p2, p64), _lib.ptr(fl, p32), _lib.ptr(nl, p64), 1)

    def perft(bs):
        return L.oz_perft_playouts_host(0, bs, 0, 0, 1, -1, _lib.ptr(o2, p64), _lib.ptr(p2, p64), _lib.ptr(fl, p32), None)

    def legal(bs):
        return L.oz_rules_legal_moves_host(0, bs, _lib.ptr(own, p64), _lib.ptr(opp, p64), _lib.ptr(nl, p64), 1)

    def create(bs):
        cfg = _lib.EngineConfig(0, bs, 1, 64, _lib.PRIOR_HASH, 0, 0, 1, 1.0, 0)
        h = C.c_void_p()
        rc = L.oz_engine_create(C.byref(cfg), C.byref(h))
        if rc == _lib.OZ_OK:
            L.oz_engine_destroy(h)
        return rc

    for fn in (apply, perft, legal, create):
        for bad in (0x400, 7 | 0x400, 8 | 0x200 | 0x400, 8 | 0x800, 6 | 0x100 | 0x800):
            assert fn(bad) == _lib.OZ_ERR_INVALID, (fn.__name__, hex(bad))
        with pytest.raises(AssertionError):
            _lib.check(fn(8 | 0x800))
    for n in (6, 8):
        assert L.oz_net_blob_floats(n | SCORING_STANDARD, 128) == L.oz_net_blob_floats(n, 128) > 0
        assert L.oz_net_blob_floats(n | 0x100 | SCORING_STANDARD, 128) == L.oz_net_blob_floats(n, 128)
    assert L.oz_net_blob_floats(8 | 0x800, 128) == -1
    if torch.cuda.is_available():
        return
    for fn in (apply, perft, legal, create):                    # a valid flag reaches the device check: no CPU fallback
        for good in (8 | SCORING_STANDARD, 8 | 0x100 | SCORING_STANDARD):
            assert fn(good) == _lib.OZ_ERR_CUDA, (fn.__name__, hex(good))
        with pytest.raises(_lib.OzError):
            _lib.check(fn(8 | SCORING_STANDARD))


def test_board_arg_scoring():
    from othellozero_b200 import _lib, engine
    assert _lib.SCORINGS == ("reference", "standard")
    assert engine.board_arg(8) == 8 and engine.board_arg(8, "reference", "reference") == 8
    assert engine.board_arg(8, scoring="standard") == 8 | 0x400
    assert engine.board_arg(6, "standard", "standard") == 6 | 0x100 | 0x400
    assert engine.board_arg(4, "standard", "reference") == 4 | 0x100
    for bad in ("draw", "Standard", None):
        with pytest.raises(ValueError):
            engine.board_arg(8, "reference", bad)
    with pytest.raises(ValueError):
        engine.Engine(8, 1, 64, scoring="tournament")
    from othellozero_b200 import othello, selfplay
    with pytest.raises(ValueError):
        othello.game_class("reference", "tournament")
    with pytest.raises(ValueError):
        selfplay.make_b200_worker(scoring="tournament")


@pytest.mark.parametrize("rules", ["reference", "standard"])
def test_scoring_oracle_sources_differ_by_the_patched_statements(rules):
    """Each draw-scoring oracle is its base oracle's source with one statement added to orc_winner and the terminal
    reward statement of simulate_rec replaced; every other line is the same."""
    ref = open(os.path.join(os.path.dirname(oracle.__file__), "oz_oracle.c")).read().splitlines()
    base = ref if rules == "reference" else oracle_standard.source().splitlines()
    got = oracle_scoring.source(rules).splitlines()
    assert len(got) == len(base) + 1
    i = next(k for k, (a, b) in enumerate(zip(base, got)) if a != b)
    assert got[i] == oracle_scoring.WINNER_DRAW.rstrip("\n") and got[i + 1] == base[i]
    j = next(k for k, (a, b) in enumerate(zip(base[i + 1:], got[i + 2:])) if a != b) + i + 1
    assert base[j] == oracle_scoring.REWARD_ANCHOR.rstrip("\n") and got[j + 1] == oracle_scoring.REWARD_DRAW.rstrip("\n")
    assert got[j + 2:] == base[j + 1:] and got[i + 1:j + 1] == base[i:j]
    if rules == "standard":                                      # the standard-rule oracle's own difference: one break
        k = next(k for k, (a, b) in enumerate(zip(ref, base)) if a != b)
        assert base[k].strip().startswith("break;") and base[k + 1:] == ref[k:]
    with pytest.raises(ValueError):
        oracle_scoring.source("quirk")


def _board(n, black_rows, white_rows):
    b = np.zeros((n, n, 2), dtype=np.uint8)
    for r in black_rows:
        b[r, :, 0] = 1
    for r in white_rows:
        b[r, :, 1] = 1
    return b


@pytest.mark.parametrize("rules", ["reference", "standard"])
def test_scoring_oracle_draw_semantics(rules):
    D = oracle_scoring.load(rules)
    full = _board(4, [0, 1], [2, 3])                              # 8 : 8, no empty square
    gapped = _board(8, [0, 1, 2], [4, 5, 6])                      # 24 : 24, rows 3 and 7 empty and unplayable
    won = _board(4, [0, 1, 2], [3])
    for b, pts in ((full, 8), (gapped, 24)):
        assert D.has_finished(b) and oracle.has_finished(b)
        assert D.winner(b) == (2, pts) and oracle.winner(b) == (0, pts)
    assert D.winner(won) == oracle.winner(won) == (0, 12)
    assert D.winner(won[..., ::-1]) == oracle.winner(won[..., ::-1]) == (1, 12)
    # a drawn terminal is worth 0: one move before a full 8 : 8 board, WHITE's only move (3,3) flips (2,2) and ends the
    # game drawn; the search's only edge then has Q 0.0 (python float), where the reference oracle backs up -1
    final = full.copy()
    final[1, 1] = [0, 1]
    final[3, 0] = [1, 0]
    pre = final.copy()
    pre[3, 3] = 0
    pre[2, 2] = [1, 0]
    assert oracle.valid_actions(pre, 1) == [(3, 3)] and np.array_equal(oracle.flip_board(pre, 1, 3, 3), final)
    assert D.has_finished(final) and D.winner(final) == (2, 8)
    for M, q in ((D.Mcts(4), 0.0), (oracle.Mcts(4), -1.0)):
        for _ in range(3):
            M.simulate(pre, 1)
        rq, _, rtag = M.node_stats(pre[..., ::-1])
        assert rq[3, 3] == q and rtag[3, 3] == 1 and np.signbit(rq[3, 3]) == np.signbit(q)


def _drawn_record(n=6, k=5):
    rng = np.random.default_rng(3)
    rec = {"n_moves": np.array([k, k], dtype=np.int32), "winner": np.array([2, 1], dtype=np.int32),
           "black": rng.integers(0, 2 ** 36, (2, 64), dtype=np.uint64), "white": rng.integers(0, 2 ** 36, (2, 64), dtype=np.uint64),
           "action": rng.integers(0, n, (2, 64)).astype(np.uint8) * 9, "player": (np.arange(64)[None, :] % 2).repeat(2, 0).astype(np.uint8)}
    return rec


def test_examples_of_a_drawn_game_have_z_zero():
    from othellozero_b200 import selfplay
    n = 6
    rec = _drawn_record(n)
    batch = selfplay.records_to_examples_batch(rec, n)
    for g in range(2):
        single = selfplay.records_to_examples(rec, g, n)
        assert len(single) == len(batch[g]) == 8 * 5
        for (b1, p1, z1), (b2, p2, z2) in zip(single, batch[g]):
            assert np.array_equal(b1, b2) and np.array_equal(p1, p2) and z1 == z2
    assert all(z == 0 for _, _, z in batch[0])
    assert [z for _, _, z in batch[1][::8]] == [-1, 1, -1, 1, -1]   # WHITE won: +1 where WHITE (player 1) moved


def test_packed_rows_carry_winner_two_to_z_zero():
    from othellozero_b200 import dist, iteration
    n = 6
    rec = _drawn_record(n)
    rows = dist.pack_records(rec)
    assert rows.shape == (10, 3) and ((rows[:, 2] >> np.uint64(16)) & np.uint64(0xFF)).tolist() == [2] * 5 + [1] * 5
    black, white, action, z = iteration.unpack_rows(rows)
    assert z.tolist() == [0] * 5 + [-1, 1, -1, 1, -1]
    boards, policies, zz = iteration.training_arrays(rows, n)
    assert boards.shape == (80, n, n, 2) and zz.dtype == np.float32
    assert (zz[:40] == 0).all() and not np.signbit(zz[:40]).any() and set(zz[40:].tolist()) == {-1.0, 1.0}


def test_train_accepts_z_zero():
    from othellozero_b200 import dist, iteration, net as oznet, train
    n, Ch = 6, 128
    rows = dist.pack_records(_drawn_record(n))
    arrays = iteration.training_arrays(rows[:5], n)                # the drawn game only: every target is z = 0
    assert (arrays[2] == 0).all()
    blob = oznet.init_weights(n, Ch, seed=1)
    new, hist = train.train_blob(blob, arrays, n, Ch, epochs=1, batch_size=8, device="cpu", seed=0, ddp=False)
    assert new.shape == blob.shape and np.isfinite(new).all() and np.isfinite(np.array(hist)).all()


def test_iteration_config_and_cli_take_scoring(monkeypatch):
    from othellozero_b200 import iteration
    assert iteration.IterationConfig().scoring == "reference"
    with pytest.raises(SystemExit):
        iteration.main(["--scoring", "tournament"])
    seen = {}

    class Stop(Exception):
        pass

    def fake_trainer(cfg):
        seen["cfg"] = cfg
        raise Stop

    monkeypatch.setattr(iteration, "Trainer", fake_trainer)
    with pytest.raises(Stop):
        iteration.main(["--scoring", "standard", "--rules", "standard"])
    assert seen["cfg"].scoring == "standard" and seen["cfg"].rules == "standard"


def test_game_classes_carry_the_scoring():
    from othellozero_b200.othello import OthelloGame, StandardOthelloGame, game_class
    assert game_class() is OthelloGame and game_class("standard") is StandardOthelloGame
    assert game_class("reference", "reference") is OthelloGame
    assert game_class("standard", "reference") is StandardOthelloGame
    for rules, base in (("reference", OthelloGame), ("standard", StandardOthelloGame)):
        cls = game_class(rules, "standard")
        assert cls is game_class(rules, "standard") and issubclass(cls, base)
        assert cls.rules == rules and cls.scoring == "standard"
    assert OthelloGame.scoring == StandardOthelloGame.scoring == "reference"
