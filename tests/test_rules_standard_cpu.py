"""Standard Othello rules without a GPU: the host build of the bitboard header's standard flip forms against a naive
restatement, the full-tree perft of both rule sets from the host bitboard code and from the oracle (the two rule sets
first differ at ply 7), the oracle's standard playouts against the host's, and the C-ABI's checks of the rules flag."""
import ctypes as C

import numpy as np
import pytest

import oracle
import oracle_standard
from rules_util import (golden_positions, host_play, lib, naive_flips, random_positions, standard_playout_positions)

PERFT_STANDARD = {8: [4, 12, 56, 244, 1396, 8200, 55092, 390216], 6: [4, 12, 56, 244, 1364, 7604, 47740, 308716]}
PERFT_REFERENCE_7_8 = {8: [55032, 389164], 6: [47712, 308244]}
S = oracle_standard.load()   # the oracle under standard rules (same API as `oracle`)


@pytest.fixture(scope="module")
def L():
    return lib()


def _check_all_empty_squares(L, n, own, opp):
    empty = [r * 8 + c for r in range(n) for c in range(n) if not ((own | opp) >> (r * 8 + c)) & 1]
    legal = L.bbr_legal(own, opp, n)
    for sq in empty:
        want = naive_flips(own, opp, sq, n)
        assert L.bbr_flip_standard(sq, own, opp) == want, (n, hex(own), hex(opp), sq)
        assert L.bbr_flip_standard_compact(sq, own, opp) == want, (n, hex(own), hex(opp), sq)
        assert bool((legal >> sq) & 1) == (want != 0)        # legal moves are the standard ones under both rule sets


def test_standard_flips_on_golden_positions(L):
    pos = golden_positions()
    assert len(pos) > 50
    for n, own, opp in pos:
        _check_all_empty_squares(L, n, own, opp)


@pytest.mark.parametrize("n", [4, 6, 8])
def test_standard_flips_on_arbitrary_positions(L, n):
    count = 40_000                                            # x 3 board sizes: 120 000 positions
    owns, opps = random_positions(count, n, seed=1000 + n)
    rng = np.random.default_rng(n)
    squares = [r * 8 + c for r in range(n) for c in range(n)]
    differs = 0
    for own, opp in zip(owns, opps):
        empty = [s for s in squares if not ((own | opp) >> s) & 1]
        if not empty:
            continue
        sq = int(rng.choice(empty))
        want = naive_flips(own, opp, sq, n)
        assert L.bbr_flip_standard(sq, own, opp) == want, (n, hex(own), hex(opp), sq)
        assert L.bbr_flip_standard_compact(sq, own, opp) == want, (n, hex(own), hex(opp), sq)
        differs += L.bbr_flip_reference(sq, own, opp) != want
    # the inputs do exercise the flip-through quirk where it exists (it needs 5 squares in a line: not on 4x4)
    assert differs > count // 50 if n >= 6 else differs == 0


@pytest.mark.parametrize("n", [4, 6, 8])
def test_standard_flips_along_standard_playouts(L, n):
    pos = standard_playout_positions(L, n, games=60, seed=7 + n)
    assert len(pos) > 60 * (n * n - 4) // 2
    for own, opp in pos:
        _check_all_empty_squares(L, n, own, opp)


@pytest.mark.parametrize("n", [6, 8])
def test_host_perft(L, n):
    assert [int(L.bbr_perft(n, d, 1)) for d in range(1, 9)] == PERFT_STANDARD[n]
    assert [int(L.bbr_perft(n, d, 0)) for d in (7, 8)] == PERFT_REFERENCE_7_8[n]


@pytest.mark.parametrize("n", [6, 8])
def test_oracle_perft(n):
    assert [S.perft(n, d) for d in range(1, 9)] == PERFT_STANDARD[n]
    assert [oracle.perft(n, d) for d in (7, 8)] == PERFT_REFERENCE_7_8[n]


def test_oracle_perft_depth_9():
    assert S.perft(8, 9) == 3_005_320


def test_standard_oracle_is_the_oracle_with_one_break():
    """The standard-rule oracle differs from the reference oracle's source by the single `break` of the standard rule."""
    import os
    ref = open(os.path.join(os.path.dirname(oracle.__file__), "oz_oracle.c")).read().splitlines()
    std = oracle_standard.source().splitlines()
    assert len(std) == len(ref) + 1
    i = next(k for k, (a, b) in enumerate(zip(ref, std)) if a != b)
    assert std[i].strip().startswith("break;") and std[i + 1:] == ref[i:]


def test_oracle_standard_flip_squares_match_the_naive_rule():
    for n, own, opp in golden_positions()[:40]:
        board = oracle.bits_to_board(own, opp, n)
        for r in range(n):
            for c in range(n):
                sq = r * 8 + c
                if ((own | opp) >> sq) & 1:
                    continue
                got = S.flip_squares(board, 0, r, c)
                want = naive_flips(own, opp, sq, n)
                assert sum(1 << (i * 8 + j) for i in range(n) for j in range(n) if got[i, j]) == want


@pytest.mark.parametrize("n", [6, 8])
def test_oracle_standard_playouts_equal_the_host_bitboard_ones(L, n):
    """The oracle's engine-RNG playout under standard rules, replayed move by move through the host play_move."""
    differ = 0
    for g in range(40):
        ref = S.playout(n, 3, g)
        own, opp = oracle.board_to_bits(oracle.initial_board(n))
        player = 0
        for a in ref["moves"]:
            own, opp, fl, _ = host_play(L, (a // n) * 8 + a % n, own, opp, n)
            player ^= fl & 1
        black, white = (own, opp) if player == 0 else (opp, own)
        assert (black, white) == (ref["black"], ref["white"])
        differ += oracle.playout(n, 3, g)["moves"] != ref["moves"]
    assert differ > 20


def test_unknown_rules_are_rejected():
    from othellozero_b200 import engine
    with pytest.raises(ValueError):
        engine.apply_moves([1], [2], [3], 8, rules="classic")
    with pytest.raises(ValueError):
        engine.Engine(8, 1, 64, rules="Standard")
    assert engine.board_arg(6, "standard") == 6 | 0x100 and engine.board_arg(6) == 6


def test_abi_rules_flag_validation():
    import torch
    from othellozero_b200 import _lib
    L = _lib.load()
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
        for bad in (8 | 0x200, 8 | 0x100 | 0x200, 0x100, 7 | 0x100, -1):
            assert fn(bad) == _lib.OZ_ERR_INVALID, (fn.__name__, hex(bad))
        with pytest.raises(AssertionError):
            _lib.check(fn(8 | 0x200))
    assert L.oz_net_blob_floats(8 | _lib.RULES_STANDARD, 128) == L.oz_net_blob_floats(8, 128) > 0
    assert L.oz_net_blob_floats(6 | _lib.RULES_STANDARD, 128) == L.oz_net_blob_floats(6, 128) > 0
    assert L.oz_net_blob_floats(8 | 0x200, 128) == -1
    if torch.cuda.is_available():
        return
    for fn in (apply, perft, legal, create):                    # a valid flag reaches the device check: no CPU fallback
        assert fn(8 | _lib.RULES_STANDARD) == _lib.OZ_ERR_CUDA, fn.__name__
        with pytest.raises(_lib.OzError):
            _lib.check(fn(8 | _lib.RULES_STANDARD))
