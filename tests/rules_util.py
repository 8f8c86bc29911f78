"""Standard Othello flipping restated naively (one square at a time along each ray), and inputs for the tests that check
the bitboard forms of it (tests/test_rules_standard_cpu.py, tests/test_gpu_rules_standard.py)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(HERE, "_bb_host_rules.so")
_lib = None
DIRS = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]
M64 = (1 << 64) - 1


def naive_flips(own: int, opp: int, sq: int, n: int) -> int:
    """Standard rule: along each ray, the opponent discs up to the FIRST own disc flip; nothing flips without one."""
    r0, c0 = divmod(sq, 8)
    f = 0
    for dr, dc in DIRS:
        r, c, run = r0 + dr, c0 + dc, 0
        while 0 <= r < n and 0 <= c < n and (opp >> (r * 8 + c)) & 1:
            run |= 1 << (r * 8 + c)
            r, c = r + dr, c + dc
        if run and 0 <= r < n and 0 <= c < n and (own >> (r * 8 + c)) & 1:
            f |= run
    return f


def full_mask(n: int) -> int:
    return sum(1 << (r * 8 + c) for r in range(n) for c in range(n))


def lib():
    """Builds/loads tests/_bb_host_rules.cpp (host build of the product bitboard header's rule-set code)."""
    global _lib
    if _lib is None:
        src = os.path.join(HERE, "_bb_host_rules.cpp")
        hdr = os.path.join(HERE, "..", "othellozero_b200", "csrc", "oz_bitboard.cuh")
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-o", _SO, src])
        L = C.CDLL(_SO)
        u64 = C.c_uint64
        L.bbr_legal.argtypes = [u64, u64, C.c_int]
        L.bbr_legal.restype = u64
        for name in ("bbr_flip_reference", "bbr_flip_standard", "bbr_flip_standard_compact"):
            getattr(L, name).argtypes = [C.c_int, u64, u64]
            getattr(L, name).restype = u64
        L.bbr_play.argtypes = [C.c_int, C.c_int, C.POINTER(u64), C.POINTER(u64), C.c_int, C.POINTER(u64)]
        L.bbr_play.restype = C.c_uint
        L.bbr_perft.argtypes = [C.c_int, C.c_int, C.c_int]
        L.bbr_perft.restype = C.c_uint64
        L.bbr_initial.argtypes = [C.c_int, C.POINTER(u64), C.POINTER(u64)]
        _lib = L
    return _lib


def host_play(L, sq: int, own: int, opp: int, n: int, standard: bool = True):
    """play_move<RULES> on the host -> (own', opp', flags, next_legal) in the frame of the side to move next."""
    o, p, nl = C.c_uint64(own), C.c_uint64(opp), C.c_uint64(0)
    fl = L.bbr_play(int(standard), sq, C.byref(o), C.byref(p), n, C.byref(nl))
    return o.value, p.value, int(fl), nl.value


def golden_positions():
    """(n, own, opp) of every position of tests/golden/rules.json, from both sides."""
    d = json.load(open(os.path.join(HERE, "golden", "rules.json")))
    out = []
    for ns, recs in d.items():
        for r in recs:
            b, w = int(r["b"], 16), int(r["w"], 16)
            out += [(int(ns), b, w), (int(ns), w, b)]
    return out


def random_positions(count: int, n: int, seed: int):
    """Arbitrary (not necessarily reachable) disjoint own/opp pairs on an N x N board, densities varied so that long
    opponent runs, and runs with own discs inside and beyond them, are common."""
    rng = np.random.default_rng(seed)
    sq = np.array([r * 8 + c for r in range(n) for c in range(n)], dtype=np.uint64)
    p_empty = rng.uniform(0.05, 0.6, size=count)
    p_own = rng.uniform(0.1, 0.6, size=count)
    u = rng.random((count, sq.size))
    empty = u < p_empty[:, None]
    own_m = ~empty & (rng.random((count, sq.size)) < p_own[:, None])
    opp_m = ~empty & ~own_m
    bits = np.uint64(1) << sq
    own = (own_m * bits).sum(axis=1, dtype=np.uint64)
    opp = (opp_m * bits).sum(axis=1, dtype=np.uint64)
    return [int(x) for x in own], [int(x) for x in opp]


def standard_playout_positions(L, n: int, games: int, seed: int):
    """Every position (own, opp = side to move first) of `games` uniformly random games under the standard rules."""
    full = full_mask(n)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(games):
        own, opp = _initial(L, n)
        legal = L.bbr_legal(own, opp, n)
        while legal:
            out.append((own, opp))
            moves = [s for s in range(64) if (legal >> s) & 1]
            own, opp, _, legal = host_play(L, int(rng.choice(moves)), own, opp, n)
        assert not (own | opp) & ~full
    return out


def _initial(L, n):
    b, w = C.c_uint64(0), C.c_uint64(0)
    L.bbr_initial(n, C.byref(b), C.byref(w))
    return b.value, w.value
