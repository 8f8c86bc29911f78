"""Thin Python handle on the C-ABI engine (include/oz_b200.h).  numpy in, numpy out; every
call is a CUDA launch behind `liboz_b200.so` — there is no CPU implementation here."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (PRIOR_HASH, PRIOR_HOST, PRIOR_NET, SCORINGS, SOLVE_MAX_EMPTIES, SOLVE_NONE, WINNER_DRAW, board_arg,
                   channels_arg, check, f32p, f64p, i8p, i32p, ptr, u8p, u32p, u64p)

M64 = (1 << 64) - 1


def _e4m3_values() -> np.ndarray:
    """float32 value of each e4m3 (OCP E4M3FN) byte: 1 sign, 4 exponent (bias 7), 3 mantissa bits; 0x7f / 0xff = NaN."""
    b = np.arange(256)
    e, m = (b >> 3) & 15, b & 7
    mag = np.where(e == 0, m / 8.0 * 2.0 ** -6, (1 + m / 8.0) * 2.0 ** (e - 7))
    v = np.where(b & 128, -mag, mag)
    v[(b & 127) == 127] = np.nan
    return v.astype(np.float32)


E4M3_VALUES = _e4m3_values()


def _u64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.uint64)


def _i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


# ---- stateless rules (Othello/__init__.py) ------------------------------------------------------
def legal_moves(own, opp, board_size: int = 8, device: int = 0, rules: str = "reference") -> np.ndarray:
    """get_player_valid_actions as masks (Othello/__init__.py:208-214). own/opp: uint64 arrays.  Legal moves are the
    same under both rule sets; `rules` is checked and otherwise ignored."""
    bs = board_arg(board_size, rules)
    own, opp = _u64(np.atleast_1d(own)), _u64(np.atleast_1d(opp))
    assert own.shape == opp.shape
    out = np.zeros(own.shape, dtype=np.uint64)
    check(_lib.load().oz_rules_legal_moves_host(device, bs, ptr(own, u64p), ptr(opp, u64p), ptr(out, u64p), own.size))
    return out


def apply_moves(own, opp, sq, board_size: int = 8, device: int = 0, rules: str = "reference"):
    """flip_board_squares + turn logic (Othello/__init__.py:237-247,147-159), with the reference's flip rule or, for
    rules="standard", standard Othello flipping.  Returns (own', opp', flags, next_legal) in the frame of the side to
    move next."""
    bs = board_arg(board_size, rules)
    own, opp, sq = _u64(np.atleast_1d(own)), _u64(np.atleast_1d(opp)), _i32(np.atleast_1d(sq))
    assert own.shape == opp.shape == sq.shape
    o2, p2 = np.zeros_like(own), np.zeros_like(own)
    fl = np.zeros(own.shape, dtype=np.uint32)
    nl = np.zeros_like(own)
    check(_lib.load().oz_rules_apply_host(device, bs, ptr(own, u64p), ptr(opp, u64p), ptr(sq, i32p),
                                          ptr(o2, u64p), ptr(p2, u64p), ptr(fl, u32p), ptr(nl, u64p), own.size))
    return o2, p2, fl, nl


def score(black, white, device: int = 0):
    """get_board_players_points (Othello/__init__.py:258-260) -> (black_points, white_points) int32 arrays."""
    black, white = _u64(np.atleast_1d(black)), _u64(np.atleast_1d(white))
    cb = np.zeros(black.shape, dtype=np.int32)
    cw = np.zeros(black.shape, dtype=np.int32)
    check(_lib.load().oz_rules_score_host(device, ptr(black, u64p), ptr(white, u64p), ptr(cb, i32p), ptr(cw, i32p),
                                          black.size))
    return cb, cw


def perft_playouts(n_games: int, board_size: int = 8, seed: int = 0, first_game_id: int = 0, max_moves: int = -1,
                   want_moves: bool = False, device: int = 0, rules: str = "reference"):
    """Random playouts (agents.py:20-24,71-84) with the engine RNG under `rules`.  Returns dict of arrays."""
    bs = board_arg(board_size, rules)
    black = np.zeros(n_games, dtype=np.uint64)
    white = np.zeros(n_games, dtype=np.uint64)
    info = np.zeros(n_games, dtype=np.uint32)
    moves = np.zeros((n_games, 64), dtype=np.uint8) if want_moves else None
    check(_lib.load().oz_perft_playouts_host(device, bs, seed & M64, first_game_id & M64, n_games, max_moves,
                                             ptr(black, u64p), ptr(white, u64p), ptr(info, u32p), ptr(moves, u8p)))
    return dict(black=black, white=white, **decode_perft_info(info), moves=moves)


def decode_perft_info(info) -> dict:
    """The per-game info word of oz_perft_playouts_*: plies in bits 0-7, side to move in bit 8, finished in bit 9, passes
    in bits 16-31."""
    info = np.asarray(info, dtype=np.uint32)
    return dict(plies=(info & 0xFF).astype(np.int32), player=((info >> 8) & 1).astype(np.int32),
                finished=((info >> 9) & 1).astype(bool), passes=(info >> 16).astype(np.int32))


def solve_endgame(own, opp, board_size: int = 8, max_empties: int = SOLVE_MAX_EMPTIES, per_move: bool = False,
                  device: int = 0, rules: str = "reference") -> dict:
    """Exact endgame solver (oz_endgame_solve_host): the final disc margin own - opp under perfect play by both sides,
    side to move = own, empties left at the end not counted.  Returns dict(margin int8 [n], move_margin int8 [n, 64] by
    square bit or None, nodes uint64 [n]).  per_move=True also solves every legal root move with the full window
    (SOLVE_NONE on squares that are not legal moves; the whole row for a finished position or one whose mover must pass).
    Every position must have at most max_empties (<= SOLVE_MAX_EMPTIES) empties, else AssertionError.  The margin does
    not depend on the scoring: see perfect_play_winner."""
    bs = board_arg(board_size, rules)
    own, opp = _u64(np.atleast_1d(own)), _u64(np.atleast_1d(opp))
    assert own.shape == opp.shape and own.ndim == 1
    margin = np.zeros(own.size, dtype=np.int8)
    move_margin = np.zeros((own.size, 64), dtype=np.int8) if per_move else None
    nodes = np.zeros(own.size, dtype=np.uint64)
    check(_lib.load().oz_endgame_solve_host(device, bs, ptr(own, u64p), ptr(opp, u64p), own.size, int(max_empties),
                                            ptr(margin, i8p), ptr(move_margin, i8p), ptr(nodes, u64p)))
    return dict(margin=margin, move_margin=move_margin, nodes=nodes)


def perfect_play_winner(margin, player, scoring: str = "reference") -> np.ndarray:
    """Winner codes of solved positions (the records' codes: 0 BLACK, 1 WHITE, WINNER_DRAW) from the mover's exact
    margin and colour (player 0 = BLACK): a positive margin is a win for the mover, a negative one for the opponent, and
    margin 0 is a BLACK win under reference scoring (Othello/__init__.py:254-256) and a draw under standard scoring."""
    if scoring not in SCORINGS:
        raise ValueError(f"scoring must be one of {SCORINGS}, got {scoring!r}")
    margin, player = np.asarray(margin).astype(np.int64), np.asarray(player).astype(np.int64)
    even = WINNER_DRAW if scoring == "standard" else 0
    return np.where(margin > 0, player, np.where(margin < 0, 1 - player, even)).astype(np.int32)


def probe_l2_read(megabytes: int = 32, passes: int = 50, device: int = 0) -> float:
    """Measured L2 read bandwidth in GB/s (oz_probe_l2_read): the table gather's roofline denominator."""
    out = C.c_double(0.0)
    check(_lib.load().oz_probe_l2_read(device, megabytes, passes, C.byref(out)))
    return float(out.value)


class Engine:
    """oz_engine handle: node pools + per-game state for `max_games` concurrent games on one GPU.  `rules` is the rule
    set of every simulation and self-play move: "reference" (default) or "standard" Othello flipping.  `scoring` is how a
    finished game with equal disc counts is scored: "reference" (default) counts it as a BLACK win, "standard" as a draw
    (value 0 in the search, winner code 2 in self-play records)."""

    def __init__(self, board_size: int = 8, max_games: int = 1, nodes_per_game: int = 8192,
                 prior_mode: int = PRIOR_HASH, c_puct: float = 1.0, seed: int = 0, device: int = 0,
                 log_visits: bool = False, eval_cache_log2: int = 0, vl_width: int = 1, rules: str = "reference",
                 scoring: str = "reference"):
        bs = board_arg(board_size, rules, scoring)
        self._L = _lib.load()
        self.board_size = board_size
        self.rules = rules
        self.precision, self.channels = "bf16", 0  # of the loaded network (load_weights)
        self.scoring = scoring
        self.nsq = board_size * board_size
        self.max_games = max_games
        self.prior_mode = prior_mode
        self.device = device
        self.log_visits = log_visits
        self.vl_width = max(1, int(vl_width))
        self.max_leaves = max_games * self.vl_width
        cfg = _lib.EngineConfig(device, bs, max_games, nodes_per_game, prior_mode, int(log_visits),
                                int(eval_cache_log2), int(vl_width), float(c_puct), seed & M64)
        h = C.c_void_p()
        check(self._L.oz_engine_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.n_games = self.n_slots = 0

    def close(self):
        if getattr(self, "_h", None):
            self._L.oz_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- search ------------------------------------------------------------------------------
    def reset(self, n_games: int, black=None, white=None, player=None, game_ids=None):
        black, white, player, game_ids = _u64(black), _u64(white), _i32(player), _u64(game_ids)
        check(self._L.oz_search_reset(self._h, n_games, ptr(black, u64p), ptr(white, u64p), ptr(player, i32p),
                                      ptr(game_ids, u64p)))
        self.n_games = self.n_slots = n_games

    def set_roots(self, black, white, player=None):
        black, white, player = _u64(black), _u64(white), _i32(player)
        check(self._L.oz_search_set_roots(self._h, ptr(black, u64p), ptr(white, u64p), ptr(player, i32p)))

    def search(self, num_sims: int, predict_batch=None):
        """num_sims sequential simulations per game.  predict_batch(own, opp) -> (pi [L,N*N] f32, v [L] f32)
        is required in PRIOR_HOST mode."""
        nl = C.c_int32(0)
        check(self._L.oz_search_begin(self._h, num_sims, C.byref(nl)))
        while nl.value > 0:
            if predict_batch is None:
                raise _lib.OzError("engine is in PRIOR_HOST mode: a predict_batch callback is required")
            L = nl.value
            own = np.zeros(L, dtype=np.uint64)
            opp = np.zeros(L, dtype=np.uint64)
            check(self._L.oz_search_get_leaves(self._h, ptr(own, u64p), ptr(opp, u64p), L))
            pi, v = predict_batch(own, opp)
            pi = np.ascontiguousarray(pi, dtype=np.float32).reshape(L, self.nsq)
            v = np.ascontiguousarray(v, dtype=np.float32).reshape(L)
            check(self._L.oz_search_put_priors(self._h, ptr(pi, f32p), ptr(v, f32p), L))
            check(self._L.oz_search_continue(self._h, C.byref(nl)))

    def visits(self):
        """-> (visits [n_games, 64] by square bit r*8+c, ns [n_games])"""
        v = np.zeros((self.n_slots, 64), dtype=np.int32)
        ns = np.zeros(self.n_slots, dtype=np.int32)
        check(self._L.oz_search_get_visits(self._h, ptr(v, i32p), ptr(ns, i32p)))
        return v, ns

    def root_stats(self, game: int = 0):
        q = np.zeros(64)
        p = np.zeros(64)
        tag = np.zeros(64, dtype=np.int32)
        check(self._L.oz_search_get_root_stats(self._h, game, ptr(q, f64p), ptr(p, f64p), ptr(tag, i32p)))
        return q, p, tag

    def status(self):
        s = np.zeros(self.n_slots, dtype=np.int32)
        check(self._L.oz_search_get_status(self._h, ptr(s, i32p)))
        return s

    def counters(self) -> dict:
        c = np.zeros(8, dtype=np.uint64)
        check(self._L.oz_engine_counters(self._h, ptr(c, u64p)))
        names = ["sims", "nodes", "terminal_visits", "cache_hits", "cache_aliases", "max_depth", "transpositions", "moves"]
        return {k: int(x) for k, x in zip(names, c)}

    def launches(self) -> int:
        n = C.c_uint64(0)
        check(self._L.oz_engine_launches(self._h, C.byref(n)))
        return int(n.value)

    def sync(self):
        check(self._L.oz_engine_sync(self._h))

    # -- self-play ---------------------------------------------------------------------------------
    def selfplay_begin(self, n_games: int, num_sims: int, temperature: float = 1.0, e_greedy: float = 1.0,
                       max_moves: int = -1, black=None, white=None, player=None, game_ids=None):
        """n_games may exceed max_games: the first max_games episodes start at once, the others are queued and a slot
        whose episode ends starts the next one (records cover all n_games, indexed by game)."""
        black, white, player, game_ids = _u64(black), _u64(white), _i32(player), _u64(game_ids)
        for a in (black, white, player, game_ids):
            assert a is None or a.size >= n_games, "start arrays must cover every game"

        check(self._L.oz_selfplay_begin(self._h, n_games, ptr(black, u64p), ptr(white, u64p), ptr(player, i32p),
                                        ptr(game_ids, u64p), num_sims, float(temperature), float(e_greedy),
                                        max_moves))
        self.n_games = n_games
        self.n_slots = min(n_games, self.max_games)

    def selfplay_run(self, steps: int = -1) -> int:
        na = C.c_int32(0)
        check(self._L.oz_selfplay_run(self._h, steps, C.byref(na)))
        return na.value

    def selfplay_records(self) -> dict:
        g = self.n_games
        rb = np.zeros((g, 64), dtype=np.uint64)
        rw = np.zeros((g, 64), dtype=np.uint64)
        ra = np.zeros((g, 64), dtype=np.uint8)
        rp = np.zeros((g, 64), dtype=np.uint8)
        nm = np.zeros(g, dtype=np.int32)
        win = np.zeros(g, dtype=np.int32)
        rv = np.zeros((g, 64, 64), dtype=np.int32) if self.log_visits else None
        check(self._L.oz_selfplay_get_records(self._h, ptr(rb, u64p), ptr(rw, u64p), ptr(ra, u8p), ptr(rp, u8p),
                                              ptr(nm, i32p), ptr(win, i32p), ptr(rv, i32p)))
        return dict(black=rb, white=rw, action=ra, player=rp, n_moves=nm, winner=win, visits=rv)

    def positions(self):
        g = self.n_slots
        b = np.zeros(g, dtype=np.uint64)
        w = np.zeros(g, dtype=np.uint64)
        p = np.zeros(g, dtype=np.int32)
        check(self._L.oz_selfplay_get_positions(self._h, ptr(b, u64p), ptr(w, u64p), ptr(p, i32p)))
        return b, w, p

    # -- network -----------------------------------------------------------------------------------
    def load_weights(self, blob: np.ndarray, channels: int, precision: str = "bf16"):
        """`precision`: "bf16" or "fp8" (conv3, conv4, fc1 on e4m3 operands, DESIGN.md 13); fixed by the first load."""
        arg = channels_arg(channels, precision)
        blob = np.ascontiguousarray(blob, dtype=np.float32)
        check(self._L.oz_net_load_weights(self._h, ptr(blob, f32p), blob.size, arg))
        self.precision, self.channels = precision, int(channels)

    def load_weights_dev(self, dev_ptr: int, n_floats: int, channels: int, precision: str = "bf16"):
        check(self._L.oz_net_load_weights_dev(self._h, C.c_void_p(dev_ptr), n_floats, channels_arg(channels, precision)))
        self.precision, self.channels = precision, int(channels)

    def fp8_scales(self) -> dict:
        """Scales of the loaded FP8 network: "act" = [sa_2, sa_3, sa_4] (inputs of conv3, conv4, fc1) and the
        per-output-channel weight scales "conv3", "conv4", "fc1".  A value x is stored as e4m3_rn(x / scale)."""
        C_ = self.channels
        out = np.zeros(3 + 2 * C_ + 1024, dtype=np.float32)
        check(self._L.oz_net_fp8_scales(self._h, ptr(out, f32p)))
        return {"act": out[:3].copy(), "conv3": out[3:3 + C_].copy(), "conv4": out[3 + C_:3 + 2 * C_].copy(),
                "fc1": out[3 + 2 * C_:].copy()}

    def net_forward(self, own, opp, want_logits: bool = True):
        own, opp = _u64(np.atleast_1d(own)), _u64(np.atleast_1d(opp))
        n = own.size
        pi = np.zeros((n, self.nsq), dtype=np.float32)
        lg = np.zeros((n, self.nsq), dtype=np.float32) if want_logits else None
        v = np.zeros(n, dtype=np.float32)
        check(self._L.oz_net_forward_host(self._h, ptr(own, u64p), ptr(opp, u64p), n, ptr(pi, f32p), ptr(lg, f32p),
                                          ptr(v, f32p)))
        return pi, lg, v

    def activation(self, layer: int, n_boards: int, rows: int, channels: int) -> np.ndarray:
        """bf16 activations of the last forward as float32 [n_boards, rows, channels] (debug/tests).  An FP8 network
        stores layers 1..3 as e4m3: those come back decoded, in units of their scale (fp8_scales()["act"][layer - 1])."""
        if self.precision == "fp8" and 1 <= layer <= 3:
            raw8 = np.zeros(n_boards * rows * channels, dtype=np.uint8)
            check(self._L.oz_net_get_activation(self._h, layer, raw8.ctypes.data_as(C.c_void_p), raw8.nbytes))
            return E4M3_VALUES[raw8].reshape(n_boards, rows, channels)
        raw = np.zeros(n_boards * rows * channels, dtype=np.uint16)
        check(self._L.oz_net_get_activation(self._h, layer, raw.ctypes.data_as(C.c_void_p), raw.nbytes))
        return (raw.astype(np.uint32) << 16).view(np.float32).reshape(n_boards, rows, channels)

    def set_timing(self, on: bool):
        check(self._L.oz_net_set_timing(self._h, int(on)))

    def stream(self) -> int:
        return int(self._L.oz_engine_stream(self._h) or 0)

    def load_weights_from_tensor(self, t, channels: int, precision: str = "bf16"):
        """float32 CUDA tensor (e.g. just received by an NCCL broadcast) -> fold + cast on device."""
        assert t.is_cuda and t.dtype.is_floating_point and t.element_size() == 4 and t.is_contiguous()
        self.load_weights_dev(t.data_ptr(), t.numel(), channels, precision)

    # -- dist (NCCL through the C-ABI, oz_dist.cu) ---------------------------------------------------------------
    @staticmethod
    def dist_unique_id() -> bytes:
        """Rank 0: the 128-byte NCCL id to ship to the other ranks (any channel: a pipe, a file, torch.distributed)."""
        buf = np.zeros(128, dtype=np.uint8)
        check(_lib.load().oz_dist_unique_id(ptr(buf, u8p)))
        return buf.tobytes()

    def dist_init(self, rank: int, world: int, unique_id: bytes):
        buf = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
        assert buf.size == 128
        check(self._L.oz_dist_init(self._h, rank, world, ptr(buf, u8p)))

    def dist_broadcast_weights(self, blob, channels: int, root: int = 0, precision: str = "bf16"):
        """C1: `root` passes the float32 blob, the others None; every rank ends with the weights loaded."""
        arg = channels_arg(channels, precision)
        blob = None if blob is None else np.ascontiguousarray(blob, dtype=np.float32)
        n = int(self._L.oz_net_blob_floats(self.board_size, channels))
        check(self._L.oz_dist_broadcast_weights(self._h, ptr(blob, f32p), n, arg, root))
        self.precision, self.channels = precision, int(channels)

    def dist_gather_examples(self, rows: np.ndarray) -> np.ndarray:
        """C2: packed example rows [n, 3] uint64 of this rank -> the concatenation over all ranks, in rank order."""
        rows = np.ascontiguousarray(rows, dtype=np.uint64).reshape(-1, 3)
        total = C.c_int64(0)
        check(self._L.oz_dist_gather_examples(self._h, ptr(rows, u64p) if rows.size else None, rows.shape[0], None, 0,
                                              C.byref(total)))
        out = np.zeros((int(total.value), 3), dtype=np.uint64)
        check(self._L.oz_dist_gather_examples(self._h, ptr(rows, u64p) if rows.size else None, rows.shape[0],
                                              ptr(out, u64p) if out.size else None, out.shape[0], C.byref(total)))
        return out

    def layer_times(self):
        ms = np.zeros(8, dtype=np.float32)
        check(self._L.oz_net_layer_times(self._h, ptr(ms, f32p)))
        return ms
