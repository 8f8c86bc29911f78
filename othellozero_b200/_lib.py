"""ctypes binding of liboz_b200.so (include/oz_b200.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# OZ_B200_LIB: another build of the same ABI (A/B runs of kernel variants); default = the in-tree library
SO = os.environ.get("OZ_B200_LIB") or os.path.join(HERE, "liboz_b200.so")

OZ_OK, OZ_ERR_INVALID, OZ_ERR_CUDA, OZ_ERR_NOMEM, OZ_ERR_STATE = 0, -1, -2, -3, -4
PRIOR_HASH, PRIOR_HOST, PRIOR_NET = 0, 1, 2
MOVE_SWAPPED, MOVE_PASSED, MOVE_FINISHED = 1, 2, 4
GAME_IDLE, GAME_ACTIVE, GAME_WAIT_LEAF, GAME_FINISHED, GAME_POOL_FULL = 0, 1, 2, 3, 4
RULES_STANDARD = 0x100  # OZ_RULES_STANDARD, OR-ed into a board_size argument
RULES = ("reference", "standard")
SCORING_STANDARD = 0x400  # OZ_SCORING_STANDARD, OR-ed into a board_size argument
SCORINGS = ("reference", "standard")
WINNER_DRAW = 2  # OZ_WINNER_DRAW: self-play winner code of a drawn game under standard scoring
SOLVE_MAX_EMPTIES = 20  # OZ_SOLVE_MAX_EMPTIES: the endgame solver's limit
SOLVE_NONE = -128  # OZ_SOLVE_NONE: not a legal move (move_margin) / not searched (margin)
VALUES = ("reference", "standard")  # OZ_VALUES_REFERENCE / OZ_VALUES_STANDARD: how the search backs values up
SOLVE_LEAVES_MAX = 12  # OZ_SOLVE_LEAVES_MAX: the largest solve_leaves (empties of a leaf the search solves)
DIRICHLET_ALPHA_MAX = 1e6  # OZ_DIRICHLET_ALPHA_MAX: the largest dirichlet_alpha
SAMPLE_MOVES_MAX = 64  # OZ_SAMPLE_MOVES_MAX: the largest sample_moves (opening plies played in proportion to visits)
NET_FP8 = 0x10000  # OZ_NET_FP8, OR-ed into a channels argument
PRECISIONS = ("bf16", "fp8")


def board_arg(board_size: int, rules: str = "reference", scoring: str = "reference") -> int:
    """The C-ABI board_size argument for a rule set: "reference" (the reference's flip rule, the default) or
    "standard" (standard Othello flipping), and a scoring: "reference" (a draw counts as a BLACK win, the default) or
    "standard" (a draw is a draw).  Anything else raises ValueError."""
    if rules not in RULES:
        raise ValueError(f"rules must be one of {RULES}, got {rules!r}")
    if scoring not in SCORINGS:
        raise ValueError(f"scoring must be one of {SCORINGS}, got {scoring!r}")
    return board_size | (RULES_STANDARD if rules == "standard" else 0) | (SCORING_STANDARD if scoring == "standard" else 0)


def values_arg(values: str = "reference", solve_leaves: int = 0, scoring: str = "reference") -> int:
    """The C-ABI values argument of oz_search_set_values: "reference" (negate a child's value at every ply, the
    reference's backup, the default) or "standard" (negate it only when the move swapped the side to move).
    solve_leaves = K in [0, SOLVE_LEAVES_MAX] solves new leaves with at most K empties exactly; K > 0 needs
    values="standard" and scoring="standard".  Anything else raises ValueError."""
    if values not in VALUES:
        raise ValueError(f"values must be one of {VALUES}, got {values!r}")
    if isinstance(solve_leaves, bool) or not isinstance(solve_leaves, int) or not 0 <= solve_leaves <= SOLVE_LEAVES_MAX:
        raise ValueError(f"solve_leaves must be an int in [0, {SOLVE_LEAVES_MAX}], got {solve_leaves!r}")
    if solve_leaves and (values != "standard" or scoring != "standard"):
        raise ValueError("solve_leaves > 0 needs values='standard' and scoring='standard' (under reference scoring a "
                         f"drawn final position is not a function of the margin); got values={values!r}, "
                         f"scoring={scoring!r}")
    return VALUES.index(values)


def exploration_arg(dirichlet_alpha: float = 0.0, dirichlet_fraction: float = 0.25, sample_moves: int = 0):
    """The C-ABI arguments of oz_search_set_exploration: (alpha, fraction, M).  dirichlet_alpha = alpha >= 0 (0: no root
    noise, the default; at most DIRICHLET_ALPHA_MAX) mixes Dirichlet(alpha) noise into each root's priors once, with weight dirichlet_fraction in
    [0, 1]; sample_moves = M in [0, SAMPLE_MOVES_MAX] plays self-play's first M plies in proportion to the root visit
    counts.  Non-finite values and anything out of range raise ValueError."""
    import math
    for name, x in (("dirichlet_alpha", dirichlet_alpha), ("dirichlet_fraction", dirichlet_fraction)):
        if isinstance(x, bool) or not isinstance(x, (int, float)) or not math.isfinite(x):
            raise ValueError(f"{name} must be a finite number, got {x!r}")
    if not 0 <= dirichlet_alpha <= DIRICHLET_ALPHA_MAX:
        raise ValueError(f"dirichlet_alpha must be in [0, {DIRICHLET_ALPHA_MAX:g}], got {dirichlet_alpha!r}")
    if not 0 <= dirichlet_fraction <= 1:
        raise ValueError(f"dirichlet_fraction must be in [0, 1], got {dirichlet_fraction!r}")
    if isinstance(sample_moves, bool) or not isinstance(sample_moves, int) or not 0 <= sample_moves <= SAMPLE_MOVES_MAX:
        raise ValueError(f"sample_moves must be an int in [0, {SAMPLE_MOVES_MAX}], got {sample_moves!r}")
    return float(dirichlet_alpha), float(dirichlet_fraction), int(sample_moves)


def channels_arg(channels: int, precision: str = "bf16") -> int:
    """The C-ABI channels argument of the weight loaders for a network precision: "bf16" (the default) or "fp8" (conv3,
    conv4 and fc1 on e4m3 operands, DESIGN.md 13).  Anything else raises ValueError."""
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")
    return int(channels) | (NET_FP8 if precision == "fp8" else 0)


class EngineConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("board_size", C.c_int32), ("max_games", C.c_int32),
                ("nodes_per_game", C.c_int32), ("prior_mode", C.c_int32), ("log_visits", C.c_int32),
                ("eval_cache_log2", C.c_int32), ("vl_width", C.c_int32), ("c_puct", C.c_double), ("seed", C.c_uint64)]


u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
i8p = C.POINTER(C.c_int8)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/oz_b200.h declares
SIGNATURES = {
    "oz_last_error": (C.c_char_p, []),
    "oz_abi_version": (C.c_int, []),
    "oz_device_count": (C.c_int, [i32p]),
    "oz_rules_legal_moves_host": (C.c_int, [C.c_int32, C.c_int32, u64p, u64p, u64p, C.c_int64]),
    "oz_rules_legal_moves_dev": (C.c_int, [C.c_int32, vp, vp, vp, C.c_int64, vp]),
    "oz_rules_apply_host": (C.c_int, [C.c_int32, C.c_int32, u64p, u64p, i32p, u64p, u64p, u32p, u64p, C.c_int64]),
    "oz_rules_apply_dev": (C.c_int, [C.c_int32, vp, vp, vp, vp, vp, vp, vp, C.c_int64, vp]),
    "oz_rules_score_host": (C.c_int, [C.c_int32, u64p, u64p, i32p, i32p, C.c_int64]),
    "oz_rules_score_dev": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
    "oz_perft_playouts_host": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.c_int64, C.c_int32, u64p,
                                         u64p, u32p, u8p]),
    "oz_perft_playouts_dev": (C.c_int, [C.c_int32, C.c_uint64, C.c_uint64, C.c_int64, C.c_int32, vp, vp, vp, vp, vp]),
    "oz_endgame_solve_host": (C.c_int, [C.c_int32, C.c_int32, u64p, u64p, C.c_int64, C.c_int32, i8p, i8p, u64p]),
    "oz_endgame_solve_dev": (C.c_int, [C.c_int32, vp, vp, C.c_int64, C.c_int32, vp, vp, vp, vp]),
    "oz_engine_create": (C.c_int, [C.POINTER(EngineConfig), C.POINTER(vp)]),
    "oz_engine_destroy": (C.c_int, [vp]),
    "oz_engine_sync": (C.c_int, [vp]),
    "oz_engine_stream": (vp, [vp]),
    "oz_search_reset": (C.c_int, [vp, C.c_int32, u64p, u64p, i32p, u64p]),
    "oz_search_set_roots": (C.c_int, [vp, u64p, u64p, i32p]),
    "oz_search_begin": (C.c_int, [vp, C.c_int32, i32p]),
    "oz_search_continue": (C.c_int, [vp, i32p]),
    "oz_search_get_leaves": (C.c_int, [vp, u64p, u64p, C.c_int32]),
    "oz_search_put_priors": (C.c_int, [vp, f32p, f32p, C.c_int32]),
    "oz_search_get_visits": (C.c_int, [vp, i32p, i32p]),
    "oz_search_get_root_stats": (C.c_int, [vp, C.c_int32, f64p, f64p, i32p]),
    "oz_search_get_status": (C.c_int, [vp, i32p]),
    "oz_engine_counters": (C.c_int, [vp, u64p]),
    "oz_search_set_values": (C.c_int, [vp, C.c_int32, C.c_int32]),
    "oz_search_solve_counters": (C.c_int, [vp, u64p]),
    "oz_search_set_exploration": (C.c_int, [vp, C.c_double, C.c_double, C.c_int32]),
    "oz_selfplay_begin": (C.c_int, [vp, C.c_int32, u64p, u64p, i32p, u64p, C.c_int32, C.c_double, C.c_double,
                                    C.c_int32]),
    "oz_selfplay_run": (C.c_int, [vp, C.c_int32, i32p]),
    "oz_selfplay_get_records": (C.c_int, [vp, u64p, u64p, u8p, u8p, i32p, i32p, i32p]),
    "oz_selfplay_get_positions": (C.c_int, [vp, u64p, u64p, i32p]),
    "oz_net_load_weights": (C.c_int, [vp, f32p, C.c_int64, C.c_int32]),
    "oz_net_load_weights_dev": (C.c_int, [vp, vp, C.c_int64, C.c_int32]),
    "oz_net_blob_floats": (C.c_int64, [C.c_int32, C.c_int32]),
    "oz_net_forward_host": (C.c_int, [vp, u64p, u64p, C.c_int32, f32p, f32p, f32p]),
    "oz_net_forward_dev": (C.c_int, [vp, vp, vp, C.c_int32, vp, vp, vp]),
    "oz_net_get_activation": (C.c_int, [vp, C.c_int32, vp, C.c_int64]),
    "oz_net_fp8_scales": (C.c_int, [vp, f32p]),
    "oz_engine_launches": (C.c_int, [vp, u64p]),
    "oz_net_layer_times": (C.c_int, [vp, f32p]),
    "oz_net_set_timing": (C.c_int, [vp, C.c_int32]),
    "oz_probe_l2_read": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, f64p]),
    "oz_dist_unique_id": (C.c_int, [u8p]),
    "oz_dist_init": (C.c_int, [vp, C.c_int32, C.c_int32, u8p]),
    "oz_dist_destroy": (C.c_int, [vp]),
    "oz_dist_broadcast_weights": (C.c_int, [vp, f32p, C.c_int64, C.c_int32, C.c_int32]),
    "oz_dist_gather_examples": (C.c_int, [vp, u64p, C.c_int64, u64p, C.c_int64, C.POINTER(C.c_int64)]),
}

_lib = None


class OzError(RuntimeError):
    pass


def load():
    """Loads the shared library (building is __graft_entry__.build()'s / othellozero_b200.build's job)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise OzError(f"{SO} is missing: run `python -m othellozero_b200.build` (needs nvcc). "
                          "There is no CPU fallback.")
        L = C.CDLL(SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the ABI is incomplete
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    """Maps C-ABI error codes to the exceptions the reference raises (SURVEY §8b 'Errors')."""
    if rc == OZ_OK:
        return
    msg = load().oz_last_error().decode(errors="replace")
    if rc == OZ_ERR_INVALID:
        raise AssertionError(msg)
    if rc == OZ_ERR_NOMEM:
        raise MemoryError(msg)
    raise OzError(msg)


def ptr(arr, typ):
    return arr.ctypes.data_as(typ) if arr is not None else None
