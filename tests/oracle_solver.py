"""The CPU oracle with an exact endgame solver: the parity target of the endgame-solver tests, under either rule set.

The oracle (oracle/oz_oracle.c) restates the reference's rules by walking squares; the standard-rule oracle
(tests/oracle_standard.py) is the same source with the flip walk's `break`.  This module takes either source and APPENDS
two functions written over the oracle's own orc_game_play / orc_valid_actions / orc_points - no bitboards, so nothing is
shared with the device kernel but the rules they both state:
  - orc_solve_margin(board, n, player): the exact final disc margin (mover minus opponent, empties not counted) under
    perfect play by both sides, by plain alpha-beta negamax;
  - orc_solve_minimax(board, n, player): the same search without pruning, which pins the pruned one at few empties.
Nothing above the appended text changes (a test checks it).  The result is compiled with the oracle's own Makefile and
bound with the oracle package's own Python wrappers, plus solve_margin / solve_minimax / solve_move_margins.

    import oracle_solver
    O = oracle_solver.load("reference")       # same API as `oracle`, plus the solver
    O.solve_margin(board, player)             # board (N,N,2), player 0 = BLACK / 1 = WHITE to move
"""
import ctypes as C
import importlib.util
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_standard

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
RULES = ("reference", "standard")

SOLVER = r"""
/* ------------------------------------------------------------------------- */
/* Exact endgame solver (appended by tests/oracle_solver.py)                  */
/* ------------------------------------------------------------------------- */
/* Value of g from g->player's side: the final disc margin under perfect play.  orc_game_play passes automatically, so
 * a child's side to move is either the opponent (negate) or the same player again (do not).  A finished game is worth
 * its disc difference; a mover without a move (only possible at the root) passes. */
static int orc_solve_rec(const orc_game *g, int alpha, int beta, int prune) {
    int k0, k1;
    if (g->finished) {
        orc_points(g->board, g->n, &k0, &k1);
        return g->player == 0 ? k0 - k1 : k1 - k0;
    }
    int acts[ORC_MAXSQ];
    int k = orc_valid_actions(g->board, g->n, g->player, acts);
    if (k == 0) {
        orc_game h = *g;
        h.player = 1 - g->player;
        if (!orc_has_actions(h.board, h.n, h.player)) {
            orc_points(g->board, g->n, &k0, &k1);
            return g->player == 0 ? k0 - k1 : k1 - k0;
        }
        return -orc_solve_rec(&h, -beta, -alpha, prune);
    }
    int best = -1000;
    for (int i = 0; i < k; ++i) {
        orc_game h = *g;
        orc_game_play(&h, acts[i] / g->n, acts[i] % g->n);
        int same = !h.finished && h.player == g->player;
        int v;
        if (h.finished) {
            orc_points(h.board, h.n, &k0, &k1);
            v = g->player == 0 ? k0 - k1 : k1 - k0;
        } else if (same) {
            v = orc_solve_rec(&h, alpha, beta, prune);
        } else {
            v = -orc_solve_rec(&h, -beta, -alpha, prune);
        }
        if (v > best) best = v;
        if (prune) {
            if (best > alpha) alpha = best;
            if (alpha >= beta) break;
        }
    }
    return best;
}

static int orc_solve_entry(const uint8_t *board, int n, int player, int prune) {
    orc_game g;
    g.n = n;
    memcpy(g.board, board, ORC_BOARD_BYTES(n));
    g.player = player;
    g.round = 1;
    g.finished = orc_has_finished(board, n);
    return orc_solve_rec(&g, -1000, 1000, prune);
}

int orc_solve_margin(const uint8_t *board, int n, int player) { return orc_solve_entry(board, n, player, 1); }
int orc_solve_minimax(const uint8_t *board, int n, int player) { return orc_solve_entry(board, n, player, 0); }
"""

_mods = {}


def so_path(rules: str) -> str:
    return os.path.join(HERE, f"_oracle_solver_{rules}.so")


def base_source(rules: str) -> str:
    """The source the solver is appended to: the oracle's, or the standard-rule oracle's."""
    if rules not in RULES:
        raise ValueError(f"rules must be one of {RULES}, got {rules!r}")
    if rules == "standard":
        return oracle_standard.source()
    return open(os.path.join(ORACLE, "oz_oracle.c")).read()


def source(rules: str = "reference") -> str:
    return base_source(rules) + SOLVER


def build(rules: str = "reference", force: bool = False) -> str:
    so = so_path(rules)
    deps = [os.path.join(ORACLE, "oz_oracle.c"), os.path.join(ORACLE, "Makefile"), os.path.abspath(__file__),
            os.path.abspath(oracle_standard.__file__)]
    if not force and os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in deps):
        return so
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "oz_oracle.c"), "w") as f:
            f.write(source(rules))
        # the oracle's own Makefile, so that every build uses the same compiler flags
        subprocess.check_call(["make", "-C", tmp, "-s", "-f", os.path.join(ORACLE, "Makefile"), "liboz_oracle.so"])
        shutil.copyfile(os.path.join(tmp, "liboz_oracle.so"), so + ".tmp")
    os.replace(so + ".tmp", so)
    return so


def load(rules: str = "reference"):
    """The oracle package's module bound to the solver build for `rules` (a module object of its own), with
    solve_margin(board, player), solve_minimax(board, player) and solve_move_margins(board, player) added."""
    if rules not in _mods:
        so = so_path(rules)
        base_source(rules)  # validates `rules`
        spec = importlib.util.spec_from_file_location(f"oracle_solver_{rules}", os.path.join(ORACLE, "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._SO = so
        mod.build = lambda force=False: build(rules, force)

        def _solver(name):
            fn = getattr(mod.lib(), name)
            fn.argtypes = [C.POINTER(C.c_uint8), C.c_int, C.c_int]
            fn.restype = C.c_int
            return lambda board, player: int(fn(mod._u8(mod.as_board(board)), np.asarray(board).shape[0], int(player)))

        def solve_margin(board, player):
            return _solver("orc_solve_margin")(board, player)

        def solve_minimax(board, player):
            return _solver("orc_solve_minimax")(board, player)

        def solve_move_margins(board, player):
            """{square bit r*8+c: exact margin for the mover after that move} over the mover's legal moves: the child
            is played as orc_game_play does (flip, then the opponent moves unless it has to pass)."""
            b = mod.as_board(board)
            n = b.shape[0]
            out = {}
            for r, c in mod.valid_actions(b, player):
                child = mod.flip_board(b, player, r, c)
                nxt = 1 - player if mod.valid_actions(child, 1 - player) else player
                v = solve_margin(child, nxt)
                out[r * 8 + c] = v if nxt == player else -v
            return out

        mod.solve_margin, mod.solve_minimax, mod.solve_move_margins = solve_margin, solve_minimax, solve_move_margins
        _mods[rules] = mod
    return _mods[rules]
