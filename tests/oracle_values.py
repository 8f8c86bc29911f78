"""The CPU oracle under standard search values, with and without leaf solving: the parity target of the standard-values
tests, on any of the four rule/scoring bases.

The oracle (oracle/oz_oracle.c) restates the reference's MCTS.simulate, which negates the child's value at every ply
although its frame swaps only when the opponent can move.  Standard values change one statement and keep one result:
  - simulate_rec keeps orc_has_actions(next, n, 1) (did the move swap the side to move?) ...
  - ... and negates the value returned by the child once more when it did not (the move passed or finished the game).
With K > 0 leaves are solved: the oracle solver of tests/oracle_solver.py is appended (orc_solve_margin, declared before
simulate_rec), and before tbl_find, at depth >= 1, a state with at most K empties (it is not finished: that test comes
first) returns val_neg of the integer sign(orc_solve_margin(state, n, 0)), like a terminal.
The base source is the oracle's for rules/scoring = reference, the standard-rule oracle's (tests/oracle_standard.py) and
the draw-scoring oracle's (tests/oracle_scoring.py) otherwise.  Every anchor must occur exactly once; the result is
compiled with the oracle's own Makefile and bound with the oracle package's own Python wrappers.

    import oracle_values
    V = oracle_values.load("standard", "standard", 8)   # rules, scoring, K; same API as `oracle`
"""
import importlib.util
import os
import shutil
import subprocess
import tempfile

import oracle_scoring
import oracle_solver
import oracle_standard

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
RULES = ("reference", "standard")
SCORINGS = ("reference", "standard")
SOLVE_LEAVES_MAX = 12

SWAP_ANCHOR = ("    if (orc_has_actions(next, n, 1)) { orc_invert(next, n, tmp); memcpy(next, tmp, ORC_BOARD_BYTES(n)); }\n")
SWAP = ("    int swapped = orc_has_actions(next, n, 1); /* standard values: did the move swap the side to move? */\n"
        "    if (swapped) { orc_invert(next, n, tmp); memcpy(next, tmp, ORC_BOARD_BYTES(n)); }\n")
CALL_ANCHOR = "    orc_val value = simulate_rec(m, next, depth + 1);\n"
NEGATE = "    if (!swapped) value = val_neg(value); /* standard values: the child is in the mover's frame */\n"
DECL_ANCHOR = "static orc_val simulate_rec(orc_mcts *m, const uint8_t *state, int depth) {\n"
DECL = "int orc_solve_margin(const uint8_t *board, int n, int player); /* appended: tests/oracle_solver.py */\n"
LEAF_ANCHOR = "    int idx = tbl_find(m, state);\n"


def leaf(k: int) -> str:
    return ("    if (depth >= 1) { /* standard values: a new leaf with <= K empties is solved, not expanded */\n"
            "        int k0, k1;\n"
            "        orc_points(state, n, &k0, &k1);\n"
            f"        if (nsq - k0 - k1 <= {k}) {{\n"
            "            int s = orc_solve_margin(state, n, 0);\n"
            "            orc_val r; r.is_int = 1; r.i = (s > 0) - (s < 0); r.f = (float)r.i;\n"
            "            return val_neg(r);\n"
            "        }\n"
            "    }\n")


def patches(k: int = 0):
    """(anchor, replacement) pairs of the variant with K = k."""
    out = [(SWAP_ANCHOR, SWAP), (CALL_ANCHOR, CALL_ANCHOR + NEGATE)]
    if k:
        out += [(DECL_ANCHOR, DECL + DECL_ANCHOR), (LEAF_ANCHOR, leaf(k) + LEAF_ANCHOR)]
    return out


def _check(rules, scoring, k):
    if rules not in RULES:
        raise ValueError(f"rules must be one of {RULES}, got {rules!r}")
    if scoring not in SCORINGS:
        raise ValueError(f"scoring must be one of {SCORINGS}, got {scoring!r}")
    if not 0 <= k <= SOLVE_LEAVES_MAX or (k and scoring != "standard"):
        raise ValueError(f"K must be in [0, {SOLVE_LEAVES_MAX}], and 0 unless scoring is standard (got {k})")


def base_source(rules: str = "reference", scoring: str = "reference") -> str:
    """The source the value patches apply to."""
    _check(rules, scoring, 0)
    if scoring == "standard":
        return oracle_scoring.source(rules)
    if rules == "standard":
        return oracle_standard.source()
    return open(os.path.join(ORACLE, "oz_oracle.c")).read()


def source(rules: str = "reference", scoring: str = "reference", k: int = 0) -> str:
    _check(rules, scoring, k)
    src = base_source(rules, scoring)
    for anchor, replacement in patches(k):
        if src.count(anchor) != 1:
            raise RuntimeError(f"oracle source: the values anchor {anchor.strip()!r} is not unique")
        src = src.replace(anchor, replacement)
    return src + oracle_solver.SOLVER if k else src


def so_path(rules: str, scoring: str, k: int) -> str:
    return os.path.join(HERE, f"_oracle_values_{rules}_{scoring}_{k}.so")


def build(rules: str = "reference", scoring: str = "reference", k: int = 0, force: bool = False) -> str:
    so = so_path(rules, scoring, k)
    deps = [os.path.join(ORACLE, "oz_oracle.c"), os.path.join(ORACLE, "Makefile"), os.path.abspath(__file__)] + [
        os.path.abspath(m.__file__) for m in (oracle_standard, oracle_scoring, oracle_solver)]
    if not force and os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in deps):
        return so
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "oz_oracle.c"), "w") as f:
            f.write(source(rules, scoring, k))
        # the oracle's own Makefile, so that every build uses the same compiler flags (no FMA contraction)
        subprocess.check_call(["make", "-C", tmp, "-s", "-f", os.path.join(ORACLE, "Makefile"), "liboz_oracle.so"])
        shutil.copyfile(os.path.join(tmp, "liboz_oracle.so"), so + ".tmp")
    os.replace(so + ".tmp", so)
    return so


_mods = {}


def load(rules: str = "reference", scoring: str = "reference", k: int = 0):
    """The oracle package's module bound to the standard-values build for (rules, scoring, K) (a module object of its
    own; the other oracles are untouched).  With K > 0 it also has solve_margin(board, player) (tests/oracle_solver.py)."""
    key = (rules, scoring, k)
    if key not in _mods:
        _check(rules, scoring, k)
        spec = importlib.util.spec_from_file_location(f"oracle_values_{rules}_{scoring}_{k}",
                                                      os.path.join(ORACLE, "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._SO = so_path(rules, scoring, k)
        mod.build = lambda force=False: build(rules, scoring, k, force)
        if k:
            import ctypes as C

            import numpy as np

            def solve_margin(board, player):
                fn = mod.lib().orc_solve_margin
                fn.argtypes = [C.POINTER(C.c_uint8), C.c_int, C.c_int]
                fn.restype = C.c_int
                return int(fn(mod._u8(mod.as_board(board)), np.asarray(board).shape[0], int(player)))

            mod.solve_margin = solve_margin
        _mods[key] = mod
    return _mods[key]
