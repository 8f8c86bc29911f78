"""The CPU oracle under standard Othello rules: the parity target of the standard-rule tests.

The oracle (oracle/oz_oracle.c) restates the reference, whose flip walk has no `break` after the bracketing own disc.
Standard Othello is that same walk WITH the break, and nothing else differs (legal moves, passes, the end of the game,
scoring, the search and the episode driver are shared).  So this module builds the oracle's own source with that one
statement inserted - the anchor must occur exactly once, or the build fails - and binds it with the oracle package's own
Python wrappers.  Every other line of the standard-rule oracle is the reference oracle's, pinned by the golden vectors;
its flip rule is pinned by the perft table (tests/test_rules_standard_cpu.py).

    import oracle_standard
    S = oracle_standard.load()          # same API as `oracle`: perft, playout, flip_squares, flip_board, Mcts, ...
"""
import importlib.util
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
SO = os.path.join(HERE, "_oracle_standard.so")

# orc_flip_squares: the own disc that brackets the run yields it ...
ANCHOR = """                for (int i = 0; i < ln; ++i) {
                    if (flip) flip[lr[i] * n + lc[i]] = 1;
                    ++yields;
                }
"""
# ... and under standard rules the walk in this direction ends there
BREAK = "                break; /* standard Othello: the first own disc ends the run */\n"

_mod = None


def source() -> str:
    src = open(os.path.join(ORACLE, "oz_oracle.c")).read()
    if src.count(ANCHOR) != 1:
        raise RuntimeError("oracle/oz_oracle.c: the bracketing-disc anchor of orc_flip_squares is not unique")
    return src.replace(ANCHOR, ANCHOR + BREAK)


def build(force: bool = False) -> str:
    src = os.path.join(ORACLE, "oz_oracle.c")
    deps = [src, os.path.join(ORACLE, "Makefile"), os.path.abspath(__file__)]
    if not force and os.path.exists(SO) and os.path.getmtime(SO) >= max(os.path.getmtime(d) for d in deps):
        return SO
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "oz_oracle.c"), "w") as f:
            f.write(source())
        # the oracle's own Makefile, so that both builds use the same compiler flags (no FMA contraction)
        subprocess.check_call(["make", "-C", tmp, "-s", "-f", os.path.join(ORACLE, "Makefile"), "liboz_oracle.so"])
        shutil.copyfile(os.path.join(tmp, "liboz_oracle.so"), SO + ".tmp")
    os.replace(SO + ".tmp", SO)
    return SO


def load():
    """The oracle package's module bound to the standard-rule build (a second module object, `oracle` is untouched)."""
    global _mod
    if _mod is None:
        spec = importlib.util.spec_from_file_location("oracle_standard_rules", os.path.join(ORACLE, "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._SO = SO
        mod.build = build
        _mod = mod
    return _mod
