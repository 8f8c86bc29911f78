"""The CPU oracle under standard scoring (a finished game with equal disc counts is a draw): the parity target of the
draw-scoring tests, under either rule set.

The oracle (oracle/oz_oracle.c) restates the reference, whose winner is max() over {BLACK, WHITE}: a draw goes to BLACK.
Standard scoring changes two statements and nothing else (rules, passes, the end of the game, the search and the episode
driver are shared):
  - orc_winner returns 2 on equal counts (the engine's OZ_WINNER_DRAW), before the `k0 >= k1` test;
  - the terminal reward of simulate_rec maps winner 2 to the integer 0 (a draw is worth nothing to either side).
So this module builds the oracle's own source - for rules="standard" the standard-rule oracle's source
(tests/oracle_standard.py), i.e. the same file with the flip walk's `break` - with those two statements patched at
anchors that must occur exactly once, compiles it with the oracle's own Makefile and binds it with the oracle package's
own Python wrappers.

    import oracle_scoring
    D = oracle_scoring.load("reference")   # reference rules, standard scoring; same API as `oracle`
    S = oracle_scoring.load("standard")    # standard rules, standard scoring
"""
import importlib.util
import os
import shutil
import subprocess
import tempfile

import oracle_standard

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
RULES = ("reference", "standard")

# (anchor, replacement): orc_winner ...
WINNER_ANCHOR = "    if (k0 >= k1) { if (pts) *pts = k0; return 0; }\n"
WINNER_DRAW = "    if (k0 == k1) { if (pts) *pts = k0; return 2; } /* standard scoring: equal counts are a draw */\n"
# ... and the terminal reward of simulate_rec
REWARD_ANCHOR = "        orc_val r; r.is_int = 1; r.i = (orc_winner(state, n, NULL) == 0) ? 1 : -1; r.f = (float)r.i;\n"
REWARD_DRAW = ("        orc_val r; r.is_int = 1; { int w = orc_winner(state, n, NULL); r.i = (w == 0) ? 1 : (w == 2) ? 0 : -1; }"
               " r.f = (float)r.i; /* standard scoring: a draw is 0 */\n")
PATCHES = ((WINNER_ANCHOR, WINNER_DRAW + WINNER_ANCHOR), (REWARD_ANCHOR, REWARD_DRAW))

_mods = {}


def so_path(rules: str) -> str:
    return os.path.join(HERE, f"_oracle_scoring_{rules}.so")


def base_source(rules: str) -> str:
    """The source the scoring patches apply to: the oracle's, or the standard-rule oracle's."""
    if rules not in RULES:
        raise ValueError(f"rules must be one of {RULES}, got {rules!r}")
    if rules == "standard":
        return oracle_standard.source()
    return open(os.path.join(ORACLE, "oz_oracle.c")).read()


def source(rules: str = "reference") -> str:
    src = base_source(rules)
    for anchor, replacement in PATCHES:
        if src.count(anchor) != 1:
            raise RuntimeError(f"oracle/oz_oracle.c: the scoring anchor {anchor.strip()!r} is not unique")
        src = src.replace(anchor, replacement)
    return src


def build(rules: str = "reference", force: bool = False) -> str:
    so = so_path(rules)
    deps = [os.path.join(ORACLE, "oz_oracle.c"), os.path.join(ORACLE, "Makefile"), os.path.abspath(__file__),
            os.path.abspath(oracle_standard.__file__)]
    if not force and os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in deps):
        return so
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "oz_oracle.c"), "w") as f:
            f.write(source(rules))
        # the oracle's own Makefile, so that every build uses the same compiler flags (no FMA contraction)
        subprocess.check_call(["make", "-C", tmp, "-s", "-f", os.path.join(ORACLE, "Makefile"), "liboz_oracle.so"])
        shutil.copyfile(os.path.join(tmp, "liboz_oracle.so"), so + ".tmp")
    os.replace(so + ".tmp", so)
    return so


def load(rules: str = "reference"):
    """The oracle package's module bound to the standard-scoring build for `rules` (a module object of its own; `oracle`
    and the standard-rule oracle are untouched)."""
    if rules not in _mods:
        so = so_path(rules)
        base_source(rules)  # validates `rules`
        spec = importlib.util.spec_from_file_location(f"oracle_scoring_{rules}", os.path.join(ORACLE, "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._SO = so
        mod.build = lambda force=False: build(rules, force)
        _mods[rules] = mod
    return _mods[rules]
