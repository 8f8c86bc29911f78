"""The CPU oracle with root exploration: Dirichlet noise on each root's priors, once per node, and self-play opening
moves drawn in proportion to the root visit counts.  The parity target of the exploration tests, over any rules /
scoring / values base.

The engine's definition (include/oz_b200.h, DESIGN.md 15) restated in C and patched into the oracle's source at anchors
that must occur exactly once:
  - the sampler (uniforms, the engine's own log and exp, the polar normal, Marsaglia-Tsang gamma, the Dirichlet draw)
    and the mix, inserted before orc_mcts_simulate;
  - a per-node flag (orc_node.noised) and a per-search noise key (orc_mcts.x_base / x_on);
  - the "noise the root once" hook at the start of orc_mcts_simulate: a root that has a node and no flag gets its noise;
  - the proportional draw in orc_execute_episode, before the temperature-0 tie draw, which it replaces, as it replaces
    the first arg-max (the e_greedy coin still applies).
Every floating-point operation is a plain IEEE +, -, *, / or sqrt, and the oracle's Makefile compiles without FMA
contraction, so the noise is the device's bit for bit.  alpha, the fraction and M are globals of the build
(set_explore); the search API keys its noise with mcts_explore_key(m, seed, game_id), the episode driver with its own
(seed, game id).

    import oracle_explore
    X = oracle_explore.load("standard", "standard", "standard")   # rules, scoring, values (, K)
    X.set_explore(0.3, 0.25, 8)
"""
import ctypes as C
import importlib.util
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_scoring
import oracle_solver
import oracle_standard
import oracle_values

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
VALUES = ("reference", "standard")

NODE_ANCHOR = "    float v;\n} orc_node;\n"
NODE = "    float v;\n    int noised; /* root exploration: the node's noise is mixed in (it has served as a root) */\n} orc_node;\n"
MCTS_ANCHOR = "    int max_depth;\n} orc_mcts;\n"
MCTS = ("    int max_depth;\n    uint64_t x_base; /* root exploration: episode_key(seed, game id) of the noise stream */\n"
        "    int x_on;\n} orc_mcts;\n")
SIM_ANCHOR = "/* OthelloMCTS.simulate(state, player), othelo_mcts.py:22-26. player: 0=BLACK,1=WHITE. */\n"
HOOK_ANCHOR = "    m->sims++;\n    simulate_rec(m, s, 0);\n"
HOOK = "    if (m->x_on && orc_x_alpha > 0.0) orc_x_noise_root(m, s); /* a root's first descent: its noise, once */\n"
KEY_ANCHOR = "    uint64_t base = orc_episode_key(seed, game_id);\n"
KEY = "    m->x_base = base; m->x_on = 1;\n"
TIE_ANCHOR = "        if (temperature == 0) { /* othelo_mcts.py:58-61: one-hot on random.choice(bests) */\n"
SAMPLE = """        int x_sampled = 0;
        if (p < orc_x_moves) { /* root exploration: the move is drawn in proportion to the visit counts */
            int cnt[ORC_MAXSQ], xa[ORC_MAXSQ], tot = 0, run = 0, pick = -1;
            orc_mcts_visits(m, canon, cnt);
            int xk = orc_valid_actions(canon, n, 0, xa);
            for (int i = 0; i < xk; ++i) tot += cnt[xa[i]];
            if (tot > 0) {
                uint32_t u = pick_index(orc_episode_draw(base, p, 3), (uint32_t)tot);
                for (int i = 0; i < xk && pick < 0; ++i) { run += cnt[xa[i]]; if ((uint32_t)run > u) pick = xa[i]; }
                for (int i = 0; i < nsq; ++i) policy[i] = (i == pick) ? 1.0 : 0.0;
                x_sampled = 1;
            }
        }
        if (!x_sampled && temperature == 0) { /* othelo_mcts.py:58-61: one-hot on random.choice(bests) */
"""

SAMPLER = r"""
/* ---- root exploration (tests/oracle_explore.py): the engine's Dirichlet root noise, restated ---- */
static double orc_x_alpha = 0.0, orc_x_eps = 0.0;
static int orc_x_moves = 0;
void orc_x_set(double alpha, double eps, int moves) { orc_x_alpha = alpha; orc_x_eps = eps; orc_x_moves = moves; }

static double orc_x_uniform(uint64_t w) { return (double)((w >> 11) + 1ull) * (1.0 / 9007199254740992.0); }

double orc_x_log(double x) {
    uint64_t b;
    memcpy(&b, &x, 8);
    int e = (int)((b >> 52) & 0x7ffull) - 1023;
    b = (b & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull;
    if (b > 0x3FF6A09E667F3BCDull) { b -= 0x0010000000000000ull; ++e; }
    double m;
    memcpy(&m, &b, 8);
    double f = m - 1.0;
    double s = f / (2.0 + f);
    double z = s * s;
    double p = 0.08695652173913043;
    p = p * z + 0.09523809523809523;
    p = p * z + 0.10526315789473684;
    p = p * z + 0.11764705882352941;
    p = p * z + 0.13333333333333333;
    p = p * z + 0.15384615384615385;
    p = p * z + 0.18181818181818182;
    p = p * z + 0.2222222222222222;
    p = p * z + 0.2857142857142857;
    p = p * z + 0.4;
    p = p * z + 0.6666666666666666;
    double lm = 2.0 * s + (s * z) * p;
    return (double)e * 6.93147180369123816490e-01 + (lm + (double)e * 1.90821492927058770002e-10);
}

static double orc_x_pow2(int k) { uint64_t b = (uint64_t)(k + 1023) << 52; double d; memcpy(&d, &b, 8); return d; }

double orc_x_exp(double x) { /* x <= 0 */
    if (x < -746.0) return 0.0;
    double t = x * 1.4426950408889634;
    int k = (int)(t + (t < 0.0 ? -0.5 : 0.5));
    double r = (x - (double)k * 6.93147180369123816490e-01) - (double)k * 1.90821492927058770002e-10;
    double p = 1.6059043836821613e-10;
    p = p * r + 2.08767569878681e-09;
    p = p * r + 2.505210838544172e-08;
    p = p * r + 2.755731922398589e-07;
    p = p * r + 2.7557319223985893e-06;
    p = p * r + 2.48015873015873e-05;
    p = p * r + 0.0001984126984126984;
    p = p * r + 0.001388888888888889;
    p = p * r + 0.008333333333333333;
    p = p * r + 0.041666666666666664;
    p = p * r + 0.16666666666666666;
    p = p * r + 0.5;
    p = p * r + 1.0;
    p = p * r + 1.0;
    if (k >= -1022) return p * orc_x_pow2(k);
    p = p * orc_x_pow2(k + 600);
    return p * orc_x_pow2(-600);
}

double orc_x_gamma(double alpha, uint64_t key) {
    uint64_t t = 0;
    double a = alpha < 1.0 ? alpha + 1.0 : alpha;
    double d = a - 0.3333333333333333;
    double c = 1.0 / sqrt(9.0 * d);
    double g = d;
    for (int it = 0; it < 256; ++it) {
        double z = 0.0;
        for (int jt = 0; jt < 256; ++jt) {
            double x = 2.0 * orc_x_uniform(orc_sm64(key + t)) - 1.0;
            double y = 2.0 * orc_x_uniform(orc_sm64(key + t + 1)) - 1.0;
            t += 2;
            double s = x * x + y * y;
            if (s >= 1.0 || s == 0.0) continue;
            z = x * sqrt((-2.0 * orc_x_log(s)) / s);
            break;
        }
        double v = 1.0 + c * z;
        if (v <= 0.0) continue;
        v = (v * v) * v;
        double u = orc_x_uniform(orc_sm64(key + t));
        t += 1;
        double z2 = z * z;
        if (u < 1.0 - (0.0331 * z2) * z2 || orc_x_log(u) < 0.5 * z2 + d * ((1.0 - v) + orc_x_log(v))) {
            g = d * v;
            break;
        }
    }
    if (alpha < 1.0) g = g * orc_x_exp(orc_x_log(orc_x_uniform(orc_sm64(key + t))) / alpha);
    return g;
}

/* eta[0..k) of the root stream rk: g_j = Gamma(alpha) from key sm64(rk + j), eta_j = g_j / (sum in ascending j) */
void orc_x_dirichlet(double alpha, int k, uint64_t rk, double *eta) {
    double g[ORC_MAXSQ];
    for (int j = 0; j < k; ++j) g[j] = orc_x_gamma(alpha, orc_sm64(rk + (uint64_t)j));
    double s = g[0];
    for (int j = 1; j < k; ++j) s = s + g[j];
    for (int j = 0; j < k; ++j) eta[j] = s > 0.0 ? g[j] / s : 1.0 / (double)k;
}

void orc_mcts_x_key(orc_mcts *m, uint64_t seed, uint64_t game_id) { m->x_base = orc_episode_key(seed, game_id); m->x_on = 1; }

/* the root `state` (canonical) gets its noise if it has a node without the flag; a single legal move is only flagged */
static void orc_x_noise_root(orc_mcts *m, const uint8_t *state) {
    int idx = tbl_find(m, state);
    if (idx < 0) return;
    orc_node *nd = &m->nodes[idx];
    if (nd->noised) return;
    nd->noised = 1;
    node_actions(m, nd);
    if (nd->nact < 2) return;
    int n = m->n;
    uint64_t own = 0, opp = 0;
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) {
            if (B_AT(state, n, r, c, 0)) own |= 1ull << (r * 8 + c);
            if (B_AT(state, n, r, c, 1)) opp |= 1ull << (r * 8 + c);
        }
    uint64_t rk = orc_sm64(orc_sm64(m->x_base ^ own) + opp);
    double eta[ORC_MAXSQ];
    orc_x_dirichlet(orc_x_alpha, nd->nact, rk, eta);
    double keep = 1.0 - orc_x_eps;
    for (int i = 0; i < nd->nact; ++i) {
        double a = keep * nd->p[nd->act[i]];
        double b = orc_x_eps * eta[i];
        nd->p[nd->act[i]] = a + b;
    }
}

"""


def _check(rules, scoring, values, k):
    if values not in VALUES:
        raise ValueError(f"values must be one of {VALUES}, got {values!r}")
    if k and values != "standard":
        raise ValueError("K > 0 needs standard values")


def base_source(rules="reference", scoring="reference", values="reference", k=0) -> str:
    """The source the exploration patches apply to."""
    _check(rules, scoring, values, k)
    if values == "standard":
        return oracle_values.source(rules, scoring, k)
    return oracle_values.base_source(rules, scoring)


def patches():
    return [(NODE_ANCHOR, NODE), (MCTS_ANCHOR, MCTS), (SIM_ANCHOR, SAMPLER + SIM_ANCHOR), (HOOK_ANCHOR, HOOK + HOOK_ANCHOR),
            (KEY_ANCHOR, KEY_ANCHOR + KEY), (TIE_ANCHOR, SAMPLE)]


def source(rules="reference", scoring="reference", values="reference", k=0) -> str:
    src = base_source(rules, scoring, values, k)
    for anchor, replacement in patches():
        if src.count(anchor) != 1:
            raise RuntimeError(f"oracle source: the exploration anchor {anchor.strip()!r} is not unique")
        src = src.replace(anchor, replacement)
    return src


def so_path(rules, scoring, values, k) -> str:
    return os.path.join(HERE, f"_oracle_explore_{rules}_{scoring}_{values}_{k}.so")


def build(rules="reference", scoring="reference", values="reference", k=0, force=False) -> str:
    so = so_path(rules, scoring, values, k)
    deps = [os.path.join(ORACLE, "oz_oracle.c"), os.path.join(ORACLE, "Makefile"), os.path.abspath(__file__)] + [
        os.path.abspath(m.__file__) for m in (oracle_standard, oracle_scoring, oracle_solver, oracle_values)]
    if not force and os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in deps):
        return so
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "oz_oracle.c"), "w") as f:
            f.write(source(rules, scoring, values, k))
        # the oracle's own Makefile, so that every build uses the same compiler flags (no FMA contraction)
        subprocess.check_call(["make", "-C", tmp, "-s", "-f", os.path.join(ORACLE, "Makefile"), "liboz_oracle.so"])
        shutil.copyfile(os.path.join(tmp, "liboz_oracle.so"), so + ".tmp")
    os.replace(so + ".tmp", so)
    return so


_mods = {}


def load(rules="reference", scoring="reference", values="reference", k=0):
    """The oracle package's module bound to the exploring build of the base (a module object of its own), plus
    set_explore(alpha, fraction, M), mcts_explore_key(mcts, seed, game_id), x_log, x_exp and dirichlet(alpha, k, rk)."""
    key = (rules, scoring, values, k)
    if key not in _mods:
        _check(rules, scoring, values, k)
        spec = importlib.util.spec_from_file_location(f"oracle_explore_{rules}_{scoring}_{values}_{k}",
                                                      os.path.join(ORACLE, "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._SO = so_path(*key)
        mod.build = lambda force=False: build(*key, force=force)

        def lib():
            L = mod.lib()
            if not hasattr(L, "_x_bound"):
                L.orc_x_set.argtypes = [C.c_double, C.c_double, C.c_int]
                L.orc_x_log.argtypes = [C.c_double]
                L.orc_x_log.restype = C.c_double
                L.orc_x_exp.argtypes = [C.c_double]
                L.orc_x_exp.restype = C.c_double
                L.orc_x_gamma.argtypes = [C.c_double, C.c_uint64]
                L.orc_x_gamma.restype = C.c_double
                L.orc_x_dirichlet.argtypes = [C.c_double, C.c_int, C.c_uint64, C.POINTER(C.c_double)]
                L.orc_mcts_x_key.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
                L._x_bound = True
            return L

        def dirichlet(alpha, k, rk):
            out = np.zeros(k)
            lib().orc_x_dirichlet(float(alpha), int(k), rk & (2**64 - 1), out.ctypes.data_as(C.POINTER(C.c_double)))
            return out

        mod.set_explore = lambda alpha, fraction, moves=0: lib().orc_x_set(float(alpha), float(fraction), int(moves))
        mod.mcts_explore_key = lambda m, seed, game_id: lib().orc_mcts_x_key(m._h, seed & (2**64 - 1), game_id)
        mod.x_log = lambda x: lib().orc_x_log(float(x))
        mod.x_exp = lambda x: lib().orc_x_exp(float(x))
        mod.x_gamma = lambda alpha, key: lib().orc_x_gamma(float(alpha), key & (2**64 - 1))
        mod.dirichlet = dirichlet
        _mods[key] = mod
    return _mods[key]


def episode_key(seed: int, game_id: int) -> int:
    """The engine's episode stream key, sm64(sm64(seed ^ 0x5EEDC01D) + game_id), in Python."""
    return _sm64((_sm64(seed ^ 0x5EEDC01D) + game_id) & (2**64 - 1))


def root_key(base: int, own: int, opp: int) -> int:
    """The noise stream key of a root: sm64(sm64(base ^ own) + opp)."""
    return _sm64((_sm64(base ^ own) + opp) & (2**64 - 1))


def _sm64(x: int) -> int:
    M = 2**64 - 1
    x = (x + 0x9E3779B97F4A7C15) & M
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
    return z ^ (z >> 31)
