"""Root exploration without a GPU: the oracle's Dirichlet sampler (the engine's definition restated in C,
tests/oracle_explore.py) against the Dirichlet distribution, its own log and exp against libm, the proportional draw of
sampled opening moves, argument checks, header constants and the iteration driver's flags."""
import math
import os
import random
import re

import numpy as np
import pytest
from scipy import stats

import oracle_explore

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def X():
    oracle_explore.build()
    return oracle_explore.load()


# ---- 1. the sampler's marginals: Dir(alpha, ..., alpha) over k moves has Beta(alpha, (k-1) alpha) components ----------
@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5])
@pytest.mark.parametrize("k", [2, 10, 33])
def test_dirichlet_marginals(X, alpha, k):
    draws = 3000
    base = oracle_explore.episode_key(11, int(alpha * 1000) + k)
    eta = np.stack([X.dirichlet(alpha, k, oracle_explore.root_key(base, i, 0x1234)) for i in range(draws)])
    assert (eta > 0).all()
    assert np.abs(eta.sum(axis=1) - 1.0).max() <= 1e-15
    beta = stats.beta(alpha, (k - 1) * alpha)
    # A double rounds every value within 2^-54 of 1 to 1.0 (16 % of Beta(0.03, 0.03)), which a KS test against a
    # continuous cdf reads as a jump.  So the KS test takes the values up to 1/2, where doubles resolve both the sample
    # and the cdf, against the conditional cdf F(x) / F(1/2); a binomial test takes how many lie above 1/2.
    half = beta.cdf(0.5)
    for j in sorted({0, k // 2, k - 1}):    # first, middle and last legal move: each is a Beta marginal
        x = eta[:, j]
        lo = x[x <= 0.5]
        assert stats.kstest(lo, lambda t: beta.cdf(t) / half).pvalue > 1e-3, (alpha, k, j)
        assert stats.binomtest(int((x > 0.5).sum()), draws, 1.0 - half).pvalue > 1e-3, (alpha, k, j)
        # mean and variance within 5 standard errors (the variance's from the sample's fourth central moment)
        mean, var = x.mean(), x.var()
        assert abs(mean - beta.mean()) < 5 * math.sqrt(beta.var() / draws), (alpha, k, j)
        m4 = ((x - mean) ** 4).mean()
        assert abs(var - beta.var()) < 5 * math.sqrt((m4 - var * var) / draws), (alpha, k, j)
    # the components are exchangeable: the moves' means agree with 1/k overall
    assert abs(eta.mean() - 1.0 / k) < 1e-12


def test_noise_stream_is_keyed_by_root(X):
    base = oracle_explore.episode_key(5, 17)
    a = X.dirichlet(0.3, 8, oracle_explore.root_key(base, 0x81, 0x42))
    assert np.array_equal(a, X.dirichlet(0.3, 8, oracle_explore.root_key(base, 0x81, 0x42)))
    for other in (oracle_explore.root_key(base, 0x81, 0x43), oracle_explore.root_key(base, 0x80, 0x42),
                  oracle_explore.root_key(oracle_explore.episode_key(5, 18), 0x81, 0x42),
                  oracle_explore.root_key(oracle_explore.episode_key(6, 17), 0x81, 0x42)):
        assert not np.array_equal(a, X.dirichlet(0.3, 8, other))


# ---- 2. the engine's own log and exp ----------------------------------------------------------------------------------
LOG_ULP, EXP_ULP = 2, 1   # the bounds the sampler's log and exp keep against correctly rounded results


def test_log_against_libm(X):
    rng = random.Random(3)
    xs = [rng.uniform(2.0 ** -53, 1.0) for _ in range(40000)]                       # uniforms, the polar s
    xs += [math.exp(rng.uniform(-700.0, 700.0)) for _ in range(20000)]              # any normal
    xs += [1.0 + rng.uniform(-1e-3, 1e-3) for _ in range(20000)]                    # near 1, where log is small
    xs += [2.0 ** -1022, 2.0 ** -53, 0.5, 1.0, 2.0, math.sqrt(0.5), math.sqrt(2.0), 1.7976931348623157e308]
    worst = 0.0
    for x in xs:
        ref = math.log(x)
        got = X.x_log(x)
        worst = max(worst, 0.0 if got == ref else abs(got - ref) / math.ulp(ref))
    assert worst <= LOG_ULP, worst
    assert X.x_log(1.0) == 0.0


def test_exp_against_libm(X):
    rng = random.Random(4)
    xs = [-rng.uniform(0.0, 745.0) * rng.random() ** 3 for _ in range(60000)] + [-rng.uniform(0.0, 1e-6) for _ in range(5000)]
    xs += [0.0, -1.0, -0.5 * math.log(2.0), -708.0, -709.0]
    worst = 0.0
    for x in xs:
        ref = math.exp(x)
        got = X.x_exp(x)
        if ref >= 2.2250738585072014e-308:   # normal results; subnormals are rounded once from a scaled result
            worst = max(worst, 0.0 if got == ref else abs(got - ref) / math.ulp(ref))
        else:
            assert abs(got - ref) <= 2 * math.ulp(ref), x
    assert worst <= EXP_ULP, worst
    assert X.x_exp(0.0) == 1.0 and X.x_exp(-800.0) == 0.0 and X.x_exp(-1e300) == 0.0


def test_gamma_small_alpha_underflow_is_finite(X):
    # alpha << 1: U^(1/alpha) underflows to 0 for most draws; the Dirichlet draw then stays finite and sums to 1
    eta = X.dirichlet(1e-4, 5, 99)
    assert np.isfinite(eta).all() and abs(eta.sum() - 1.0) <= 1e-15


def test_largest_alpha_stays_normalised(X):
    # alpha at its bound (OZ_DIRICHLET_ALPHA_MAX) with the most legal moves a root row holds: the sum does not overflow,
    # eta is the uniform distribution to double precision, and the mixed priors still sum to 1
    eta = X.dirichlet(1e6, 64, 12345)
    assert np.isfinite(eta).all() and abs(eta.sum() - 1.0) <= 1e-14 and np.abs(eta * 64 - 1.0).max() < 0.02


# ---- 3. sampled opening moves: the draw follows the visit counts ------------------------------------------------------
def test_sampled_first_move_follows_visit_counts(X):
    n, sims, games = 6, 40, 4000
    X.set_explore(0.0, 0.25, 1)       # no noise: every game's first root has the same visit counts
    try:
        first = X.execute_episode(n, sims, seed=9, game_id=0, max_moves=1, log_visits=True)
        counts = first["visits"][0].astype(np.int64)
        legal = np.flatnonzero(counts)
        assert len(legal) >= 2 and len(set(counts[legal].tolist())) > 1
        seen = np.zeros(n * n, np.int64)
        for g in range(games):
            out = X.execute_episode(n, sims, seed=9, game_id=g, max_moves=1, log_visits=True)
            assert np.array_equal(out["visits"][0], first["visits"][0])
            seen[out["moves"][0]] += 1
        expected = games * counts[legal] / counts.sum()
        assert seen[legal].sum() == games
        assert stats.chisquare(seen[legal], expected).pvalue > 1e-3
        # without sampling every game plays the first arg-max
        X.set_explore(0.0, 0.25, 0)
        assert X.execute_episode(n, sims, seed=9, game_id=1, max_moves=1)["moves"][0] == int(np.argmax(counts))
    finally:
        X.set_explore(0.0, 0.0, 0)


def test_oracle_without_exploration_is_the_base(X):
    import oracle
    X.set_explore(0.0, 0.0, 0)
    for g in range(3):
        a = X.execute_episode(6, 12, e_greedy=0.9, seed=1, game_id=g, log_visits=True)
        b = oracle.execute_episode(6, 12, e_greedy=0.9, seed=1, game_id=g, log_visits=True)
        assert a["moves"] == b["moves"] and a["winner"] == b["winner"]
        assert all(np.array_equal(x, y) for x, y in zip(a["visits"], b["visits"]))


def test_source_patches_are_unique_on_every_base():
    for rules in ("reference", "standard"):
        for scoring in ("reference", "standard"):
            for values in ("reference", "standard"):
                src = oracle_explore.source(rules, scoring, values)
                assert src.count("orc_x_noise_root(m, s)") == 1 and src.count("x_sampled = 1") == 1
    assert "orc_solve_margin" in oracle_explore.source("standard", "standard", "standard", 6)


# ---- 4. arguments, constants, the driver's flags ------------------------------------------------------------------------
def test_exploration_arg():
    from othellozero_b200 import _lib
    assert _lib.exploration_arg() == (0.0, 0.25, 0)
    assert _lib.exploration_arg(0.3, 0.5, 64) == (0.3, 0.5, 64)
    for bad in (dict(dirichlet_alpha=-0.1), dict(dirichlet_alpha=float("nan")), dict(dirichlet_alpha=float("inf")),
                dict(dirichlet_alpha=1.000001e6), dict(dirichlet_alpha=1e306), dict(dirichlet_fraction=1.5), dict(dirichlet_fraction=-0.01), dict(dirichlet_fraction=float("nan")),
                dict(sample_moves=65), dict(sample_moves=-1), dict(sample_moves=2.0), dict(sample_moves=True),
                dict(dirichlet_alpha="0.3")):
        with pytest.raises(ValueError):
            _lib.exploration_arg(**bad)


def test_header_constants_and_signature():
    from othellozero_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "oz_b200.h")).read()
    assert int(re.search(r"#define OZ_SAMPLE_MOVES_MAX (\d+)", hdr).group(1)) == _lib.SAMPLE_MOVES_MAX == 64
    assert float(re.search(r"#define OZ_DIRICHLET_ALPHA_MAX (\S+)", hdr).group(1)) == _lib.DIRICHLET_ALPHA_MAX == 1e6
    assert _lib.exploration_arg(1e6)[0] == 1e6
    assert "int oz_search_set_exploration(oz_engine* e, double alpha, double fraction, int32_t sample_moves);" in hdr
    assert "oz_search_set_exploration" in _lib.SIGNATURES
    assert "DRAW_SAMPLE_MOVE = 3u" in open(os.path.join(ROOT, "othellozero_b200", "csrc", "oz_bitboard.cuh")).read()


def test_python_entry_points_take_the_options():
    import inspect
    from othellozero_b200 import arena, engine, iteration, mcts, selfplay
    for fn in (engine.Engine.__init__, selfplay.SelfPlay.__init__, selfplay.execute_episodes, selfplay.make_b200_worker):
        p = inspect.signature(fn).parameters
        assert p["dirichlet_alpha"].default == 0.0 and p["dirichlet_fraction"].default == 0.25
        assert p["sample_moves"].default == 0
    p = inspect.signature(mcts.OthelloMCTS.__init__).parameters
    assert p["dirichlet_alpha"].default == 0.0 and p["dirichlet_fraction"].default == 0.25
    for fn in (arena.pit, arena.duels_between_neural_networks, arena.evaluate_neural_network):
        assert "dirichlet_alpha" not in inspect.signature(fn).parameters   # the arena never explores
    cfg = iteration.IterationConfig()
    assert (cfg.dirichlet_alpha, cfg.dirichlet_fraction, cfg.sample_moves) == (0.0, 0.25, 0)
    with pytest.raises(ValueError):
        selfplay.make_b200_worker(dirichlet_alpha=-1.0)


@pytest.mark.parametrize("argv", [["--dirichlet-alpha", "-0.5"], ["--dirichlet-fraction", "1.5"],
                                  ["--sample-moves", "65"], ["--dirichlet-alpha", "nan"]])
def test_cli_rejects_bad_exploration(argv, capsys):
    from othellozero_b200 import iteration
    with pytest.raises(SystemExit) as ex:
        iteration.main(argv)
    assert ex.value.code == 2
    err = capsys.readouterr().err
    assert "dirichlet" in err or "sample_moves" in err


def test_cli_help_lists_the_flags(capsys):
    from othellozero_b200 import iteration
    with pytest.raises(SystemExit):
        iteration.main(["--help"])
    out = capsys.readouterr().out
    for flag in ("--dirichlet-alpha", "--dirichlet-fraction", "--sample-moves"):
        assert flag in out
    assert "self-play only" in out
