"""Root exploration on one GPU: self-play throughput and game diversity by leg.

Legs (each run `--reps` times, alternated: off, noise, noise+sampled, off, ...), at bench.py's default shape: 8x8,
C = 512 network (init_weights seed 0), 100 simulations per move, `--games` (8192) games from the initial position
through 4096 slots, evaluation cache 2^24, e_greedy 1.0, T = 1, reference rules, scoring and values:
  off              no exploration
  noise            dirichlet_alpha 0.5, dirichlet_fraction 0.25
  noise_sampled    the same with sample_moves 16
The cost of the noise itself is measured without the network, in two tree-only legs with closed-form hash priors
(`--hash-games` (32768) games through 4096 slots, otherwise the same shape), both on the exploring kernel:
  hash_sampled         sample_moves 16 only: the EXPLORE kernel without the noise hook doing any work
  hash_noise_sampled   the same with dirichlet_alpha 0.5, dirichlet_fraction 0.25
Their difference is what drawing and mixing the noise costs the tree kernel, once per move of every game.
These are measurement settings, not recommended defaults.  Reported per leg (medians of the reps): sims/s, games/s,
expansions per simulation (counter nodes / sims), network evaluations per simulation (expansions that neither hit the
evaluation cache nor shared another game's evaluation in the same step), evaluation-cache hits and aliases per simulation,
distinct games (action sequences), distinct positions at plies 10, 20 and 30 (among games that reached them), and the
share of kernel time spent in tree_step_kernel from one extra run of the whole leg under torch.profiler (CUDA activities).

Prints one JSON line with the GPU name and power limit read in the same run.

usage: python tools/explore_ab.py [--reps 3] [--games 8192] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.rules_ab import gpu_info  # noqa: E402
from tools.values_ab import profile_share, run_job  # noqa: E402

G, SIMS, C_ = 4096, 100, 512
LEGS = {"off": (0.0, 0.25, 0), "noise": (0.5, 0.25, 0), "noise_sampled": (0.5, 0.25, 16),
        "hash_sampled": (0.0, 0.25, 16), "hash_noise_sampled": (0.5, 0.25, 16)}
PLIES = (10, 20, 30)


def diversity(rec) -> dict:
    n = np.asarray(rec["n_moves"]).astype(np.int64)
    act = np.asarray(rec["action"])
    out = {"distinct_games": len({act[g, :n[g]].tobytes() for g in range(n.size)})}
    black, white = np.asarray(rec["black"], np.uint64), np.asarray(rec["white"], np.uint64)
    for p in PLIES:
        sel = n > p
        out[f"distinct_positions_ply{p}"] = len(set(zip(black[sel, p].tolist(), white[sel, p].tolist())))
        out[f"games_reaching_ply{p}"] = int(sel.sum())
    return out


def selfplay_leg(E, blob, leg, games, budget_s, device, profile=False) -> dict:
    alpha, eps, m = LEGS[leg]
    hash_leg = leg.startswith("hash")
    e = E.Engine(8, max_games=G, nodes_per_game=SIMS * 61 + 64, prior_mode=E.PRIOR_HASH if hash_leg else E.PRIOR_NET,
                 c_puct=1.0, seed=0, device=device, eval_cache_log2=0 if hash_leg else 24, dirichlet_alpha=alpha,
                 dirichlet_fraction=eps, sample_moves=m)
    try:
        if not hash_leg:
            e.load_weights(blob, C_)
        e.selfplay_begin(games, SIMS, 1.0, 1.0, -1, None, None, None, np.arange(games, dtype=np.uint64))
        e.sync()
        if profile:
            return {"tree_kernel_share": profile_share(lambda: run_job(e, budget_s))}
        t0 = time.perf_counter()
        complete = run_job(e, budget_s)
        dt = time.perf_counter() - t0
        c = e.counters()
        rec = e.selfplay_records()
        done = int((np.asarray(rec["winner"]) >= 0).sum())
    finally:
        e.close()
    sims = max(c["sims"], 1)
    return {"sims_per_s": c["sims"] / dt, "games_per_s": done / dt, "seconds": dt, "complete": complete,
            "games_finished": done, "sims": c["sims"], "moves": c["moves"], "expansions_per_sim": c["nodes"] / sims,
            "net_evals_per_sim": (c["nodes"] - c["cache_hits"] - c["cache_aliases"]) / sims,
            "cache_hits_per_sim": c["cache_hits"] / sims, "cache_aliases_per_sim": c["cache_aliases"] / sims,
            **diversity(rec)}


def games_of(leg, args) -> int:
    return args.hash_games if leg.startswith("hash") else args.games


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--games", type=int, default=8192)
    ap.add_argument("--hash-games", type=int, default=32768)
    ap.add_argument("--leg-budget-s", type=float, default=120.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("explore_ab.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E, net as oznet
    blob = oznet.init_weights(8, C_, seed=0)
    samples = {leg: [] for leg in LEGS}
    for _ in range(args.reps):
        for leg in LEGS:
            samples[leg].append(selfplay_leg(E, blob, leg, games_of(leg, args), args.leg_budget_s, args.device))
    result = {"tool": "explore_ab", **gpu_info(args.device), "reps": args.reps, "games": args.games,
              "hash_games": args.hash_games, "slots": G,
              "sims_per_move": SIMS, "channels": C_, "e_greedy": 1.0, "legs": {}}
    keys = ("sims_per_s", "games_per_s", "seconds", "expansions_per_sim", "net_evals_per_sim", "cache_hits_per_sim",
            "cache_aliases_per_sim")
    for leg, (alpha, eps, m) in LEGS.items():
        s = samples[leg]
        med = {key: statistics.median(x[key] for x in s) for key in keys}
        div = {k: v for k, v in s[0].items() if k.startswith(("distinct", "games_reaching"))}
        assert all({k: x[k] for k in div} == div for x in s), "a leg's games differ between reps"
        share = selfplay_leg(E, blob, leg, games_of(leg, args), args.leg_budget_s, args.device, profile=True)
        result["legs"][leg] = {"dirichlet_alpha": alpha, "dirichlet_fraction": eps, "sample_moves": m, **med, **div,
                               "complete": all(x["complete"] for x in s), **share, "samples": s}
    a, b = result["legs"]["hash_sampled"], result["legs"]["hash_noise_sampled"]
    # seconds per simulation with and without the noise, times the simulations per move: the device time one noised
    # root adds to the whole job, spread over the moves of every game in flight
    result["noise_cost"] = {"tree_only_sims_per_s_ratio": b["sims_per_s"] / a["sims_per_s"],
                            "job_seconds_per_noised_root": (1.0 / b["sims_per_s"] - 1.0 / a["sims_per_s"]) * SIMS}
    result["note"] = ("medians of alternated legs; diversity counts are identical in every rep (the games are "
                      "deterministic); tree_kernel_share = tree_step_kernel time / all kernel time under torch.profiler")
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
