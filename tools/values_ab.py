"""Standard search values and leaf solving on one GPU: self-play throughput by leg, and colour-balanced strength matches.

Throughput legs (each run `--reps` times, legs alternated: ref, std0, std6, ..., ref, std0, ...), all under standard rules
and standard scoring, at bench.py's default shape: 8x8, C = 512 network (init_weights seed 0), 100 simulations per move,
`--games` (8192) games from the initial position through 4096 slots, evaluation cache 2^24, e_greedy 0.9, T = 1:
  ref        values="reference"
  stdK       values="standard", solve_leaves=K for K in `--ks` (0 6 8 10 12)
A leg plays the whole job unless it runs past `--leg-budget-s`; then it stops there and reports the part it ran
("complete": false).  Reported per leg (medians of the reps): sims/s, games/s (finished games over the wall time),
network evaluations per simulation (counter nodes / sims), leaves solved, solver positions, and the share of kernel time
spent in tree_step_kernel from one extra run of the whole leg (same budget) under torch.profiler (CUDA activities).

Strength: the same network (init_weights seed 0) plays both sides at 8x8 and 100 simulations per move under standard
rules and scoring, through arena.pit.  `--starts` seeded random openings of 4-8 plies are each played twice, colours
swapped, so every pairing has 2 x starts games.  Pairings: standard values K = 0 against reference values, and standard
values at the recommended K against K = 0.  The recommended K is the largest K of the sweep whose sims/s stays within 10 %
of K = 0's (0 when none does).  Reported: W/D/L of the first side, its score (W + D/2) / games with a 95 % normal interval.

Prints one JSON line with the GPU name and power limit read in the same run.

usage: python tools/values_ab.py [--reps 3] [--games 8192] [--ks 0 6 8 10 12] [--starts 256] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.rules_ab import gpu_info  # noqa: E402

STD = "standard"
G, SIMS, C_ = 4096, 100, 512


def leg_name(values, k):
    return "ref" if values == "reference" else f"std{k}"


def selfplay_leg(E, blob, values, k, games, budget_s, device, profile=False) -> dict:
    e = E.Engine(8, max_games=G, nodes_per_game=SIMS * 61 + 64, prior_mode=E.PRIOR_NET, c_puct=1.0, seed=0,
                 device=device, eval_cache_log2=24, rules=STD, scoring=STD, values=values, solve_leaves=k)
    try:
        e.load_weights(blob, C_)
        e.selfplay_begin(games, SIMS, 1.0, 0.9, -1, None, None, None, np.arange(games, dtype=np.uint64))
        e.sync()
        if profile:
            return {"tree_kernel_share": profile_share(lambda: run_job(e, budget_s))}
        t0 = time.perf_counter()
        complete = run_job(e, budget_s)
        dt = time.perf_counter() - t0
        c, sc = e.counters(), e.solve_counters()
        rec = e.selfplay_records()
        done = int((np.asarray(rec["winner"]) >= 0).sum())
    finally:
        e.close()
    return {"sims_per_s": c["sims"] / dt, "games_per_s": done / dt, "seconds": dt, "complete": complete,
            "games_finished": done, "net_evals_per_sim": c["nodes"] / max(c["sims"], 1), "sims": c["sims"],
            "solved_leaves": sc["solved_leaves"], "solver_nodes": sc["solver_nodes"]}


def run_job(e, budget_s) -> bool:
    """Plays the queued job to its end, or until budget_s has passed (-> False); ends with a device synchronise."""
    t0 = time.perf_counter()
    complete = True
    while e.selfplay_run(SIMS):                    # about one move of every game in flight per call
        if time.perf_counter() - t0 > budget_s:
            complete = False
            break
    e.sync()
    return complete


def profile_share(run) -> float:
    """tree_step_kernel's share of all kernel time while run() plays the whole leg (every game phase)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    tree = total = 0.0
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            d = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            total += d
            if "tree_step_kernel" in ev.name:
                tree += d
    return tree / total if total else float("nan")


def openings(n_starts, seed):
    """Seeded random openings of 4-8 plies under standard rules (the engine's random playouts)."""
    from othellozero_b200 import engine as E
    plies = np.random.default_rng(seed).integers(4, 9, size=n_starts)
    black = np.zeros(n_starts, np.uint64); white = np.zeros(n_starts, np.uint64); player = np.zeros(n_starts, np.int32)
    for p in range(4, 9):
        idx = np.nonzero(plies == p)[0]
        if idx.size:
            out = E.perft_playouts(int(idx.size), 8, seed, first_game_id=p << 32, max_moves=p, rules=STD)
            assert not out["finished"].any()
            black[idx], white[idx], player[idx] = out["black"], out["white"], out["player"]
    return black, white, player


def match(net, a, b, starts, device) -> dict:
    """Side a = (values, K) against side b, every start twice with colours swapped -> W/D/L of a."""
    from othellozero_b200 import arena
    black, white, player = starts
    wdl = np.zeros(3, int)
    for a_black in (True, False):
        vals = (a[0], b[0]) if a_black else (b[0], a[0])
        ks = (a[1], b[1]) if a_black else (b[1], a[1])
        out = arena.pit(8, net, net, SIMS, 1.0, n_games=black.size, device=device, rng=np.random.default_rng(7),
                        start_black=black, start_white=white, start_player=player, rules=STD, scoring=STD,
                        values=vals, solve_leaves=ks)
        w = np.asarray(out["winner"])
        a_code = 0 if a_black else 1
        wdl += [int((w == a_code).sum()), int((w == 2).sum()), int(((w != a_code) & (w != 2)).sum())]
    n = int(wdl.sum())
    score = (wdl[0] + 0.5 * wdl[1]) / n
    x = np.array([1.0] * wdl[0] + [0.5] * wdl[1] + [0.0] * wdl[2])
    half = 1.96 * x.std(ddof=1) / math.sqrt(n) if n > 1 else float("nan")
    return {"a": {"values": a[0], "solve_leaves": a[1]}, "b": {"values": b[0], "solve_leaves": b[1]}, "games": n,
            "wins": int(wdl[0]), "draws": int(wdl[1]), "losses": int(wdl[2]), "score": score,
            "score_95ci": [score - half, score + half]}


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--games", type=int, default=8192)
    ap.add_argument("--ks", type=int, nargs="+", default=[0, 6, 8, 10, 12])
    ap.add_argument("--leg-budget-s", type=float, default=120.0)
    ap.add_argument("--starts", type=int, default=256)
    ap.add_argument("--no-strength", action="store_true")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("values_ab.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E, net as oznet
    from othellozero_b200.net import B200NNet
    blob = oznet.init_weights(8, C_, seed=0)
    legs = [("reference", 0)] + [(STD, k) for k in args.ks]
    samples = {leg_name(*l): [] for l in legs}
    for _ in range(args.reps):
        for values, k in legs:
            samples[leg_name(values, k)].append(selfplay_leg(E, blob, values, k, args.games, args.leg_budget_s,
                                                             args.device))
    result = {"tool": "values_ab", **gpu_info(args.device), "reps": args.reps, "games": args.games, "slots": G,
              "sims_per_move": SIMS, "channels": C_, "rules": STD, "scoring": STD, "legs": {}}
    for values, k in legs:
        name = leg_name(values, k)
        s = samples[name]
        med = {key: statistics.median(x[key] for x in s) for key in ("sims_per_s", "games_per_s", "net_evals_per_sim",
                                                                         "solved_leaves", "solver_nodes", "seconds")}
        share = selfplay_leg(E, blob, values, k, args.games, args.leg_budget_s, args.device, profile=True)
        result["legs"][name] = {"values": values, "solve_leaves": k, **med, "complete": all(x["complete"] for x in s),
                                **share, "samples": s}
    base = result["legs"]["std0"]["sims_per_s"] if "std0" in result["legs"] else None
    rec = 0
    for k in args.ks:
        leg = result["legs"][f"std{k}"]
        if k and base and leg["complete"] and leg["sims_per_s"] >= 0.9 * base:
            rec = max(rec, k)
    result["recommended_k"] = rec
    result["recommended_k_rule"] = "largest K whose self-play sims/s stays within 10 % of K = 0's"
    if not args.no_strength:
        net = B200NNet((8, 8), C_, device=args.device, max_batch=8, blob=blob)
        starts = openings(args.starts, seed=2026)
        t0 = time.perf_counter()
        result["strength"] = [match(net, (STD, 0), ("reference", 0), starts, args.device)]
        if rec:
            result["strength"].append(match(net, (STD, rec), (STD, 0), starts, args.device))
        result["strength_seconds"] = time.perf_counter() - t0
    result["note"] = ("medians of alternated legs; a leg that passed --leg-budget-s reports the part it ran; "
                      "tree_kernel_share = tree_step_kernel time / all kernel time under torch.profiler")
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
