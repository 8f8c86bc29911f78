"""Throughput of the exact endgame solver (engine.solve_endgame) on one GPU, and its cost inside a training iteration.

Points: 8x8 positions at 10 and 12 empties by default (14 and 16 on request: at 12 empties a position already takes
about 2e5 nodes on average in value mode and one call of 2^15 positions about 9 s on a B200, and every two more empties
multiply that by roughly ten), taken from perft_playouts (engine-RNG random games) stopped at ply
60 - e, keeping positions with exactly e empties whose mover has a move.  Per point, rule set and mode (value: one work
item per position; per_move: one per legal root move) the call is timed `--reps` times, legs alternated (rules x mode in
turn within each repetition), and the median reported as positions/s and nodes/s with the median call time.  A call
includes its host<->device copies and ends in a synchronise.

Iteration leg: self-play of one BASELINE configs[4]-shaped iteration on one GPU (4096 episodes, 8x8, C = 512 network,
100 simulations per move, e_greedy 0.9, 4096 in flight), then selfplay.solve_record_winners at K = 12 and K = 14 on its
records: the solve_s phase of `iteration --solve-empties K` next to selfplay_s.

Prints one JSON line with the GPU name and power limit read in the same run.

usage: python tools/solve_bench.py [--reps 3] [--points 10,12] [--out FILE]
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

RULES = ("reference", "standard")
MODES = ("value", "per_move")
COUNT = {10: 1 << 16, 12: 1 << 15, 14: 1 << 14, 16: 1 << 14}


def positions(E, e: int, count: int, rules: str, seed: int):
    pp = E.perft_playouts(2 * count, 8, seed=seed, max_moves=60 - e, rules=rules)
    own = np.where(pp["player"] == 0, pp["black"], pp["white"])
    opp = np.where(pp["player"] == 0, pp["white"], pp["black"])
    occ = np.unpackbits((own | opp).view(np.uint8).reshape(-1, 8), axis=1).sum(axis=1)
    keep = np.flatnonzero((64 - occ == e) & (E.legal_moves(own, opp, 8, rules=rules) != 0))[:count]
    if keep.size < count:
        raise SystemExit(f"only {keep.size} positions with {e} empties")
    return own[keep], opp[keep]


def solve_leg(E, own, opp, e: int, rules: str, mode: str) -> dict:
    t0 = time.perf_counter()
    out = E.solve_endgame(own, opp, 8, max_empties=e, per_move=mode == "per_move", rules=rules)
    dt = time.perf_counter() - t0
    nodes = int(out["nodes"].sum())
    return {"call_s": dt, "positions_per_s": own.size / dt, "nodes": nodes, "nodes_per_s": nodes / dt}


def iteration_leg(E, device: int, ks=(12, 14)) -> dict:
    from othellozero_b200 import net as oznet, selfplay
    n, C, episodes = 8, 512, 4096
    blob = oznet.init_weights(n, C, seed=0)
    net = oznet.B200NNet((n, n), C, device=device, max_batch=8, blob=blob)
    sp = selfplay.SelfPlay(n, net, 1.0, max_games=episodes, num_simulations=100, device=device, seed=0)
    t0 = time.perf_counter()
    rec = sp.play(episodes, 1.0, 0.9, game_ids=np.arange(episodes, dtype=np.uint64))
    out = {"episodes": episodes, "selfplay_s": time.perf_counter() - t0, "positions": int(rec["n_moves"].sum())}
    sp.close()
    for k in ks:
        t0 = time.perf_counter()
        w = selfplay.solve_record_winners(rec, n, k, device=device)
        dt = time.perf_counter() - t0
        mask = selfplay.solvable_positions(rec, n, k)
        out[f"K{k}"] = {"solve_s": dt, "solved_positions": int(mask.sum()),
                        "solve_relabelled": int((mask & (w != rec["winner"][:, None])).sum())}
    return out


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--points", default="10,12")
    ap.add_argument("--no-iteration", action="store_true")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("solve_bench.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E
    points = [int(x) for x in args.points.split(",")]
    result = {"tool": "solve_bench", **gpu_info(args.device), "reps": args.reps, "points": {}}
    for e in points:
        data = {r: positions(E, e, COUNT[e], r, seed=e) for r in RULES}
        for r in RULES:   # warm-up: module load, scratch growth
            E.solve_endgame(data[r][0][:256], data[r][1][:256], 8, max_empties=e, per_move=True, rules=r)
        samples = {f"{r}/{m}": [] for r in RULES for m in MODES}
        for _ in range(args.reps):
            for r in RULES:
                for m in MODES:
                    samples[f"{r}/{m}"].append(solve_leg(E, *data[r], e, r, m))
        point = {"positions": COUNT[e]}
        for key, xs in samples.items():
            point[key] = {k: statistics.median(x[k] for x in xs) for k in ("call_s", "positions_per_s", "nodes_per_s")}
            point[key]["nodes"] = xs[0]["nodes"]
            point[key]["call_s_samples"] = [x["call_s"] for x in xs]
        result["points"][str(e)] = point
        print(json.dumps({"empties": e, **point}), file=sys.stderr, flush=True)
    if not args.no_iteration:
        result["iteration"] = iteration_leg(E, args.device)
    result["note"] = ("medians of alternated legs; a call includes its copies; nodes = positions visited (the same for "
                      "every repetition: the search is deterministic)")
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
