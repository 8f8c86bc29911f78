"""A/B of the two scorings (a draw counted as a BLACK win vs a draw scored as a draw) on one GPU, in one process, legs
alternated.  The scoring only changes what happens at a finished game, so the expectation is no difference beyond noise.

Legs (each run `--reps` times per scoring, in the order reference, standard, reference, standard, ...), under `--rules`:
  tree       tree_step_kernel with the closed-form hash prior: 4 x 4096 self-play games, 100 simulations per move, through
             4096 slots, wall time to the end of the job -> sims/s (tools/rules_ab.py's tree leg)
  selfplay   device self-play at BASELINE configs[2]'s shape: 8x8, 100 simulations per move, 4096 games in flight (plus a
             queue), C = 512 network, evaluation cache on, games starting at every phase; `--steps` moves timed after
             `--warmup` -> sims/s (tools/rules_ab.py's self-play leg)

The two scorings value drawn terminals differently, so the searches (and the games, in the tree leg) differ slightly; the
rate per simulation is what is compared.  Prints one JSON line with the GPU name and power limit read in the same run.

usage: python tools/scoring_ab.py [--reps 3] [--steps 10] [--warmup 3] [--rules reference] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.rules_ab import gpu_info, selfplay_leg, tree_leg  # noqa: E402

SCORINGS = ("reference", "standard")


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10, help="self-play leg: timed moves (100 engine steps each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rules", default="reference", choices=("reference", "standard"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("scoring_ab.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E, net as oznet
    blob = oznet.init_weights(8, 512, seed=0)
    legs = {"tree": lambda s: tree_leg(E, args.rules, args.device, scoring=s),
            "selfplay": lambda s: selfplay_leg(E, blob, args.rules, args.steps, args.warmup, args.device, scoring=s)}
    samples = {leg: {s: [] for s in SCORINGS} for leg in legs}
    for leg, fn in legs.items():
        for _ in range(args.reps):
            for scoring in SCORINGS:
                samples[leg][scoring].append(fn(scoring))
    result = {"tool": "scoring_ab", **gpu_info(args.device), "rules": args.rules, "reps": args.reps, "legs": {}}
    for leg in legs:
        med = {s: statistics.median(x["sims_per_s"] for x in samples[leg][s]) for s in SCORINGS}
        result["legs"][leg] = {"unit": "sims_per_s", "reference": med["reference"], "standard": med["standard"],
                               "standard_over_reference": med["standard"] / med["reference"], "samples": samples[leg]}
    result["note"] = "medians of alternated legs; the scorings value drawn terminals differently, so sims/s is compared"
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
