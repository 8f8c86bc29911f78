"""A/B of the network precisions (bf16 vs FP8 conv3/conv4/fc1, DESIGN.md 13) on one GPU, in one process, legs alternated.

Legs (each run `--reps` times per precision, in the order bf16, fp8, bf16, fp8, ...):
  selfplay   device self-play as bench.py's default line plays it: 8x8, C = 512 (init_weights seed 0), 100 simulations
             per move, 4096 games in flight plus one queued generation, evaluation cache 2^24, the steady-state mix of
             game phases from bench.synthetic_starts(spread=57) with bench's seed and game ids; `--steps` moves timed
             after `--warmup` -> sims/s, plus per-layer times (oz_net_layer_times)
  forward    oz_net_forward_dev over 4096 boards from the same starts, `--forwards` timed after a warm-up -> boards/s,
             plus per-layer times
  load       wall time of oz_net_load_weights (8x8, C = 512) on engines of 1, 8 and 4096 rows.  An FP8 load also
             quantises and runs the calibration set through the bf16 gather, conv3 and conv4 in chunks of the row
             capacity, so its extra cost grows as the capacity shrinks
Also reported: the FP8 conv3's achieved FLOP/s from its per-layer time (2 * 9 * C * C * 36 FLOP per 8x8 board), next
to the data-sheet dense FP8 rate as a reference only, and the GPU name and power limit, read in the same run.

usage: python tools/precision_ab.py [--reps 3] [--steps 10] [--warmup 3] [--forwards 50] [--out FILE]
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

import bench  # noqa: E402
from tools.rules_ab import gpu_info  # noqa: E402

PRECISIONS = ("bf16", "fp8")
LAYERS = ("conv1", "gather", "conv3", "conv4", "fc1", "fc2", "heads")
G, SIMS, C_ = 4096, 100, 512
LOAD_ROWS = (1, 8, 4096)
FP8_DENSE_DATASHEET_TFLOPS = 4500.0  # HGX B200 data sheet, one GPU, dense: a reference, not a reachable figure


def layer_ms(e) -> dict:
    ms = e.layer_times()
    return {name: float(ms[i]) for i, name in enumerate(LAYERS)} | {"forwards_averaged": int(ms[7])}


def selfplay_leg(E, blob, starts, precision, steps, warmup, device) -> dict:
    b, w, p = starts
    total = b.size
    e = E.Engine(8, max_games=G, nodes_per_game=SIMS * 61 + 64, prior_mode=E.PRIOR_NET, c_puct=1.0, seed=0,
                 device=device, eval_cache_log2=24)
    try:
        e.load_weights(blob, C_, precision)
        e.selfplay_begin(total, SIMS, 1.0, 0.9, -1, b, w, p, np.arange(total, dtype=np.uint64))  # bench's first ids
        for _ in range(warmup):
            e.selfplay_run(SIMS)
        e.sync()
        e.set_timing(True)
        e.layer_times()  # drop what the warm-up recorded
        c0 = e.counters()
        t0 = time.perf_counter()
        for _ in range(steps):
            e.selfplay_run(SIMS)
        e.sync()
        s = time.perf_counter() - t0
        c1 = e.counters()
        d = {k: c1[k] - c0[k] for k in ("sims", "moves", "nodes", "cache_hits")}
        return {"s": s, **d, "sims_per_s": d["sims"] / s, "layer_ms": layer_ms(e)}
    finally:
        e.close()


def forward_leg(E, blob, starts, precision, forwards, device) -> dict:
    import torch
    b, w, p = starts
    own = np.where(p[:G] == 0, b[:G], w[:G]).astype(np.uint64)
    opp = np.where(p[:G] == 0, w[:G], b[:G]).astype(np.uint64)
    e = E.Engine(8, max_games=G, nodes_per_game=2, prior_mode=E.PRIOR_NET, device=device)
    try:
        e.load_weights(blob, C_, precision)
        dev = torch.device("cuda", device)
        d_own = torch.as_tensor(own.view(np.int64), device=dev)
        d_opp = torch.as_tensor(opp.view(np.int64), device=dev)
        pi = torch.empty((G, 64), dtype=torch.float32, device=dev)
        v = torch.empty(G, dtype=torch.float32, device=dev)
        L = e._L

        def fwd():
            E.check(L.oz_net_forward_dev(e._h, d_own.data_ptr(), d_opp.data_ptr(), G, pi.data_ptr(), None, v.data_ptr()))
        for _ in range(5):
            fwd()
        e.set_timing(True)
        e.layer_times()
        t0 = time.perf_counter()
        for _ in range(forwards):
            fwd()
        s = time.perf_counter() - t0  # oz_net_forward_dev synchronises
        lm = layer_ms(e)
        out = {"s": s, "boards_per_s": G * forwards / s, "layer_ms": lm}
        if precision == "fp8":
            out["fp8_scales_act"] = [float(x) for x in e.fp8_scales()["act"]]
        return out
    finally:
        e.close()


def load_leg(E, blob, precision, device) -> dict:
    """Seconds per oz_net_load_weights at each row capacity: the second of two loads on one engine (the first also
    allocates)."""
    out = {}
    for rows in LOAD_ROWS:
        e = E.Engine(8, max_games=rows, nodes_per_game=2, prior_mode=E.PRIOR_NET, device=device)
        try:
            e.load_weights(blob, C_, precision)
            t0 = time.perf_counter()
            e.load_weights(blob, C_, precision)
            out[str(rows)] = time.perf_counter() - t0
        finally:
            e.close()
    return out


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10, help="self-play leg: timed moves (100 engine steps each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--forwards", type=int, default=50)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("precision_ab.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E, net as oznet
    blob = oznet.init_weights(8, C_, seed=0)
    starts = bench.synthetic_starts(E, 2 * G, 0, 0, args.device, spread=57)
    legs = {"selfplay": lambda pr: selfplay_leg(E, blob, starts, pr, args.steps, args.warmup, args.device),
            "forward": lambda pr: forward_leg(E, blob, starts, pr, args.forwards, args.device)}
    rate = {"selfplay": "sims_per_s", "forward": "boards_per_s"}
    samples = {leg: {pr: [] for pr in PRECISIONS} for leg in legs}
    for leg, fn in legs.items():
        for _ in range(args.reps):
            for pr in PRECISIONS:
                samples[leg][pr].append(fn(pr))
    result = {"tool": "precision_ab", **gpu_info(args.device), "shape": {"n": 8, "C": C_, "games": G, "sims": SIMS},
              "reps": args.reps, "legs": {}}
    for leg in legs:
        med = {pr: statistics.median(x[rate[leg]] for x in samples[leg][pr]) for pr in PRECISIONS}
        lay = {pr: {k: statistics.median(x["layer_ms"][k] for x in samples[leg][pr]) for k in LAYERS} for pr in PRECISIONS}
        result["legs"][leg] = {"unit": rate[leg], "bf16": med["bf16"], "fp8": med["fp8"], "fp8_over_bf16": med["fp8"] / med["bf16"],
                               "layer_ms_median": lay, "samples": samples[leg]}
    fl = samples["forward"]
    conv3_flop = 2.0 * 9 * C_ * C_ * 36 * G
    conv3_ms = statistics.median(x["layer_ms"]["conv3"] for x in fl["fp8"])
    result["fp8_conv3_achieved_tflops"] = conv3_flop / (conv3_ms * 1e-3) / 1e12 if conv3_ms > 0 else None
    result["bf16_conv3_achieved_tflops"] = conv3_flop / (statistics.median(x["layer_ms"]["conv3"] for x in fl["bf16"]) * 1e-3) / 1e12
    result["fp8_dense_datasheet_tflops_reference_only"] = FP8_DENSE_DATASHEET_TFLOPS
    loads = {pr: [] for pr in PRECISIONS}
    for _ in range(args.reps):
        for pr in PRECISIONS:
            loads[pr].append(load_leg(E, blob, pr, args.device))
    result["load_s_median_by_rows"] = {pr: {r: statistics.median(x[r] for x in loads[pr]) for r in map(str, LOAD_ROWS)}
                                       for pr in PRECISIONS}
    result["load_s_samples"] = loads
    result["note"] = ("medians of alternated legs; per-layer times are CUDA events on every 16th forward; conv3 FLOP/s from "
                      "the forward leg's per-layer time; load_s = oz_net_load_weights wall time (a reload) by engine rows")
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
