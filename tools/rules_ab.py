"""A/B of the two rule sets (the reference's flip rule vs standard Othello) on one GPU, in one process, legs alternated.

Legs (each run `--reps` times per rule set, in the order reference, standard, reference, standard, ...):
  perft      perft_playout_kernel: 2^20 uniformly random games to the end per launch, `--perft-launches` launches timed with
             CUDA events through oz_perft_playouts_dev -> plies/s
  tree       tree_step_kernel with the closed-form hash prior: 4 x 4096 self-play games, 100 simulations per move, through
             4096 slots, wall time to the end of the job -> sims/s
  selfplay   device self-play at BASELINE configs[2]'s shape: 8x8, 100 simulations per move, 4096 games in flight (plus a
             queue), C = 512 network, evaluation cache on, games starting at every phase (0..56 random plies under the
             leg's rules, as bench.py's steady-state window); `--steps` moves timed after `--warmup` -> sims/s

Game length and branching differ between the rule sets, so the per-game work differs too: a rate per simulation or per
ply is comparable between the legs, a rate per game is not.  Prints one JSON line with the GPU name and power limit read
in the same run.

usage: python tools/rules_ab.py [--reps 2] [--steps 10] [--warmup 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(device: int) -> dict:
    import torch
    out = {"gpu": torch.cuda.get_device_name(device)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, mx = [x.strip() for x in q.strip().split(",")]
        out.update(power_limit_w=float(pl), sm_max_mhz=float(mx))
    except Exception as exc:  # the figures are reported without them rather than not at all
        out.update(power_limit_w=None, note=f"nvidia-smi query failed: {exc}")
    return out


def perft_leg(E, rules: str, launches: int, device: int) -> dict:
    import torch
    from othellozero_b200 import _lib
    L = _lib.load()
    n_games = 1 << 20
    black = torch.empty(n_games, dtype=torch.int64, device=device)
    white = torch.empty_like(black)
    info = torch.empty(n_games, dtype=torch.int32, device=device)
    st = torch.cuda.current_stream(device)
    bs = E.board_arg(8, rules)

    def launch(i):
        _lib.check(L.oz_perft_playouts_dev(bs, 1234, i * n_games, n_games, -1, C.c_void_p(black.data_ptr()),
                                           C.c_void_p(white.data_ptr()), C.c_void_p(info.data_ptr()), None,
                                           C.c_void_p(st.cuda_stream)))

    launch(0)                                                     # warm-up
    torch.cuda.synchronize(device)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms, plies = 0.0, 0
    for i in range(launches):                                     # each launch timed on its own, plies counted exactly
        ev0.record(st)
        launch(1 + i)
        ev1.record(st)
        torch.cuda.synchronize(device)
        ms += ev0.elapsed_time(ev1)
        plies += int((info & 0xFF).sum().item())
    return {"ms": ms, "plies": plies, "plies_per_s": plies / (ms * 1e-3)}


def tree_leg(E, rules: str, device: int, scoring: str = "reference") -> dict:
    G, sims = 4096, 100
    e = E.Engine(8, max_games=G, nodes_per_game=sims * 61 + 64, prior_mode=E.PRIOR_HASH, seed=5, device=device,
                 rules=rules, scoring=scoring)
    try:
        e.selfplay_begin(G, sims, 1.0, 0.9, game_ids=np.arange(G, dtype=np.uint64))    # warm-up job
        e.selfplay_run(-1)
        e.sync()
        ids = np.arange(G, 5 * G, dtype=np.uint64)
        t0 = time.perf_counter()
        e.selfplay_begin(4 * G, sims, 1.0, 0.9, game_ids=ids)
        e.selfplay_run(-1)
        e.sync()
        s = time.perf_counter() - t0
        c = e.counters()
        draws = int((e.selfplay_records()["winner"] == 2).sum())
        return {"s": s, "sims": c["sims"], "moves": c["moves"], "terminal_visits": c["terminal_visits"], "draws": draws,
                "sims_per_s": c["sims"] / s}
    finally:
        e.close()


def steady_starts(E, n_games: int, rules: str, device: int, spread: int = 57):
    """Game g starts after g % spread uniformly random plies under `rules`; a playout that ended early starts over."""
    b = np.zeros(n_games, dtype=np.uint64)
    w = np.zeros(n_games, dtype=np.uint64)
    p = np.zeros(n_games, dtype=np.int32)
    init = E.perft_playouts(1, 8, max_moves=0, device=device)
    for k in range(spread):
        sel = np.arange(n_games) % spread == k
        out = E.perft_playouts(n_games, 8, seed=17, max_moves=k, device=device, rules=rules)
        ok = sel & ~out["finished"]
        b[sel], w[sel], p[sel] = init["black"][0], init["white"][0], 0
        b[ok], w[ok], p[ok] = out["black"][ok], out["white"][ok], out["player"][ok]
    return b, w, p


def selfplay_leg(E, blob, rules: str, steps: int, warmup: int, device: int, scoring: str = "reference") -> dict:
    G, sims, C_ = 4096, 100, 512
    total = 3 * G
    b, w, p = steady_starts(E, total, rules, device)
    e = E.Engine(8, max_games=G, nodes_per_game=sims * 61 + 64, prior_mode=E.PRIOR_NET, seed=7, device=device,
                 eval_cache_log2=22, rules=rules, scoring=scoring)
    try:
        e.load_weights(blob, C_)
        e.selfplay_begin(total, sims, 1.0, 0.9, -1, b, w, p, np.arange(total, dtype=np.uint64))
        for _ in range(warmup):
            e.selfplay_run(sims)
        e.sync()
        c0 = e.counters()
        t0 = time.perf_counter()
        for _ in range(steps):
            e.selfplay_run(sims)
        e.sync()
        s = time.perf_counter() - t0
        c1 = e.counters()
        d = {k: c1[k] - c0[k] for k in ("sims", "moves", "nodes", "cache_hits", "cache_aliases")}
        return {"s": s, **d, "sims_per_s": d["sims"] / s}
    finally:
        e.close()


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--steps", type=int, default=10, help="self-play leg: timed moves (100 engine steps each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--perft-launches", type=int, default=20)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rules_ab.py measures on a CUDA device; none is available")
    from othellozero_b200 import engine as E, net as oznet
    blob = oznet.init_weights(8, 512, seed=0)
    legs = {"perft": lambda r: perft_leg(E, r, args.perft_launches, args.device),
            "tree": lambda r: tree_leg(E, r, args.device),
            "selfplay": lambda r: selfplay_leg(E, blob, r, args.steps, args.warmup, args.device)}
    rate = {"perft": "plies_per_s", "tree": "sims_per_s", "selfplay": "sims_per_s"}
    samples = {leg: {"reference": [], "standard": []} for leg in legs}
    for leg, fn in legs.items():
        for _ in range(args.reps):
            for rules in ("reference", "standard"):
                samples[leg][rules].append(fn(rules))
    result = {"tool": "rules_ab", **gpu_info(args.device), "reps": args.reps, "legs": {}}
    for leg in legs:
        med = {r: statistics.median(x[rate[leg]] for x in samples[leg][r]) for r in ("reference", "standard")}
        result["legs"][leg] = {"unit": rate[leg], "reference": med["reference"], "standard": med["standard"],
                               "standard_over_reference": med["standard"] / med["reference"], "samples": samples[leg]}
    result["note"] = ("medians of alternated legs; the rule sets play different games (length, branching), so only "
                      "per-simulation / per-ply rates are compared")
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
