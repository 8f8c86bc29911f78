#!/usr/bin/env python
"""bench.py — self-play hot path throughput on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload selfplay|perft|tree]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[2]: 8x8 Othello self-play, 100 sims/move, 4096 concurrent games per GPU,
random-init OthelloNNet (C=512) evaluated in bf16 on the tcgen05 tower.  One "step" = 100 engine steps (one tree
kernel + one leaf-batch network evaluation each), i.e. >= 100 simulations — about one move — for every game.
`value` = MCTS simulations / s with everything resident in HBM; `e2e` = complete self-play games through the
public API with host buffers (start positions in, example records out).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_EVAL_8 = 566_428_672       # SURVEY §8d: 2*MACs of OthelloNN(C=512) on one 8x8 position
FLOP_CONV1_PER_BOARD_8 = 2 * 589_824
FLOP_CONV2_PER_BOARD_8 = 2 * 150_994_944
FLOP_CONV3_PER_BOARD_8 = 2 * 84_934_656
# conv2 as the conv1∘conv2 table gather: 484 on-board (square, tap) rows of C bf16 read + 64 rows written per 8x8 board
GATHER_BYTES_PER_BOARD_8 = (484 + 64) * 512 * 2


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def ncu_traffic(kernel_substr, fname="r1_ncu_gemm_raw.csv", algorithmic=2 * 4096 * 64 * 512 * 2, boards=4096):
    """dram__bytes_read.sum + dram__bytes_write.sum of the first matching launch in the committed ncu --set full
    capture (profiles/<fname>; `boards` = boards per launch of that capture)."""
    import csv
    p = os.path.join(ROOT, "profiles", fname)
    try:
        rows = list(csv.reader(open(p)))
        hdr, units = rows[0], rows[1]
        ir, iw, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Kernel Name")
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        for r in rows[2:]:
            if kernel_substr in r[ik]:
                return {"bytes_per_launch": float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]],
                        "at_boards_per_launch": boards, "algorithmic_bytes": algorithmic,
                        "source": "profiles/" + fname}
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (C restatement of the reference's search + PyTorch fp32 batch-1 net), one process
# per host core, each playing the first moves of an 8x8 / 100-sim episode.
# ------------------------------------------------------------------------------------------------------------
_W = {}


def _cpu_init(n, C):
    import torch
    torch.set_num_threads(1)
    from oracle import net_torch
    from othellozero_b200 import net as oznet  # weight init only (numpy); no CUDA is touched here
    _W["net"] = net_torch.TorchNet(oznet.init_weights(n, C, seed=0), n, C)
    _W["n"] = n


def _cpu_worker(args):
    wid, sims, moves, seed = args
    import oracle
    n = _W["n"]
    start = oracle.playout(n, seed, wid, max_moves=wid % 8)
    t0 = time.perf_counter()
    out = oracle.execute_episode(n, sims, c=1.0, temperature=1.0, e_greedy=0.9, predict=_W["net"].predict, seed=seed,
                                 game_id=wid, start_board=start["board"], start_player=start["player"],
                                 max_moves=moves)
    return out["sims"], len(out["moves"]), out["net_calls"], time.perf_counter() - t0


class CpuArm:
    """The oracle port on all host cores: one process per core, each playing the first move(s) of its own 8x8 episode
    (sequential sims, one batch-1 fp32 net call per expanded node - the reference's structure, SURVEY §3.2-3.4)."""

    def __init__(self, n=8, C=512, procs=None):
        import multiprocessing as mp
        cores = os.cpu_count() or 1
        self.procs = procs or min(cores, 32)
        self.pool = mp.get_context("spawn").Pool(self.procs, initializer=_cpu_init, initargs=(n, C))
        self.calls = 0

    def sample(self, sims=100, moves=1):
        t0 = time.perf_counter()
        base = self.calls * self.procs
        res = self.pool.map(_cpu_worker, [(base + w, sims, moves, 0) for w in range(self.procs)])
        self.calls += 1
        wall = time.perf_counter() - t0
        tot_sims = sum(r[0] for r in res)
        return dict(value=tot_sims / wall, unit="sims/s", cores=self.procs, kind="port",
                    sample=f"{self.procs} processes x {moves} move(s) x {sims} sims of 8x8 episodes: C oracle search + "
                           f"PyTorch fp32 batch-1 net, 1 thread each; {tot_sims} sims, {sum(r[2] for r in res)} net calls "
                           f"in {wall:.1f}s",
                    moves_per_s=sum(r[1] for r in res) / wall)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_sample(n=8, C=512, sims=100, moves=1):
    arm = CpuArm(n, C)
    try:
        arm.sample(sims, 1)  # warm: imports, thread pools, page-in
        return arm.sample(sims, moves)
    finally:
        arm.close()


# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def synthetic_starts(engine_mod, n_games, seed, first_id, device, spread=8):
    """Start positions: the initial position + k random plies (config-2 RNG), k = game index % spread.
    spread = 8  : SURVEY 8d config 3's de-correlated OPENING starts;
    spread = 57 : games of EVERY phase (0..56 plies played) - what a long-running self-play job holds at any moment."""
    b = np.zeros(n_games, dtype=np.uint64)
    w = np.zeros(n_games, dtype=np.uint64)
    p = np.zeros(n_games, dtype=np.int32)
    init = engine_mod.perft_playouts(1, 8, seed=seed, first_game_id=first_id, max_moves=0, device=device)
    for k in range(spread):
        sel = np.arange(n_games) % spread == k
        if not sel.any():
            continue
        out = engine_mod.perft_playouts(n_games, 8, seed=seed, first_game_id=first_id, max_moves=k, device=device)
        ok = sel & ~out["finished"]                      # a playout that ended early restarts from the initial position
        b[sel], w[sel], p[sel] = init["black"][0], init["white"][0], 0
        b[ok] = out["black"][ok]; w[ok] = out["white"][ok]; p[ok] = out["player"][ok]
    return b, w, p


def l2_bandwidth(E, device, mb=32, passes=50):
    """Measured L2 read bandwidth on this GPU (oz_probe_l2_read: streaming 16-byte loads over a 32 MB L2-resident buffer,
    CUDA events) - the denominator of the table gather's roofline."""
    best = max(E.probe_l2_read(mb, passes, device) for _ in range(3))
    return {"read_gbs": best, "what": f"oz_probe_l2_read: {passes} sweeps of 16-byte .cg loads over a {mb} MB L2-resident buffer, best of 3"}


DUMP_MAX_BYTES = 60 << 20   # --dump-outputs stays under 64 MB, .npy headers included


def bits64(a):
    """uint64 bitboards -> float64 [..., 2]: the low and the high 32 bits, each exact in float64."""
    a = np.asarray(a, dtype=np.uint64)
    return np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64)


def dump_outputs(out_dir, arrays):
    """Writes each array of `arrays` (float32 / float64, one row per game) as out_dir/<name>.npy, plus row_index.npy:
    the game index of every row.  When all of it exceeds DUMP_MAX_BYTES, the same fixed, seeded sample of games is kept
    in every array."""
    rows = len(next(iter(arrays.values())))
    per_row = sum(a.nbytes for a in arrays.values()) / max(1, rows) + 8
    keep = min(rows, int(DUMP_MAX_BYTES // per_row))
    idx = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dict(arrays, row_index=np.arange(rows, dtype=np.float64)).items():
        assert a.dtype in (np.float32, np.float64) and len(a) == rows, name
        np.save(os.path.join(out_dir, name + ".npy"), a[idx])


def selfplay_arrays(rec, rows):
    """The first `rows` games' self-play records (engine.Engine.selfplay_records) as float arrays."""
    return {"black": bits64(rec["black"][:rows]), "white": bits64(rec["white"][:rows]),
            **{k: rec[k][:rows].astype(np.float32) for k in ("action", "player", "n_moves", "winner")}}


class Ctx:
    pass


def selfplay_leg(cx, *, games, sims, vl, cache_log2, window, steps, warmup, mode, dump_dir=None):
    """One timed leg of the self-play hot path: `steps` x (STEPS_PER_MOVE engine steps) with `games` slots in flight.
    window = "steady": slots start at every game phase and finished slots take queued games (steady-state mix);
             "opening": every game starts within its first 8 plies (round 1's default window).
    dump_dir: where rank 0 writes the records of the job's first generation of games, each played to its end."""
    torch, dist, E, oznet, args = cx.torch, cx.dist, cx.E, cx.oznet, cx.args
    n, C, G = 8, args.channels, games
    spm = (sims + max(1, vl) - 1) // max(1, vl)
    eng = E.Engine(n, max_games=G, nodes_per_game=sims * 61 + 64, prior_mode=mode, c_puct=1.0, seed=args.seed,
                   device=cx.local, eval_cache_log2=cache_log2 if mode == E.PRIOR_NET else 0, vl_width=vl)
    try:
        if mode == E.PRIOR_NET:
            eng.load_weights_from_tensor(cx.wt, C)
            eng.set_timing(True)
        spread = 57 if window == "steady" else 8
        # every slot always holds a game: a game lasts <= 60 moves, so 1 + (steps + warmup) // 30 queued generations
        # are more than the timed region can consume
        total = G * (2 + (steps + warmup) // 30)
        if mode == E.PRIOR_HASH:
            total = 4 * G   # one tree-only step = 4 generations through the G slots (see tree_batch)
        first_id = cx.next_id + cx.rank * total
        cx.next_id += cx.world * total
        sb, sw, sp = synthetic_starts(E, total, args.seed, first_id, cx.local, spread)
        ids = np.arange(first_id, first_id + total, dtype=np.uint64)
        tree_only = mode == E.PRIOR_HASH
        zero = {k: 0 for k in ("sims", "nodes", "moves", "cache_hits", "cache_aliases")}
        stream = torch.cuda.ExternalStream(eng.stream(), device=f"cuda:{cx.local}")

        def tree_batch():
            # hash priors: whole games run inside ONE tree kernel launch, so a step is one complete job: 4 x G games through
            # the G slots - finished slots take queued games, as in the engine's normal operation; with G games only, the
            # launch ends with a long tail of a few long games on an otherwise empty GPU (ncu: 16 of 28 warps per SM
            # resident on average) and the figure measures the tail, not the kernel
            eng.selfplay_begin(total, sims, 1.0, 0.9, -1, sb, sw, sp, ids)
            eng.selfplay_run(-1)
            return eng.counters()

        if not tree_only:
            eng.selfplay_begin(total, sims, 1.0, 0.9, -1, sb, sw, sp, ids)
        for _ in range(warmup):
            tree_batch() if tree_only else eng.selfplay_run(spm)
        eng.layer_times()  # reset the per-layer accumulators
        cx.barrier()
        c0 = dict(zero) if tree_only else eng.counters()
        l0 = eng.launches()
        sampler = ClockSampler(cx.local)
        if cx.rank == 0:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        c1 = dict(zero)
        for _ in range(steps):
            if tree_only:
                cc = tree_batch()
                for k in c1:
                    c1[k] += cc[k]
            else:
                eng.selfplay_run(spm)
        ev1.record(stream)
        cx.barrier()
        clocks = sampler.stop() if cx.rank == 0 else None
        ms = ev0.elapsed_time(ev1)
        if not tree_only:
            c1 = eng.counters()
        l1 = eng.launches()
        lt = eng.layer_times() if mode == E.PRIOR_NET else np.zeros(8, dtype=np.float32)
        if dump_dir and cx.rank == 0:
            rows = total
            if not tree_only:
                # how far a game has got when the timed steps end varies by a move from run to run, so the records are
                # not comparable then; the job's first generation (the games that started in the G slots) is played on,
                # untimed, until each of its games has ended - at most one game's length, whatever --steps is
                rows = min(G, total)
                while (eng.selfplay_records()["winner"][:rows] < 0).any() and eng.selfplay_run(spm) > 0:
                    pass
            dump_outputs(dump_dir, selfplay_arrays(eng.selfplay_records(), rows))
        d = {k: c1[k] - c0[k] for k in zero}
        d_evals = d["nodes"] - d["cache_hits"] - d["cache_aliases"]   # positions that actually went through the network
        t = torch.tensor([ms, d["sims"], d_evals, d["moves"], l1 - l0, d["cache_hits"], d["cache_aliases"]],
                         dtype=torch.float64, device=f"cuda:{cx.local}")
        if cx.world > 1:
            tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            ms = float(tmax[0]); tot = [float(x) for x in tsum[1:]]
        else:
            tot = [float(x) for x in t[1:]]
        return dict(ms=ms, sims=tot[0], evals=tot[1], moves=tot[2], launches=tot[3], hits=tot[4], aliases=tot[5],
                    evals_this_rank=float(d_evals), lt=lt, clocks=clocks, spm=spm, steps=steps, total_queued=int(total),
                    engine=None)
    finally:
        eng.close()


def tensor_roofline(cx, leg, C, conv2, conv3, peaks):
    """`roofline` object of a PRIOR_NET leg: the dominant kernel (the conv3 implicit GEMM) against the measured cuBLAS
    bf16 sustained peak, plus the whole-step tensor fraction and the per-layer times."""
    lt, world = leg["lt"], cx.world
    tree_steps = leg["steps"] * leg["spm"]
    avg_leaves = leg["evals_this_rank"] / max(1, tree_steps)  # boards per forward
    peak = peaks["bf16_sustained"]
    cs = (C / 512.0) ** 2
    table = conv2 == "table"
    names = ["conv1_gather", "conv2_table_gather" if table else "conv2", "conv3", "conv4", "fc1", "fc2", "heads"]
    layer_ms = {k: float(v) for k, v in zip(names, lt[:7])}
    if table:
        # conv1+conv2 are table reads, not tensor work: the dominant kernel is the conv3 implicit GEMM
        k_ms, k_flop, k_name = float(lt[2]), FLOP_CONV3_PER_BOARD_8, "oz_gemm2_kernel (conv3 implicit GEMM, SM pair, split M tiles)"
        # profiles/r2_ncu_step_raw.csv: one engine step of the steady-state mix, ~3 710 boards per launch
        traffic = ncu_traffic("oz_gemm2_kernel", "r2_ncu_step_raw.csv", 3710 * (64 + 36) * 512 * 2 + 9 * 512 * 512 * 2, boards=3710)
        tensor_flop_per_eval = FLOP_PER_EVAL_8 - FLOP_CONV1_PER_BOARD_8 - FLOP_CONV2_PER_BOARD_8
        if conv3 == "wino":
            # F(2,3) along y: 4 GEMMs with K = 3C instead of one with 9C -> 2/3 of the direct form's MACs are EXECUTED
            k_flop = FLOP_CONV3_PER_BOARD_8 * 2 // 3
            k_name = "oz_wino_kernel (conv3 as 1-D Winograd F(2,3), SM pair; executed FLOPs = 2/3 of the direct form)"
            traffic = ncu_traffic("oz_wino_kernel", "r1_ncu_wino_raw.csv", 4096 * (96 + 36) * 512 * 2 + 12 * 512 * 512 * 2)
            tensor_flop_per_eval -= FLOP_CONV3_PER_BOARD_8 // 3
    else:
        k_ms, k_flop, k_name = float(lt[1]), FLOP_CONV2_PER_BOARD_8, "oz_gemm2_kernel (conv2 implicit GEMM, SM pair)"
        traffic = ncu_traffic("oz_gemm2_kernel")
        tensor_flop_per_eval = FLOP_PER_EVAL_8 - FLOP_CONV1_PER_BOARD_8
    achieved = k_flop * cs * avg_leaves / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
    ms = leg["ms"]
    roof = {"bound": "tensor", "kernel": k_name,
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "peak_source": f"{peaks['source']} cuBLAS bf16 sustained", "traffic": traffic,
            "frac_of_burst_peak": achieved / peaks["bf16_burst"],
            "note": "peak = cuBLAS bf16 measured back to back for 4 s (power-limited clock); frac > 1 means this "
                    "kernel, timed inside a step that also holds lower-power kernels, runs at a higher clock "
                    "than cuBLAS sustains - both sit at the 1 kW cap",
            "avg_boards_per_launch": avg_leaves, "avg_launch_ms": k_ms,
            "layer_ms": layer_ms, "forwards_timed": int(lt[7]),
            "tensor_flop_per_eval": tensor_flop_per_eval * cs,
            "whole_step_tensor_frac": (leg["evals"] / world) * tensor_flop_per_eval * cs / (ms * 1e-3) / 1e12 / peak,
            "dense_equivalent_tflops": (leg["evals"] / world) * FLOP_PER_EVAL_8 * cs / (ms * 1e-3) / 1e12}
    gather = None
    if table and lt[1] > 0:
        gb = GATHER_BYTES_PER_BOARD_8 * (C / 512.0) * avg_leaves / (float(lt[1]) * 1e-3) / 1e9
        l2 = cx.l2
        gather = {"bound": "l2", "kernel": "conv2_table_gather_kernel (conv1+conv2 as 484 table-row reads per board)",
                  "achieved": gb, "peak": l2["read_gbs"], "unit": "GB/s", "frac": gb / l2["read_gbs"],
                  "peak_source": "measured in this run: " + l2["what"],
                  "avg_launch_ms": float(lt[1]),
                  "traffic": ncu_traffic("conv2_table_gather", "r2_ncu_step_raw.csv", 3710 * GATHER_BYTES_PER_BOARD_8, boards=3710),
                  "note": "achieved = ALGORITHMIC row bytes (548 KB per board) / launch time; the rows are served by L1 (ncu: 25 % "
                          "of the sectors in the steady-state mix) and L2 (49.5 M sectors = 1.58 GB per launch in 134 us = 11.8 TB/s "
                          "= the probe's peak; DRAM reads are 0.33 GB), so the binding unit is the L2->SM path, not HBM; a frac "
                          "above 1 means L1 hits carry part of the algorithmic traffic"}
    return roof, gather


def run_ours(args):
    import torch
    import torch.distributed as dist
    from othellozero_b200 import build as ozbuild
    ozbuild.build()
    from othellozero_b200 import engine as E, net as oznet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for --impl ours)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = load_peaks()
    n, C, sims, G = 8, args.channels, args.sims, args.games
    if args.e2e_games <= 0:
        args.e2e_games = 2 * G

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.workload == "perft":
        line = perft_leg(args, E, peaks, rank, world, local, barrier, args.steps, args.warmup, dump_dir=args.dump_outputs)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        if rank == 0:
            if not args.no_cpu:
                line["cpu_baseline"] = perft_cpu_sample()
            print(json.dumps(line))
        return

    cx = Ctx()
    cx.torch, cx.dist, cx.E, cx.oznet, cx.args = torch, dist, E, oznet, args
    cx.world, cx.rank, cx.local, cx.barrier, cx.next_id = world, rank, local, barrier, 0
    mode = E.PRIOR_NET if args.workload == "selfplay" else E.PRIOR_HASH
    cx.wt = None
    if mode == E.PRIOR_NET:
        # C1: rank 0 owns the weights, everyone else receives them over NCCL and folds them on device
        nfl = oznet.blob_size(n, C)
        if rank == 0:
            cx.wt = torch.from_numpy(oznet.init_weights(n, C, seed=0)).cuda(local)
        else:
            cx.wt = torch.empty(nfl, dtype=torch.float32, device=f"cuda:{local}")
        if world > 1:
            dist.broadcast(cx.wt, src=0)
        torch.cuda.synchronize()
        cx.l2 = l2_bandwidth(E, local)
    tree_only = mode == E.PRIOR_HASH
    leg = selfplay_leg(cx, games=G, sims=sims, vl=args.vl, cache_log2=args.eval_cache_log2, window=args.window,
                       steps=args.steps, warmup=args.warmup, mode=mode, dump_dir=args.dump_outputs)
    ms = leg["ms"]
    sims_per_s = leg["sims"] / (ms / 1e3)

    # ---- e2e: complete games through the public API with HOST buffers (copies inside) ----------------------------
    e2e, rec = None, None
    if not args.no_e2e and not tree_only:
        # a fresh engine: fresh games (other ids / start positions) and an EMPTY evaluation cache, so nothing evaluated
        # during the timed region above can be reused here
        eng = E.Engine(n, max_games=G, nodes_per_game=sims * 61 + 64, prior_mode=mode, c_puct=1.0, seed=args.seed,
                       device=local, eval_cache_log2=args.eval_cache_log2, vl_width=args.vl)
        eng.load_weights_from_tensor(cx.wt, C)
        # e2e_games may exceed the G slots: the engine queues the rest and refills slots as episodes end
        NE = args.e2e_games
        e_first = (1 << 40) + rank * NE
        sb, sw, sp = synthetic_starts(E, NE, args.seed + 1, e_first, local)
        ids = np.arange(e_first, e_first + NE, dtype=np.uint64)
        barrier()
        t0 = time.perf_counter()
        eng.selfplay_begin(NE, sims, 1.0, 0.9, args.e2e_moves, sb, sw, sp, ids)             # H2D start positions
        cb = eng.counters()
        eng.selfplay_run(-1)
        rec = eng.selfplay_records()                                                       # D2H example records
        ce = eng.counters()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        eng.close()
        e_sims = ce["sims"] - cb["sims"]
        h2d = int(sb.nbytes + sw.nbytes + sp.nbytes + ids.nbytes)
        d2h = int(sum(rec[k].nbytes for k in ("black", "white", "action", "player", "n_moves", "winner")))
        te = torch.tensor([dt, float(e_sims), float((rec["winner"] >= 0).sum()), float(rec["n_moves"].sum())],
                          dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            m = te.clone(); dist.all_reduce(m, op=dist.ReduceOp.MAX)
            s = te.clone(); dist.all_reduce(s, op=dist.ReduceOp.SUM)
            dt, e_sims, e_games, e_moves = float(m[0]), float(s[1]), float(s[2]), float(s[3])
        else:
            e_games, e_moves = float(te[2]), float(te[3])
        e2e = {"value": e_sims / dt, "unit": "sims/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "games_per_s": e_games / dt, "games": int(e_games), "mean_plies": e_moves / max(1.0, NE * world),
               "seconds": dt, "slots": int(min(G, NE)),
               "what": f"{NE} complete games/GPU through {min(G, NE)} slots (finished slots take the next queued game), "
                       "from host start positions to host example records"
                       + ("" if args.e2e_moves < 0 else f", first {args.e2e_moves} moves")}
    gathered = None
    if world > 1:
        # C2: all-gather of the packed example records over NCCL (outside the timed regions)
        from othellozero_b200 import dist as ozd
        if rec is not None:
            gathered = int(ozd.gather_examples(ozd.pack_records(rec)).shape[0])
        dist.barrier()

    # ---- extras (N = 1): the other configurations the driver should witness, each a short leg with its own roofline ----
    extras = {}
    if world == 1 and not args.no_extras and not tree_only and args.vl <= 1:
        def short(name, conv3=None, **kw):
            conv3 = conv3 or args.conv3
            try:
                os.environ["OZ_NET_CONV3"] = conv3      # read when the leg's engine is created
                lg = selfplay_leg(cx, **kw)
                r = {"value": lg["sims"] / (lg["ms"] / 1e3), "unit": "sims/s", "steps": lg["steps"], "ms_per_step": lg["ms"] / lg["steps"],
                     "evals_per_sim": lg["evals"] / max(1.0, lg["sims"]), "net_evals_per_s": lg["evals"] / (lg["ms"] / 1e3)}
                if kw["mode"] == E.PRIOR_NET:
                    roof, _ = tensor_roofline(cx, lg, C, args.conv2, conv3, peaks)
                    r["roofline"] = {k: roof[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "avg_boards_per_launch",
                                                          "avg_launch_ms", "whole_step_tensor_frac", "layer_ms")}
                else:
                    r["roofline"] = tree_roofline(r["value"], lg["clocks"], peaks)
                extras[name] = r
            except Exception as ex:  # an extra must never cost the headline line
                extras[name] = {"error": repr(ex)[:300]}
            finally:
                os.environ["OZ_NET_CONV3"] = args.conv3 if args.conv2 == "table" else "direct"
        short("opening_window", games=G, sims=sims, vl=1, cache_log2=args.eval_cache_log2, window="opening", steps=5, warmup=3, mode=E.PRIOR_NET)
        extras["opening_window"]["what"] = "round 1's default window: every game within its first ~16 plies, where the evaluation cache shares most"
        short("cache_off", games=G, sims=sims, vl=1, cache_log2=0, window="steady", steps=5, warmup=3, mode=E.PRIOR_NET)
        extras["cache_off"]["what"] = "same workload without the cross-game evaluation cache: one network evaluation per expanded node"
        if args.conv2 == "table" and args.conv3 == "direct":
            short("conv3_winograd", conv3="wino", games=G, sims=sims, vl=1, cache_log2=args.eval_cache_log2, window="steady", steps=5, warmup=3,
                  mode=E.PRIOR_NET)
            extras["conv3_winograd"]["what"] = ("the headline workload with conv3 as the opt-in 1-D Winograd F(2,3) SM-pair kernel (--conv3 wino; DESIGN 3b): "
                                               "2/3 of the direct form's tensor FLOPs are executed, so its roofline fraction counts executed FLOPs")
        short("config3_vl4", games=2048, sims=800, vl=4, cache_log2=args.eval_cache_log2, window="steady", steps=3, warmup=3, mode=E.PRIOR_NET)
        extras["config3_vl4"]["what"] = ("BASELINE.json configs[3] on ONE GPU: 800 sims/move, C=512, 2048 games x virtual-loss waves of 4 (8192 leaf "
                                        "slots per step), steady-state mix of game phases (visit counts differ from the sequential reference by "
                                        "design); 512 games x waves of 8 measure 4.4 M sims/s in the same window")
        short("tree_only", games=G, sims=sims, vl=1, cache_log2=0, window="opening", steps=2, warmup=1, mode=E.PRIOR_HASH)
        extras["tree_only"]["what"] = "rules + tree kernels alone (closed-form priors, no network): complete jobs of 4 x 4096 games through 4096 slots"
        try:
            pl = perft_leg(args, E, peaks, rank, world, local, barrier, 5, 3)
            extras["perft"] = {k: pl[k] for k in ("metric", "value", "unit", "ms_per_step", "roofline", "e2e")}
            extras["perft"]["what"] = "BASELINE.json configs[1]: 1M concurrent random playouts per launch"
        except Exception as ex:
            extras["perft"] = {"error": repr(ex)[:300]}
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return

    window_txt = ("steady-state mix: slot s starts after (s % 57) random plies, so the timed region always holds games of every "
                  "phase; finished slots take queued games" if args.window == "steady" else
                  "opening window: every game starts within its first 8 plies")
    out = {
        "metric": "mcts_sims_per_sec", "value": sims_per_s, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if mode == E.PRIOR_NET else "f64", "data": "synthetic",
        "config": {"workload": ("8x8 self-play, %d sims/move, %d concurrent games per GPU, random-init OthelloNNet "
                                "C=%d bf16 leaf eval (BASELINE.json configs[%d])" % (sims, G, C, 2 if args.vl <= 1 else 3))
                   + ("; conv1+conv2 evaluated as one partial-product table gather" if args.conv2 == "table" else "")
                   if mode == E.PRIOR_NET else
                   "8x8 self-play tree+rules only, closed-form hash priors (no network)",
                   "board": 8, "sims_per_move": sims, "games_per_gpu": G, "channels": C, "e_greedy": 0.9, "temperature": 1,
                   "eval_cache_log2": args.eval_cache_log2, "vl_width": args.vl, "window": window_txt,
                   "step": (f"{leg['spm']} engine steps (tree kernel + leaf-batch net forward) = >=1 move per game"
                            if mode == E.PRIOR_NET else f"one complete job of {4 * G} games through {G} slots (whole games run inside one launch; finished slots take queued games)"),
                   "l2": "inputs larger than L2: activations 0.8 GB/forward, node pools %.1f GB" % (G * (sims * 61 + 64) * 432 / 1e9),
                   "games_queued_per_gpu": leg["total_queued"], "parallelism": f"games sharded x{world}"},
        "moves_per_s": leg["moves"] / (ms / 1e3), "games_per_s_est": leg["moves"] / (ms / 1e3) / 60.0,
        "net_evals_per_s": leg["evals"] / (ms / 1e3), "evals_per_sim": leg["evals"] / max(1.0, leg["sims"]),
        "eval_cache": {"log2_entries": args.eval_cache_log2, "hits": int(leg["hits"]), "same_step_shares": int(leg["aliases"]),
                       "note": "identical positions are evaluated once across games; outputs are unchanged"},
        "gpu_launches": int(leg["launches"]), "clocks": leg["clocks"],
    }
    if gathered is not None:
        out["nccl"] = {"weights_broadcast_floats": int(oznet.blob_size(n, C)) if mode == E.PRIOR_NET else 0,
                       "examples_gathered": gathered}
    if mode == E.PRIOR_NET:
        out["roofline"], gather = tensor_roofline(cx, leg, C, args.conv2, args.conv3, peaks)
        if gather:
            out["roofline_conv2_table"] = gather
    else:
        out["roofline"] = tree_roofline(sims_per_s / world, leg["clocks"], peaks)
    if e2e:
        out["e2e"] = e2e
    if extras:
        out["extras"] = extras
    if not args.no_cpu and world == 1:
        out["cpu_baseline"] = cpu_sample(n, C, sims, moves=args.cpu_moves)
    print(json.dumps(out))


TREE_WARP_INSTR_PER_SIM = 2130       # counted by ncu on tree_step_kernel in the hash-prior mode (profiles/r2_ncu_treeonly_raw.csv):
                                     # 1.119e11 warp instructions / 5.25e7 simulations of one job of 4 x 4096 whole games


def tree_roofline(sims_per_s_per_gpu, clocks, peaks):
    """`roofline` of a rules+tree leg (no evaluator): the kernel is bound by instruction issue / fetch, not by HBM (its ~1 KB
    of algorithmic traffic per simulation would allow 6.5e9 sims/s), so it is stated against the warp-instruction issue peak."""
    f_sm = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 148 * 4 * f_sm * 1e6 / 1e9              # warp instructions / ns: 148 SMs x 4 schedulers x 1 per clock
    achieved = sims_per_s_per_gpu * TREE_WARP_INSTR_PER_SIM / 1e9
    return {"bound": "issue", "kernel": "tree_step_kernel", "achieved": achieved, "peak": peak, "unit": "G warp-instr/s",
            "frac": achieved / peak, "traffic": None,
            "hbm_frac": sims_per_s_per_gpu * 1000 / 1e9 / peaks["hbm_gbs"],
            "note": "achieved = sims/s x 2130 warp instructions per simulation (ncu), peak = 148 SMs x 4 schedulers x sampled SM "
                    "clock; ncu: issue-active 61 %, stalls per issue: fixed-latency 2.4, instruction fetch 2.2, long scoreboard 1.1 "
                    "(instruction-cache hit rate 88 %); hbm_frac = the same throughput against the HBM peak at ~1.0 KB algorithmic bytes per simulation "
                    "(SURVEY 8d) - bandwidth is never the limiter"}


PERFT_THREAD_INSTR_PER_PLY = 624     # counted by ncu on perft_playout_kernel (profiles/r1_ncu_perft_raw.csv): 1.51e9 warp
                                     # instructions x 32 lanes / 7.7e7 plies of one 1M-game launch


def _perft_cpu_worker(a):
    wid, games, seed = a
    import oracle
    t0 = time.perf_counter()
    plies = 0
    for g in range(games):
        plies += len(oracle.playout(8, seed, wid * games + g)["moves"])
    return plies, time.perf_counter() - t0


def perft_cpu_sample(games_per_proc=4000, procs=None):
    """CPU arm of configs[1]: the oracle's C restatement of OthelloGame.play driven by the same counter RNG
    (RandomOthelloAgent loop, agents.py:20-24,71-84), one process per host core."""
    import multiprocessing as mp
    import oracle
    oracle.build()
    procs = procs or min(os.cpu_count() or 1, 32)
    with mp.get_context("spawn").Pool(procs) as pool:
        pool.map(_perft_cpu_worker, [(w, 10, 1) for w in range(procs)])  # warm: imports
        t0 = time.perf_counter()
        res = pool.map(_perft_cpu_worker, [(w, games_per_proc, 0) for w in range(procs)])
        wall = time.perf_counter() - t0
    plies = sum(r[0] for r in res)
    return dict(value=plies / wall, unit="plies/s", cores=procs, kind="port",
                sample=f"{procs} processes x {games_per_proc} random 8x8 playouts through the oracle's OthelloGame.play "
                       f"restatement: {plies} plies in {wall:.1f}s")


def perft_leg(args, E, peaks, rank, world, local, barrier, steps, warmup, dump_dir=None):
    """configs[1]: random-playout perft, 1M concurrent games per launch.  Returns the JSON line as a dict (rank 0) after the
    max/sum over ranks; the caller owns the process group.  dump_dir: where rank 0 writes the final positions of the last
    timed launch's games."""
    import ctypes as C
    import torch
    n_games = args.games if args.games > 4096 else (1 << 20)
    b = torch.empty(n_games, dtype=torch.int64, device=f"cuda:{local}")
    w = torch.empty_like(b)
    info = torch.empty(n_games, dtype=torch.int32, device=f"cuda:{local}")
    L = E._lib.load()

    def launch(seed):
        E.check(L.oz_perft_playouts_dev(8, seed, rank * n_games, n_games, -1, C.c_void_p(b.data_ptr()),
                                        C.c_void_p(w.data_ptr()), C.c_void_p(info.data_ptr()), None, None))
    for i in range(warmup):
        launch(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        launch(100 + i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = None
    if rank == 0:
        # the timed region lasts ~20 ms, shorter than one nvidia-smi period: keep the same launches running (untimed)
        # until the sampler has seen the GPU under this load
        t_end, extended = time.time() + 3.0, False
        while len(sampler.lines) < 2 and time.time() < t_end:
            extended = True
            for i in range(steps):
                launch(100 + i)
            torch.cuda.synchronize()
        clocks = sampler.stop()
        if extended:
            clocks["note"] = "timed region shorter than the sampling period: sampled while the same launches were repeated untimed"
    # every launch plays different games (seed): replay the same seeds outside the timed region to count their plies
    plies = 0
    for i in range(steps):
        launch(100 + i)
        plies += int((info & 0xFF).sum().item())
    if dump_dir and rank == 0:
        # the loop above ended with the last timed launch's seed
        fields = E.decode_perft_info(info.cpu().numpy().view(np.uint32))
        dump_outputs(dump_dir, dict({"black": bits64(b.cpu().numpy().view(np.uint64)),
                                     "white": bits64(w.cpu().numpy().view(np.uint64))},
                                    **{k: v.astype(np.float32) for k, v in fields.items()}))
    # e2e: the host-buffer entry point (results D2H inside the timed region), one launch
    E.perft_playouts(n_games, 8, seed=6, first_game_id=rank * n_games, device=local)  # warm: sizes the staging buffers
    e_calls, e_plies = 3, 0
    t0 = time.perf_counter()
    for i in range(e_calls):
        out = E.perft_playouts(n_games, 8, seed=7 + i, first_game_id=rank * n_games, device=local)
        e_plies += int(out["plies"].sum())
    dt = time.perf_counter() - t0
    t = torch.tensor([ms, float(plies), dt, float(e_plies)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        import torch.distributed as dist
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        ms, dt, plies, e_plies = float(tm[0]), float(tm[2]), int(ts[1]), int(ts[3])
    value = plies / (ms / 1e3)
    f_sm = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 148 * 4 * 32 * f_sm * 1e6 / 1e9          # thread-instructions / ns the SMs can issue at the sampled clock
    achieved = value / world * PERFT_THREAD_INSTR_PER_PLY / 1e9
    line = {"metric": "perft_plies_per_sec", "value": value, "unit": "plies/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "8x8 random-playout perft, %d concurrent games per GPU (BASELINE.json configs[1])" % n_games,
                       "l2": "state lives in registers for the whole game; 24 B written per game"},
            "gpu_launches": steps, "clocks": clocks,
            "roofline": {"bound": "int-issue", "kernel": "perft_playout_kernel", "achieved": achieved, "peak": peak,
                         "unit": "G thread-instr/s", "frac": achieved / peak, "traffic": None,
                         "note": "SURVEY 8d: the path is integer-issue bound, not HBM bound; achieved = plies/s x 624 counted "
                                 "thread-instructions per ply, peak = 148 SMs x 4 schedulers x 32 lanes x sampled SM clock; "
                                 "ncu: ALU pipe 95.6 % active (profiles/r1_ncu_perft_raw.csv)"},
            "e2e": {"value": e_plies / dt, "unit": "plies/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": int(n_games * 20), "calls": e_calls,
                    "what": "oz_perft_playouts_host with host buffers: one launch + final boards/info D2H per call (+ numpy unpacking)"}}
    return line


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "perft":
        vals, last = [], None
        t0 = time.perf_counter()
        for _ in range(args.steps):
            last = perft_cpu_sample(games_per_proc=2000)
            vals.append(last["value"])
        dt = time.perf_counter() - t0
        v = float(np.mean(vals)); last["value"] = v
        print(json.dumps({"impl": "reference", "metric": "perft_plies_per_sec", "value": v, "unit": "plies/s",
                          "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": "8x8 random-playout perft (BASELINE.json configs[1]); CPU arm = oracle port of "
                                                 "OthelloGame.play on all host cores"},
                          "cpu_baseline": last,
                          "e2e": {"value": v, "unit": "plies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    arm = CpuArm(8, args.channels)
    try:
        for _ in range(max(1, args.warmup)):
            arm.sample(args.sims, 1)
        t0 = time.perf_counter()
        tot = 0.0
        last = None
        for _ in range(args.steps):
            last = arm.sample(args.sims, args.cpu_moves)
            tot += last["value"]
        dt = time.perf_counter() - t0
    finally:
        arm.close()
    v = tot / max(1, args.steps)
    cb = dict(last); cb["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": "mcts_sims_per_sec", "value": v, "unit": "sims/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "8x8 self-play, 100 sims/move, random-init OthelloNNet C=%d (BASELINE.json configs[2]); CPU "
                               "arm = oracle port of the reference's sequential search + batch-1 fp32 net on all host "
                               "cores; step = one move (100 sims) per process" % args.channels},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="selfplay", choices=["selfplay", "tree", "perft"])
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--channels", type=int, default=512)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-games", type=int, default=0,
                    help="complete games per GPU for the e2e figure (default 2 x --games: every slot plays two episodes)")
    ap.add_argument("--e2e-moves", type=int, default=-1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-moves", type=int, default=1)
    ap.add_argument("--eval-cache-log2", type=int, default=24)
    ap.add_argument("--conv2", default="table", choices=["table", "gemm"],
                    help="conv2 as the conv1∘conv2 partial-product table gather (default) or as the tcgen05 implicit GEMM")
    ap.add_argument("--conv3", default="direct", choices=["direct", "wino"],
                    help="conv3 as the direct implicit GEMM (default) or as the opt-in Winograd F(2,3) kernel (DESIGN 3b)")
    ap.add_argument("--vl", type=int, default=1, help="virtual-loss wave width (configs[3]); 1 = sequential, bit-exact")
    ap.add_argument("--window", default="steady", choices=["steady", "opening"],
                    help="steady: slots start at every game phase (the steady-state mix of a long self-play job, independent of "
                         "--steps/--warmup); opening: every game within its first plies (round 1's window)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the short extra legs (opening window, cache off, configs[3] waves, tree only, perft) of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path computed as DIR/<name>.npy in float32/float64, "
                         "at most 64 MB (a fixed, seeded sample of games beyond that): self-play, the records of the "
                         "games that started in the slots, each played to its end untimed; tree, the last job's records; "
                         "perft, the last launch's final positions.  With several GPUs, rank 0's games")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
        return run_reference(args)
    os.environ["OZ_NET_CONV2"] = args.conv2  # read by the engine when it is created
    os.environ["OZ_NET_CONV3"] = args.conv3 if args.conv2 == "table" else "direct"
    return run_ours(args)


if __name__ == "__main__":
    main()
