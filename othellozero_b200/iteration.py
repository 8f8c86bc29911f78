"""One full training iteration on the whole node (BASELINE.json configs[4]; reference: main.py:71-148):

    self-play sharded by game  ->  C2 gather of packed example records  ->  replay buffer (main.py:21-53,87-99)
    ->  training step (Net/NNet.py:53-68: `epochs` x batch 32; train.train_blob(ddp="auto"): sharded over the GPUs when the
        batch is large enough to be worth it, otherwise one GPU replays a CUDA graph of the step and broadcasts the result)
    ->  every rank folds the new weights onto its device tower  ->  arena new vs old, games sharded (main.py:103-148)

One process per GPU (torch.distributed over NCCL); the only collectives are C2 (example gather, once), the training step's
(gradient / BatchNormalization-statistics all-reduces when it is sharded, else one broadcast of the new weights = C1), and
one all-reduce of the arena's win count.  train_blob returns the same weights on every rank either way.

    python -m othellozero_b200.iteration                       # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 -m othellozero_b200.iteration

prints one JSON line with the wall time of every phase (max over ranks)."""
from __future__ import annotations

import argparse
import json
import os
import time
from dataclasses import asdict, dataclass

import numpy as np


@dataclass
class IterationConfig:
    """Defaults = the reference's (main.py:264-309) where it has one."""
    board_size: int = 8
    channels: int = 512
    episodes: int = 100              # num_episodes, per ITERATION over all ranks (main.py default 100)
    num_simulations: int = 100
    degree_exploration: float = 1.0
    e_greedy: float = 0.9
    temperature: float = 1.0         # main.py:73-76 switches to 0 from `temperature_threshold` on
    buffer_size: int = 76_800        # training_buffer_size, in examples
    epochs: int = 10
    batch_size: int = 32
    lr: float = 1e-3
    dropout: float = 0.3
    arena_games: int = 20            # self_play_total_games
    arena_threshold: int = 11        # self_play_threshold
    arena_simulations: int = 25
    max_concurrent: int = 4096
    seed: int = 0
    rules: str = "reference"         # "standard": self-play and arena under standard Othello flipping
    scoring: str = "reference"       # "standard": a drawn game is a draw (z = 0; no arena win for either network)
    solve_empties: int = 0           # > 0: positions with <= this many empties get perfect-play targets (exact solver)
    precision: str = "bf16"          # "fp8": self-play and arena nets evaluate conv3/conv4/fc1 in FP8 (training stays fp32)
    values: str = "reference"        # "standard": self-play and arena searches negate a value only when the side swapped
    solve_leaves: int = 0            # > 0: self-play and arena searches solve new leaves with <= this many empties exactly
    dirichlet_alpha: float = 0.0     # > 0: self-play roots get Dirichlet(alpha) noise once (the arena never explores)
    dirichlet_fraction: float = 0.25  # ... mixed in with this weight
    sample_moves: int = 0            # > 0: self-play plays its first this many plies in proportion to the visit counts


def unpack_rows(rows: np.ndarray):
    """dist.pack_records rows -> (black, white, action square bit, z); z = 0 for a drawn game (winner code 2)."""
    from ._lib import WINNER_DRAW
    rows = np.asarray(rows, dtype=np.uint64).reshape(-1, 3)
    meta = rows[:, 2].astype(np.int64)
    action, player, winner = meta & 0xFF, (meta >> 8) & 0xFF, (meta >> 16) & 0xFF
    return rows[:, 0], rows[:, 1], action, np.where(winner == WINNER_DRAW, 0, np.where(winner == player, 1, -1))


def training_arrays(rows: np.ndarray, board_size: int):
    """Replay-buffer positions -> (boards (E,N,N,2) f32, one-hot policies (E,N*N) f32, z (E,) f32) with the 8
    symmetries of training.py:13-23 (E = 8 x positions)."""
    from .selfplay import expand_symmetries
    black, white, action, z = unpack_rows(rows)
    b8, p8 = expand_symmetries(black, white, action, board_size)
    n = board_size
    return (b8.reshape(-1, n, n, 2).astype(np.float32), p8.reshape(-1, n * n).astype(np.float32),
            np.repeat(z, 8).astype(np.float32))


class Trainer:
    """The state main.training keeps across iterations (main.py:66-70): current / previous network, replay buffer."""

    def __init__(self, cfg: IterationConfig, blob: np.ndarray | None = None):
        import torch
        import torch.distributed as dist
        from . import buffer, net as oznet
        from ._lib import channels_arg
        channels_arg(cfg.channels, cfg.precision)  # ValueError for an unknown precision, before any GPU work
        if cfg.precision == "fp8" and cfg.channels % 256:
            raise ValueError(f"FP8 evaluation needs channels to be a multiple of 256 (got {cfg.channels})")
        self.cfg = cfg
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.local = int(os.environ.get("LOCAL_RANK", "0")) if torch.cuda.is_available() else 0
        if blob is None:
            blob = oznet.init_weights(cfg.board_size, cfg.channels, seed=cfg.seed)
        if self.world > 1:   # C1: everyone starts from rank 0's weights
            from . import dist as ozd
            blob = ozd.broadcast_weights(blob if self.rank == 0 else None, src=0).cpu().numpy()
        self.blob = np.ascontiguousarray(blob, dtype=np.float32)
        self.old_blob = self.blob.copy()
        self.buffer = buffer.RecordBuffer(cfg.buffer_size)
        self.iteration = 0
        self.next_game_id = 0

    def _sync(self):
        import torch
        import torch.distributed as dist
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()

    def run_iteration(self) -> dict:
        import torch
        import torch.distributed as dist
        from . import arena, dist as ozd, net as oznet, selfplay, train
        cfg, n, C = self.cfg, self.cfg.board_size, self.cfg.channels
        self.iteration += 1
        phases, info = {}, {}
        dev = f"cuda:{self.local}"

        def timed(name, t0):
            self._sync()
            phases[name] = time.perf_counter() - t0

        # ---- self-play: episodes sharded round-robin by global game id (workers.py:298-303) ---------------------------
        self._sync(); t0 = time.perf_counter()
        ids = np.arange(self.next_game_id + self.rank, self.next_game_id + cfg.episodes, self.world, dtype=np.uint64)
        self.next_game_id += cfg.episodes
        net_now = oznet.B200NNet((n, n), C, device=self.local, max_batch=8, blob=self.blob, precision=cfg.precision)
        rec = None
        if ids.size:
            sp = selfplay.SelfPlay(n, net_now, cfg.degree_exploration, max_games=min(int(ids.size), cfg.max_concurrent),
                                   num_simulations=cfg.num_simulations, device=self.local, seed=cfg.seed,
                                   rules=cfg.rules, scoring=cfg.scoring, values=cfg.values,
                                   solve_leaves=cfg.solve_leaves, dirichlet_alpha=cfg.dirichlet_alpha,
                                   dirichlet_fraction=cfg.dirichlet_fraction, sample_moves=cfg.sample_moves)
            rec = sp.play(int(ids.size), cfg.temperature, cfg.e_greedy, game_ids=ids)
            info["selfplay_sims_this_rank"] = sp.engine.counters()["sims"]
            # how many of this rank's games differ from every other (move sequences): 1 when every game is the same
            # game (e_greedy = 1 without root exploration), up to the rank's game count
            nm = np.asarray(rec["n_moves"]).astype(np.int64)
            info["distinct_this_rank"] = len({rec["action"][g][:nm[g]].tobytes() for g in range(nm.size)})
            sp.close()
        timed("selfplay_s", t0)
        # ---- exact endgame targets: every rank relabels the positions of its own games ---------------------------------
        winners = None
        if cfg.solve_empties > 0:
            t0 = time.perf_counter()
            solved = relabelled = 0
            if rec is not None:
                winners = selfplay.solve_record_winners(rec, n, cfg.solve_empties, cfg.rules, cfg.scoring,
                                                        device=self.local)
                mask = selfplay.solvable_positions(rec, n, cfg.solve_empties)
                solved = int(mask.sum())
                relabelled = int((mask & (winners != np.asarray(rec["winner"])[:, None])).sum())
            info["solve_this_rank"] = (solved, relabelled)
            timed("solve_s", t0)
        # ---- C2: gather the packed example records; every rank keeps the same replay buffer ----------------------------
        t0 = time.perf_counter()
        packed = ozd.pack_records(rec, winners) if rec is not None else np.zeros((0, 3), dtype=np.uint64)
        rows = ozd.gather_examples(packed) if self.world > 1 else packed
        self.buffer.extend(rows)
        timed("gather_s", t0)
        # ---- training step, sharded over the ranks (main.py:99-101) ----------------------------------------------------
        t0 = time.perf_counter()
        arrays = training_arrays(self.buffer.positions(), n)
        new_blob, hist = train.train_blob(self.blob, arrays, n, C, epochs=cfg.epochs, batch_size=cfg.batch_size, lr=cfg.lr,
                                          dropout=cfg.dropout, device=dev if torch.cuda.is_available() else "cpu",
                                          seed=cfg.seed + self.iteration, ddp="auto" if self.world > 1 else False)
        timed("train_s", t0)
        # ---- arena: new vs old, half the games with each colour (main.py:103-131), games sharded over the ranks -------
        t0 = time.perf_counter()
        half = cfg.arena_games // 2
        mine_a = len(range(self.rank, half, self.world))
        mine_b = len(range(self.rank, cfg.arena_games - half, self.world))
        new_net = oznet.B200NNet((n, n), C, device=self.local, max_batch=8, blob=new_blob, precision=cfg.precision)
        old_net = oznet.B200NNet((n, n), C, device=self.local, max_batch=8, blob=self.old_blob, precision=cfg.precision)
        wins = draws = 0
        rng = np.random.default_rng(cfg.seed * 1000 + self.iteration * 64 + self.rank)
        for games, black_net, white_net, new_side in ((mine_a, new_net, old_net, 0), (mine_b, old_net, new_net, 1)):
            if games:
                out = arena.pit(n, black_net, white_net, cfg.arena_simulations, cfg.degree_exploration, n_games=games,
                                device=self.local, rng=rng, rules=cfg.rules, scoring=cfg.scoring, values=cfg.values,
                                solve_leaves=cfg.solve_leaves)
                wins += int((out["winner"] == new_side).sum())
                draws += int(out["draws"].sum()) if cfg.scoring == "standard" else 0
        if self.world > 1:
            t = torch.tensor([wins, draws], dtype=torch.int64, device=dev)
            dist.all_reduce(t)
            wins, draws = int(t[0].item()), int(t[1].item())
        timed("arena_s", t0)
        promoted = wins >= cfg.arena_threshold                       # main.py:135-146 (wins only: a draw is not a win)
        if promoted:
            self.old_blob = new_blob.copy()
            self.blob = new_blob
        else:
            self.blob = self.old_blob.copy()
        if self.world > 1:   # report the slowest rank per phase
            t = torch.tensor([phases[k] for k in sorted(phases)], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            phases = {k: float(v) for k, v in zip(sorted(phases), t)}
            s = torch.tensor([info.get("selfplay_sims_this_rank", 0)], dtype=torch.int64, device=dev)
            dist.all_reduce(s)
            info["selfplay_sims"] = int(s.item())
            d = torch.tensor([info.get("distinct_this_rank", 0)], dtype=torch.int64, device=dev)
            dist.all_reduce(d)
            info["selfplay_distinct_games"] = int(d.item())
        else:
            info["selfplay_sims"] = info.get("selfplay_sims_this_rank", 0)
            info["selfplay_distinct_games"] = info.get("distinct_this_rank", 0)
        solve = {}
        if cfg.solve_empties > 0:
            counts = info["solve_this_rank"]
            if self.world > 1:
                t = torch.tensor(list(counts), dtype=torch.int64, device=dev)
                dist.all_reduce(t)
                counts = (int(t[0].item()), int(t[1].item()))
            solve = dict(solved_positions=counts[0], solve_relabelled=counts[1])
        return dict(iteration=self.iteration, phases=phases, episodes=cfg.episodes, positions_gathered=int(rows.shape[0]),
                    buffer_examples=len(self.buffer), train_examples=int(arrays[0].shape[0]),
                    train_steps=cfg.epochs * ((arrays[0].shape[0] + cfg.batch_size - 1) // cfg.batch_size),
                    train_history=hist, arena_new_wins=wins, arena_draws=draws, arena_games=cfg.arena_games,
                    promoted=bool(promoted),
                    selfplay_sims=info["selfplay_sims"], selfplay_distinct_games=info["selfplay_distinct_games"],
                    selfplay_sims_per_s=info["selfplay_sims"] / max(phases["selfplay_s"], 1e-9), **solve)


def main(argv=None):
    from ._lib import PRECISIONS, RULES, SCORINGS, VALUES
    choices = {"rules": RULES, "scoring": SCORINGS, "precision": PRECISIONS, "values": VALUES}
    # the two solver flags do different things and compose: one relabels training targets, the other changes the search
    helps = {"solve_empties": "training targets: positions with <= K empties get the perfect-play winner as z "
                              "(self-play and its search unchanged)",
             "solve_leaves": "search: new leaves with <= K empties are solved exactly instead of evaluated by the "
                             "network (needs --values standard --scoring standard; targets unchanged)",
             "values": "search value backup: 'standard' negates a child's value only when the move swapped the side "
                       "to move",
             "dirichlet_alpha": "self-play only: Dirichlet(alpha) noise mixed into each root's priors once (0: none)",
             "dirichlet_fraction": "self-play only: the weight of the root noise, in [0, 1]",
             "sample_moves": "self-play only: the first M plies are drawn in proportion to the root visit counts "
                             "(the e_greedy coin still applies)"}
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    for f, v in asdict(IterationConfig()).items():
        ap.add_argument("--" + f.replace("_", "-"), type=type(v), default=v, help=helps.get(f),
                        **({"choices": choices[f]} if f in choices else {}))
    ap.add_argument("--iterations", type=int, default=1)
    args = ap.parse_args(argv)
    from ._lib import SOLVE_MAX_EMPTIES
    if not 0 <= args.solve_empties <= SOLVE_MAX_EMPTIES:
        ap.error(f"--solve-empties must be in [0, {SOLVE_MAX_EMPTIES}] (got {args.solve_empties})")
    from ._lib import exploration_arg, values_arg
    try:
        values_arg(args.values, args.solve_leaves, args.scoring)
        exploration_arg(args.dirichlet_alpha, args.dirichlet_fraction, args.sample_moves)
    except ValueError as err:
        ap.error(str(err))
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo",
                                **({"device_id": torch.device("cuda", local)} if torch.cuda.is_available() else {}))
    cfg = IterationConfig(**{f: getattr(args, f) for f in asdict(IterationConfig())})
    tr = Trainer(cfg)
    for _ in range(args.iterations):
        out = tr.run_iteration()
        if tr.rank == 0:
            print(json.dumps(dict(config=asdict(cfg), n_gpus=world, **out)), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
