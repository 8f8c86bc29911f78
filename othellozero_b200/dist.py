"""Multi-GPU plumbing: one process per GPU, games sharded by global game id, no collective inside the search loop.
NCCL (torch.distributed) is used only for C1 = weight broadcast and C2 = example gather (SURVEY §8e), replacing the
reference's sftp/scp fan-out and pickled stdout (workers.py:203-296, :180-184)."""
from __future__ import annotations

import numpy as np


def shard_game_ids(n_games_total: int, rank: int, world: int) -> np.ndarray:
    """Round-robin like WorkerManager.divide_iterations (workers.py:298-303): game g -> rank g % world."""
    return np.arange(rank, n_games_total, world, dtype=np.uint64)


def broadcast_weights(blob, src: int = 0, device=None):
    """C1: float32 weight blob from rank `src` to every rank; returns a tensor on this rank's device."""
    import torch
    import torch.distributed as dist
    backend = dist.get_backend()
    dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else "cpu")
    if dist.get_rank() == src:
        t = torch.as_tensor(np.asarray(blob, dtype=np.float32)).to(dev)
        n = torch.tensor([t.numel()], dtype=torch.int64, device=dev)
    else:
        n = torch.zeros(1, dtype=torch.int64, device=dev)
        t = None
    dist.broadcast(n, src=src)
    if t is None:
        t = torch.empty(int(n.item()), dtype=torch.float32, device=dev)
    dist.broadcast(t, src=src)
    return t


def pack_records(rec: dict, winners=None) -> np.ndarray:
    """Self-play records -> compact uint64 rows [black, white, action | player<<8 | winner<<16 | game<<32] per move
    (18 B of information per position, SURVEY §8e).  winners: optional per-position winner codes [G, 64]
    (selfplay.solve_record_winners) for the winner field in place of each game's winner."""
    nm = np.asarray(rec["n_moves"]).astype(np.int64)
    g = nm.shape[0]
    valid = np.arange(64)[None, :] < nm[:, None]
    gi = np.broadcast_to(np.arange(g, dtype=np.uint64)[:, None], (g, 64))
    if winners is None:
        win = np.broadcast_to((np.asarray(rec["winner"]).astype(np.int64) & 0xFF).astype(np.uint64)[:, None], (g, 64))
    else:
        win = (np.asarray(winners).astype(np.int64) & 0xFF).astype(np.uint64).reshape(g, 64)
    meta = rec["action"].astype(np.uint64) | (rec["player"].astype(np.uint64) << np.uint64(8)) | \
        (win << np.uint64(16)) | (gi << np.uint64(32))
    return np.stack([rec["black"][valid].astype(np.uint64), rec["white"][valid].astype(np.uint64), meta[valid]], axis=1)


def gather_examples(packed: np.ndarray, device=None) -> np.ndarray:
    """C2: all-gather of variable-length packed example rows; every rank gets the concatenation in rank order."""
    import torch
    import torch.distributed as dist
    backend = dist.get_backend()
    dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else "cpu")
    world = dist.get_world_size()
    mine = torch.as_tensor(np.ascontiguousarray(packed).view(np.int64).reshape(-1, 3)).to(dev)
    cnt = torch.tensor([mine.shape[0]], dtype=torch.int64, device=dev)
    cnts = [torch.zeros_like(cnt) for _ in range(world)]
    dist.all_gather(cnts, cnt)
    mx = int(max(int(c.item()) for c in cnts))
    pad = torch.zeros((mx, 3), dtype=torch.int64, device=dev)
    pad[:mine.shape[0]] = mine
    bufs = [torch.zeros_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    out = [b[:int(c.item())].cpu().numpy() for b, c in zip(bufs, cnts)]
    return np.concatenate(out, axis=0).view(np.uint64) if out else np.zeros((0, 3), dtype=np.uint64)
