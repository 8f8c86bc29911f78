"""Multi-GPU plumbing on hardware (SURVEY 4 pyramid top, 8e): games sharded by global id over 2 ranks must reproduce
the 1-rank job bit for bit, and the package-level iteration driver (configs[4]) runs end to end.  With fewer than two
GPUs on the box both ranks share cuda:0 and the process group is gloo (the data path has no collective; only the
example gather uses it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, SIMS, TOTAL, SEED, EG = 6, 16, 40, 11, 0.8


def _play(E, device, ids):
    e = E.Engine(N, max_games=16, nodes_per_game=SIMS * 36 + 64, prior_mode=E.PRIOR_HASH, seed=SEED, device=device)
    e.selfplay_begin(len(ids), SIMS, 1.0, EG, game_ids=ids)            # 16 slots: the rest of the shard is queued
    assert e.selfplay_run(-1) == 0
    rec = e.selfplay_records()
    e.close()
    return rec


def _rank(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from othellozero_b200 import dist as ozd, engine as E
    ndev = torch.cuda.device_count()
    device = rank % ndev
    torch.cuda.set_device(device)
    backend = "nccl" if ndev >= world else "gloo"
    dist.init_process_group(backend, init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    ids = ozd.shard_game_ids(TOTAL, rank, world)
    rec = _play(E, device, ids)
    packed = ozd.pack_records(rec)
    # the packed rows carry the LOCAL game index: replace it by the global id so the union can be compared
    packed[:, 2] = (packed[:, 2] & np.uint64(0xFFFFFFFF)) | (ids[(packed[:, 2] >> np.uint64(32)).astype(np.int64)] << np.uint64(32))
    rows = ozd.gather_examples(packed)
    if rank == 0:
        q.put((backend, rows))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_shards_reproduce_the_one_rank_games():
    from othellozero_b200 import dist as ozd, engine as E
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + os.getpid() % 500
    ps = [ctx.Process(target=_rank, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    backend, rows = q.get(timeout=600)
    for p in ps:
        p.join(timeout=120)
        assert p.exitcode == 0
    ids = np.arange(TOTAL, dtype=np.uint64)
    one = ozd.pack_records(_play(E, 0, ids))
    key = lambda r: r[np.lexsort((r[:, 1], r[:, 0], r[:, 2]))]
    assert rows.shape == one.shape and np.array_equal(key(rows), key(one)), backend
    assert len(np.unique(one[:, 2] >> np.uint64(32))) == TOTAL


def test_iteration_driver_runs_end_to_end():
    """python -m othellozero_b200.iteration (configs[4]) at toy size: every phase runs and reports."""
    cmd = [sys.executable, "-m", "othellozero_b200.iteration", "--board-size", "6", "--channels", "128", "--episodes", "12",
           "--num-simulations", "10", "--epochs", "1", "--buffer-size", "4000", "--arena-games", "6", "--arena-threshold", "4",
           "--arena-simulations", "8", "--iterations", "2", "--temperature", "0"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2
    for i, d in enumerate(lines, start=1):
        assert d["iteration"] == i and set(d["phases"]) == {"selfplay_s", "gather_s", "train_s", "arena_s"}
        assert d["positions_gathered"] >= 12 * 20 and d["train_examples"] == d["buffer_examples"] <= 4000
        assert 0 <= d["arena_new_wins"] <= 6 and d["selfplay_sims"] == 10 * d["positions_gathered"]
        assert np.isfinite(np.array(d["train_history"])).all()
    assert lines[1]["buffer_examples"] >= lines[0]["buffer_examples"]


# ---- C1 / C2 through the C-ABI (oz_dist.cu, NCCL) ------------------------------------------------------------------------
def _cabi_rank(rank, world, uid_q, out_q):
    sys.path.insert(0, ROOT)
    import numpy as np
    from othellozero_b200 import engine as E, net as oznet
    n, C = 6, 128
    e = E.Engine(n, max_games=8, nodes_per_game=2, prior_mode=E.PRIOR_NET, device=rank)
    if rank == 0:
        uid = E.Engine.dist_unique_id()
        for _ in range(world - 1):
            uid_q.put(uid)
    else:
        uid = uid_q.get(timeout=120)
    e.dist_init(rank, world, uid)
    blob = oznet.init_weights(n, C, seed=13, randomize_bn=True) if rank == 0 else None
    e.dist_broadcast_weights(blob, C, root=0)                              # C1
    own, opp = np.array([0x0000000810000000], dtype=np.uint64), np.array([0x0000001008000000], dtype=np.uint64)
    pi, lg, v = e.net_forward(own, opp)
    rows = (np.arange(3 * (2 + 3 * rank), dtype=np.uint64).reshape(-1, 3) + np.uint64(1000 * rank))
    allrows = e.dist_gather_examples(rows)                                 # C2
    empty = e.dist_gather_examples(np.zeros((0, 3), dtype=np.uint64) if rank else rows[:1])
    out_q.put((rank, lg.copy(), float(v[0]), allrows, empty))
    e.close()


def test_c_abi_broadcast_and_gather_over_nccl():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs one GPU per rank: needs at least 2 GPUs")
    from othellozero_b200 import engine as E, net as oznet
    ctx = mp.get_context("spawn")
    uid_q, out_q = ctx.Queue(), ctx.Queue()
    ps = [ctx.Process(target=_cabi_rank, args=(r, 2, uid_q, out_q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted((out_q.get(timeout=600) for _ in ps), key=lambda r: r[0])
    for p in ps:
        p.join(timeout=120)
        assert p.exitcode == 0
    # C1: both ranks evaluate with rank 0's weights - bit-identical to a local load of the same blob
    e = E.Engine(6, max_games=8, nodes_per_game=2, prior_mode=E.PRIOR_NET)
    e.load_weights(oznet.init_weights(6, 128, seed=13, randomize_bn=True), 128)
    _, lg, v = e.net_forward(np.array([0x0000000810000000], dtype=np.uint64), np.array([0x0000001008000000], dtype=np.uint64))
    e.close()
    for rank, rlg, rv, allrows, empty in res:
        assert np.array_equal(rlg, lg) and rv == float(v[0])
        # C2: concatenation in rank order
        exp = np.concatenate([np.arange(6, dtype=np.uint64).reshape(-1, 3), np.arange(15, dtype=np.uint64).reshape(-1, 3) + np.uint64(1000)])
        assert np.array_equal(allrows, exp)
        assert empty.shape == (1, 3) and np.array_equal(empty[0], [0, 1, 2])       # a rank may contribute nothing
