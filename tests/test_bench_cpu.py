"""bench.py contract on a CPU-only box: the reference arm (oracle port on the host cores) prints the agreed JSON line,
and the product arm refuses to run without a CUDA device (there is no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(*args, timeout=300):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, env=env, cwd=ROOT)


@pytest.mark.parametrize("extra,metric,unit", [(("--workload", "perft"), "perft_plies_per_sec", "plies/s"),
                                               ((), "mcts_sims_per_sec", "sims/s")])
def test_reference_arm_prints_the_contract_line(extra, metric, unit):
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", *extra)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(line)
    assert line["impl"] == "reference" and line["metric"] == metric and line["unit"] == unit
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_keeps_bitboards_exact_and_samples_within_the_cap(tmp_path, monkeypatch):
    import numpy as np
    import bench
    a = np.array([0, 1, 0x0000000810000000, 2**63 + 12345, 2**64 - 1], dtype=np.uint64)
    h = bench.bits64(a)
    assert h.dtype == np.float64 and np.array_equal((h[:, 1].astype(np.uint64) << np.uint64(32)) | h[:, 0].astype(np.uint64), a)
    arrays = {"x": np.arange(1000, dtype=np.float32).reshape(500, 2), "y": np.arange(500, dtype=np.float64)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert np.array_equal(np.load(tmp_path / "all" / "x.npy"), arrays["x"])
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4000)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    idx = np.load(tmp_path / "s1" / "row_index.npy")
    assert 0 < len(idx) < 500 and np.array_equal(idx, np.load(tmp_path / "s2" / "row_index.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "y.npy"), idx) and sum(
        np.load(tmp_path / "s1" / f"{k}.npy").nbytes for k in ("x", "y", "row_index")) <= 4000


def test_dump_arrays_of_selfplay_records_and_perft_info():
    import numpy as np
    import bench
    from othellozero_b200 import engine as E
    g = 3
    rec = {"black": np.full((g, 64), 2**64 - 2, np.uint64), "white": np.arange(g * 64, dtype=np.uint64).reshape(g, 64),
           "action": np.full((g, 64), 0xFF, np.uint8), "player": np.ones((g, 64), np.uint8),
           "n_moves": np.array([5, 60, 0], np.int32), "winner": np.array([1, -1, 0], np.int32), "visits": None}
    out = bench.selfplay_arrays(rec, 2)
    assert {k: (v.shape, v.dtype) for k, v in out.items()} == {
        "black": ((2, 64, 2), np.float64), "white": ((2, 64, 2), np.float64), "action": ((2, 64), np.float32),
        "player": ((2, 64), np.float32), "n_moves": ((2,), np.float32), "winner": ((2,), np.float32)}
    assert (out["black"][..., 0] == 2**32 - 2).all() and (out["black"][..., 1] == 2**32 - 1).all()
    assert out["n_moves"].tolist() == [5, 60] and out["winner"].tolist() == [1, -1] and (out["action"] == 255).all()
    info = np.array([0, 37 | 1 << 8, 60 | 1 << 9 | 3 << 16, 0xFF | 1 << 8 | 1 << 9 | 0xFFFF << 16], np.uint32)
    d = E.decode_perft_info(info)
    assert d["plies"].tolist() == [0, 37, 60, 255] and d["player"].tolist() == [0, 1, 0, 1]
    assert d["finished"].tolist() == [False, False, True, True] and d["passes"].tolist() == [0, 0, 3, 0xFFFF]


def test_reference_arm_refuses_dump_outputs(tmp_path):
    r = _run("--impl", "reference", "--dump-outputs", str(tmp_path / "d"), timeout=120)
    assert r.returncode != 0 and "--impl ours" in r.stderr and not (tmp_path / "d").exists()


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this check is for the CPU-only box")
    r = _run("--steps", "1")
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
