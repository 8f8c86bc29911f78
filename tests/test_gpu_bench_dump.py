"""bench.py --dump-outputs on the GPU: the same arguments give the same files, and the cross-game evaluation cache does
not change them (it only saves evaluations), so two builds can be compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--games", "256", "--steps", "2", "--warmup", "3", "--no-extras", "--no-cpu", "--no-e2e"]


def _dump(out, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *SMALL, *extra, "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}


def test_selfplay_dump_is_reproducible_and_cache_independent(tmp_path):
    a = _dump(tmp_path / "a")
    assert set(a) == {"black", "white", "action", "player", "n_moves", "winner", "row_index"}
    assert a["row_index"].tolist() == list(range(256)) and (a["winner"] >= 0).all() and (a["n_moves"] > 0).all()
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    for other in (_dump(tmp_path / "b"), _dump(tmp_path / "c", "--eval-cache-log2", "0")):
        assert set(other) == set(a) and all(np.array_equal(a[k], other[k]) for k in a)
