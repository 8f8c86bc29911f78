"""FP8 network evaluation (DESIGN.md 13): argument handling and the host emulation, without a GPU."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fp8_emul  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_precisions_and_channels_arg():
    from othellozero_b200 import _lib
    assert _lib.PRECISIONS == ("bf16", "fp8")
    assert _lib.channels_arg(512) == 512
    assert _lib.channels_arg(256, "fp8") == 256 | 0x10000
    for bad in ("fp16", "FP8", "", None):
        with pytest.raises(ValueError):
            _lib.channels_arg(512, bad)


def test_header_and_binding_agree():
    from othellozero_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "oz_b200.h")).read()
    m = re.search(r"#define OZ_NET_FP8 (0x[0-9a-fA-F]+)", hdr)
    assert m and int(m.group(1), 16) == _lib.NET_FP8
    assert "int oz_net_fp8_scales(oz_engine* e, float* out);" in hdr
    assert "oz_net_fp8_scales" in _lib.SIGNATURES


def test_precision_validated_before_device_work():
    from othellozero_b200 import net
    with pytest.raises(ValueError):
        net.B200NNet((6, 6), 256, precision="int8", blob=np.zeros(1, dtype=np.float32))


def test_iteration_precision_flag(monkeypatch):
    from othellozero_b200 import iteration
    assert iteration.IterationConfig().precision == "bf16"
    with pytest.raises(SystemExit):
        iteration.main(["--precision", "fp4"])
    with pytest.raises(ValueError):  # an unknown precision fails before any GPU work
        iteration.Trainer(iteration.IterationConfig(precision="int4"))
    with pytest.raises(ValueError, match="multiple of 256"):  # so does a channel count FP8 cannot run
        iteration.Trainer(iteration.IterationConfig(precision="fp8", board_size=6, channels=128))
    seen = {}

    class Stop(Exception):
        pass

    def fake_trainer(cfg):
        seen["cfg"] = cfg
        raise Stop

    monkeypatch.setattr(iteration, "Trainer", fake_trainer)
    with pytest.raises(Stop):
        iteration.main(["--precision", "fp8", "--board-size", "6", "--channels", "256"])
    assert seen["cfg"].precision == "fp8"


def test_e4m3_decode_table():
    import torch
    from othellozero_b200.engine import E4M3_VALUES
    ref = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(torch.float8_e4m3fn).to(torch.float32).numpy()
    same = (ref == E4M3_VALUES) | (np.isnan(ref) & np.isnan(E4M3_VALUES))
    assert same.all()


def test_emulation_without_quantisation_is_the_oracle():
    from oracle import net_torch
    from othellozero_b200 import net
    n, C = 6, 256
    blob = net.init_weights(n, C, seed=4, randomize_bn=True)
    rng = np.random.default_rng(1)
    occ, col = rng.random((12, n, n)) < 0.6, rng.random((12, n, n)) < 0.5
    x = np.stack([occ & col, occ & ~col], axis=-1).astype(np.float32)
    own, opp = net.boards_to_bits(x)
    _, elg, ev, _ = fp8_emul.forward(blob, own, opp, n, C, quantize=False)
    _, olg, ov = net_torch.forward(blob, x, n, C)
    assert np.abs(elg - olg).max() < 1e-4 and np.abs(ev - ov).max() < 1e-4


def test_emulation_quantisation_points():
    import torch
    # satfinite e4m3: 448 is the largest finite value, larger inputs saturate, rounding is to nearest even
    v = fp8_emul._e4m3(torch.tensor([500.0, -1e6, 17.0, 0.0]))
    assert v.tolist() == [448.0, -448.0, 16.0, 0.0]
    # the fused pair encoding stays within half a bf16 ulp of the odd value
    odd = torch.tensor([1.2345678, -3.3e-3, 7.0e3])
    even = torch.tensor([0.5, 2.0, -1.0])
    w = fp8_emul._pair_fused(even, odd)
    ulp = torch.tensor([2.0 ** -7, 2.0 ** -16, 2.0 ** 5])
    assert (torch.abs(w - odd) <= ulp / 2).all()


def test_fp8_calls_fail_without_a_device():
    from othellozero_b200 import _lib, engine
    try:
        _lib.load()
    except _lib.OzError:
        pytest.skip("liboz_b200.so is not built")
    cnt = np.zeros(1, dtype=np.int32)
    rc = _lib.load().oz_device_count(cnt.ctypes.data_as(_lib.i32p))
    if rc == 0 and cnt[0] > 0:
        pytest.skip("a device is present")
    with pytest.raises((_lib.OzError, AssertionError)):
        engine.Engine(6, max_games=4, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    with pytest.raises(AssertionError):  # null engine: rejected before any CUDA call
        _lib.check(_lib.load().oz_net_fp8_scales(None, None))
