"""The bf16 tower (the default evaluator) layer by layer against the rounding-faithful host emulation
(tests/fp8_emul.py, precision="bf16"), at every channel count the loader accepts.

Each layer is fed the device's own input through `inject`, so a layer can differ from the emulation only through the
order of its fp32 sums.  For an output with |bias| + sum |terms| = M, a K-term fp32 sum in any order is within
(K - 1) * u * M of the exact sum (u = 2^-24); the emulation's rounding of the exact sum, the bias add on both sides and
the emulation's own rounding add at most 4 * u * M more.  So the pre-activations differ by at most
delta = (K + 3) * u * M.  Two values x, y that round to bf16 codes with another code between them lie at least half
their codes' distance apart, so every element must either be the adjacent bf16 code of the emulation's value or lie
within 2 * delta of it.  Near zero, where the bf16 grid is finer than delta, that second clause is the ReLU edge.  Per
layer:

- act2, table gather: the nine table entries are device GEMM results rounded to bf16 (or the fused pair encoding), so
  each may be one bf16 step, at most 2^-7 of its size, from the emulation's.  The gather itself adds in the same order
  as the emulation.  delta = 2^-6 * M, with M = |bias| + sum of the nine |entries|.
- act2, OZ_NET_CONV2=gemm: K = 9C over act1.  act1 itself is the conv1 table row, computed in the same order on both
  sides, and must be equal bit for bit.
- act3: K = 9C; with OZ_NET_CONV3=wino each of the three products summed into an output row has K = 3C, and the
  epilogue's three fp32 adds are included: delta = (3C + 4) * u * M, M = the three products' sum |terms| + |bias|.
- act4: K = 9C.  f1: K = (n-4)^2 C.  f2: K = 1024.  Logits and value: K = 512 (the value also through tanhf).

Outside those bounds a difference means a wrong kernel.  Inside them a difference is a rounding flip, which needs a
value within fp32 noise of a bf16 rounding boundary, so flips must also be rare: FRAC_MAX bounds the fraction of
differing elements in each layer.

Batches: B = 1 first on a fresh engine, then B = B_RAGGED = max_games.  299 boards leave the last tile of every layer
partial: 8x8 conv3 tiles hold 7 half-boards (598 = 7 * 85 + 3), 8x8 conv4 8 boards, 6x6 conv3 8, 6x6 conv4 32, fc1, fc2
and the heads 128, the 8x8 conv2 GEMM 2, the 6x6 split conv2 GEMM 7 half-boards, the Winograd kernel 7 (8x8) or 16
(6x6) boards.  At 8x8 and C >= 384, conv3 then has more tiles than the GPU has SMs (86 m-tiles times C/128 or C/256 n
tiles), and the gather's 2-CTAs-per-SM grid walks more than one board per CTA.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import fp8_emul  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(HERE)
U32 = 2.0 ** -24
B_RAGGED = 299
# Measured on an NVIDIA B200 (1000 W power limit), 299 boards: at most 3.7e-3 of a layer's elements differ (f1 at 8x8,
# C = 1024, K = 16384 terms).  The flip rate grows with K: act3 and act4 up to 2.0e-3, the gather's act2 up to 1.7e-4,
# the conv2 GEMM's act2 up to 1.1e-3, f2 up to 2.7e-4.
FRAC_MAX = 1e-2
CHANNELS = [128, 256, 384, 512, 640, 768, 896, 1024]
LAYERS = ["act1", "act2", "act3", "act4", "f1", "f2"]  # Engine.activation layers 0..5


def _positions(n, count, seed):
    own, opp = [], []
    for g in range(count):
        po = oracle.playout(n, seed, g, max_moves=g % (n * n - 6))
        b, w, p = po["black"], po["white"], po["player"]
        own.append(w if p else b)
        opp.append(b if p else w)
    return np.array(own, dtype=np.uint64), np.array(opp, dtype=np.uint64)


def _engine(n, C, blob, conv2="table", conv3="direct", max_games=B_RAGGED):
    """An engine in the given conv2 / conv3 mode (read from the environment when an engine is created)."""
    from othellozero_b200 import engine
    saved = {k: os.environ.get(k) for k in ("OZ_NET_CONV2", "OZ_NET_CONV3")}
    os.environ["OZ_NET_CONV2"], os.environ["OZ_NET_CONV3"] = conv2, conv3
    try:
        e = engine.Engine(n, max_games=max_games, nodes_per_game=2, prior_mode=engine.PRIOR_NET)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    e.load_weights(blob, C)
    return e


def _shape(name, n, C):
    return {"act1": (n * n, C), "act2": (n * n, C), "act3": ((n - 2) ** 2, C), "act4": ((n - 4) ** 2, C),
            "f1": (1, 1024), "f2": (1, 512)}[name]


def _delta(name, n, C, conv2, conv3, M):
    if name == "act2" and conv2 == "table":
        return 2.0 ** -6 * M
    if name == "act3" and conv3 == "wino":
        return (3 * C + 4) * U32 * M
    K = {"act2": 9 * C, "act3": 9 * C, "act4": 9 * C, "f1": (n - 4) ** 2 * C, "f2": 1024}[name]
    return (K + 3) * U32 * M


def _mismatch(dev, emu, delta):
    """(fraction of differing elements, number of differences that are neither adjacent bf16 codes nor within
    2 * delta).  Activations are non-negative, so their bf16 codes are ordered like their values."""
    diff = dev != emu
    if not diff.any():
        return 0.0, 0
    cd = dev[diff].view(np.uint32) >> 16
    ce = emu[diff].view(np.uint32) >> 16
    ok = (np.abs(cd.astype(np.int64) - ce.astype(np.int64)) <= 1) | (np.abs(dev[diff] - emu[diff]) <= 2 * delta[diff])
    return float(diff.mean()), int((~ok).sum())


def _check_batch(e, blob, own, opp, n, C, conv2, conv3, act2=None):
    """Every layer of one forward on `e` against the emulation fed the device's input to that layer.  For the
    Winograd conv3, act2 is never stored: `act2` is then the act2 of a direct-conv3 engine on the same boards, which runs
    the same gather code (t2_square) and so computes the very values the Winograd gather transforms.  It is checked
    against the emulation too: a gather bug shared by both engines would otherwise go unseen.
    -> {layer: fraction of differing elements}."""
    B = own.size
    pi, lg, v = e.net_forward(own, opp)
    first = {"gemm": 0, "table": 1}[conv2] + (conv3 == "wino")
    dev = {name: e.activation(li, B, *_shape(name, n, C)) for li, name in enumerate(LAYERS) if li >= first}
    if act2 is not None:
        dev["act2"] = act2
    mags = {}
    epi, elg, ev, hid = fp8_emul.forward(blob, own, opp, n, C, precision="bf16", conv2=conv2, conv3=conv3, inject=dev,
                                         magnitudes=mags)
    fracs = {}
    if "act1" in dev:
        assert np.array_equal(dev["act1"], hid["act1"]), "act1 differs from the conv1 table rows"
    for name in LAYERS[1:]:
        d = _delta(name, n, C, conv2, conv3, mags[name])
        frac, bad = _mismatch(dev[name], hid[name], d)
        fracs[name] = frac
        where = np.argwhere(dev[name] != hid[name])[:4].tolist()
        assert bad == 0 and frac <= FRAC_MAX, (
            f"{name} (n={n} C={C} conv2={conv2} conv3={conv3} B={B}): {bad} elements beyond one bf16 step and "
            f"2 * delta, {frac:.3e} of elements differ; first differences at [board, row, channel] {where}")
    # the heads from the device's f2: logits and value within the fp32 summation bound, the policy from the logits
    dl = (512 + 3) * U32 * mags["logits"]
    assert (np.abs(lg - elg) <= dl).all(), np.abs(lg - elg).max()
    dv = (512 + 3) * U32 * mags["v"] + 4 * U32
    assert (np.abs(v - ev) <= dv).all(), np.abs(v - ev).max()
    assert np.abs(pi - epi).max() <= 2 * float(dl.max()) + 1e-6
    assert np.allclose(pi.sum(axis=1), 1.0, atol=1e-5)
    return fracs


def _check(n, C, conv2="table", conv3="direct", randomize_bn=True, seed=0):
    """B = 1 on a fresh engine, then B = max_games = B_RAGGED.  Prints the fraction of differing elements per layer."""
    from othellozero_b200 import net
    blob = net.init_weights(n, C, seed=seed, randomize_bn=randomize_bn)
    own, opp = _positions(n, B_RAGGED + 1, seed)
    batches = [(own[-1:], opp[-1:]), (own[:B_RAGGED], opp[:B_RAGGED])]
    e = _engine(n, C, blob, conv2, conv3)
    ref = _engine(n, C, blob, "table", "direct") if conv3 == "wino" else None
    try:
        for o, p in batches:
            act2 = None
            if ref is not None:
                ref.net_forward(o, p, want_logits=False)
                act2 = ref.activation(1, o.size, n * n, C)
            fr = _check_batch(e, blob, o, p, n, C, conv2, conv3, act2)
            print(f"flips n={n} C={C} conv2={conv2} conv3={conv3} bn={randomize_bn} B={o.size}: "
                  + " ".join(f"{k}={v:.2e}" for k, v in fr.items()))
    finally:
        e.close()
        if ref is not None:
            ref.close()


CASES = ([(6, 384, "table", "wino", True), (8, 640, "table", "wino", True), (8, 896, "table", "wino", True),
          (6, 1024, "table", "wino", True)]
         + [(8, 384, "gemm", "direct", True), (6, 512, "gemm", "direct", True), (6, 896, "gemm", "direct", True)]
         + [(8, 384, "table", "direct", False), (8, 512, "table", "direct", False)]
         + [(n, C, "table", "direct", True) for n in (6, 8) for C in CHANNELS])


@pytest.mark.parametrize("n,C,conv2,conv3,randomize_bn", CASES)
def test_bf16_tower_matches_emulation(n, C, conv2, conv3, randomize_bn):
    """C % 256 == 128 runs conv3 and conv4 (and the conv2 GEMM) on the one-SM GEMM with 128-column tiles and an odd
    number of n tiles; C % 256 == 0 on the SM-pair GEMM.  fc1 and fc2 always run on the SM-pair GEMM, the heads on the
    one-SM GEMM.  The gather covers C in ceil(C / 256) 16-byte chunks per lane."""
    _check(n, C, conv2, conv3, randomize_bn, seed=C + n)


@pytest.mark.parametrize("var,cases", [
    ("OZ_NET_NO_2SM", [(8, 512, "table", "direct"), (6, 256, "gemm", "direct")]),    # conv3..fc2 on the one-SM GEMM
    ("OZ_NET_NO_SPLIT", [(8, 384, "table", "direct"), (6, 384, "gemm", "direct")]),  # whole-board tiles only
])
def test_bf16_tower_matches_emulation_in_process_modes(var, cases):
    # a fresh process: these variables are read once per process
    code = (f"import sys\nsys.path.insert(0, {HERE!r})\nimport test_gpu_net_bf16 as t\n"
            f"for n, C, c2, c3 in {cases!r}:\n    t._check(n, C, c2, c3, seed=C + n)\nprint('CHECKED')\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, **{var: "1"}), capture_output=True,
                         text=True, timeout=1800)
    print(out.stdout)
    assert out.returncode == 0 and "CHECKED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


@pytest.mark.parametrize("n,C", [(8, 384), (6, 512)])
def test_bf16_no_pdl_and_fused_tail_are_bit_identical(n, C, monkeypatch):
    """OZ_NET_NO_PDL=1 and OZ_NET_TAIL=fused (read per engine) change launches, not arithmetic."""
    from othellozero_b200 import net
    blob = net.init_weights(n, C, seed=40 + C, randomize_bn=True)
    own, opp = _positions(n, B_RAGGED, 40)
    outs = []
    for env in ({}, {"OZ_NET_NO_PDL": "1"}, {"OZ_NET_TAIL": "fused"}):
        for k in ("OZ_NET_NO_PDL", "OZ_NET_TAIL"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = _engine(n, C, blob)
        pi, lg, v = e.net_forward(own, opp)
        outs.append([pi, lg, v] + [e.activation(li, B_RAGGED, *_shape(LAYERS[li], n, C)) for li in range(1, 6)])
        e.close()
    names = ["pi", "logits", "v"] + LAYERS[1:]
    for other, mode in zip(outs[1:], ("OZ_NET_NO_PDL=1", "OZ_NET_TAIL=fused")):
        for a, b, name in zip(outs[0], other, names):
            assert np.array_equal(a, b), f"{name} differs with {mode}"
