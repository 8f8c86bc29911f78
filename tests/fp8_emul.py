"""Host emulation of the network tower in torch on the CPU, in both precisions the device runs: the bf16 tower (the
default) and the FP8 tower (DESIGN.md 13).

It follows the device pipeline step by step and reproduces every rounding it makes.  Both precisions share:

- conv1 table: fp32 taps in order, BN fold, ReLU, bf16.
- conv1∘conv2 table: the per-tap products table1 . W2'^T.  Even channels are rounded to bf16.  Odd channels use the fused
  pair encoding of pack_pair_fused (oz_net.cu).
- the gather: bias, then taps 0..8 added in order in fp32.
- fc2 and the heads: bf16 weights, fp32 accumulation, the bf16 f2.

FP8 (precision="fp8"), given the device's scales (Engine.fp8_scales):

- act2 = e4m3(relu(acc) * (1 / sa_2)).
- conv3, conv4: e4m3 x e4m3 products (exact) summed, then e4m3(relu(fma(acc, alpha, beta))), with alpha and beta
  computed in fp32 exactly as the device computes them.
- fc1: the same with a bf16 output.

bf16 (precision="bf16"):

- act2 = bf16(relu(acc)).
- conv3, conv4, fc1: bf16(W * s) weights (fold_weights_kernel), exact products summed, then bf16(relu(acc + bias')) with
  one fp32 add (the add.f32x2 + cvt.rn.relu.bf16x2 epilogue of both GEMM kernels).
- conv2="gemm" (OZ_NET_CONV2=gemm): act1 is the conv1 table row of each square's pattern, and conv2 is the same bf16
  GEMM and epilogue over act1, with zero padding.
- conv3="wino" (OZ_NET_CONV3=wino): F(2,3) over ky.  U = bf16 of g0, (g0+g1+g2)*0.5, (g0-g1+g2)*0.5 and g2 in fp32
  (wino_weights_kernel); V = bf16 of the differences d0-d2, d1+d2, d2-d1, d1-d3 of bf16 act2 rows; four exact product
  sums M0..M3; rows 2ty and 2ty+1 = bf16(relu(((M0+M1)+M2)+b)) and bf16(relu(((M1-M2)-M3)+b)) in fp32 in that order.

The sums of exact products are taken in float64 and rounded once to fp32.  The device sums in fp32 in the tensor core's
order, so the two agree up to that summation order.  That difference is far below an e4m3 or bf16 step, so it flips a
rounding only where a value sits almost exactly on a rounding boundary.

quantize=False switches every rounding off.  What remains is the BN-folded fp32 network, which must agree with
oracle/net_torch.py.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle import net_torch

E4M3_MAX = 448.0
BN_EPS = np.float32(1e-3)


def _bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float32)


def _e4m3(x: torch.Tensor) -> torch.Tensor:
    """round-to-nearest e4m3 with satfinite, as float32."""
    return x.to(torch.float32).clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(torch.float32)


def _pair_fused(even: torch.Tensor, odd: torch.Tensor) -> torch.Tensor:
    """pack_pair_fused (oz_net.cu): the fp32 value the gather adds for an odd table channel."""
    lo = (even.to(torch.bfloat16).view(torch.int16).to(torch.int64)) & 0xFFFF
    ob = odd.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    sign = ob & 0x80000000
    m = ((ob & 0x7FFFFFFF) - lo + 32768).clamp(min=0)
    mag = (m & 0xFFFF0000) | lo
    mag = torch.where(mag >= 0x7F800000, 0x7F7F0000 | lo, mag)
    w = (sign | mag).to(torch.int64)
    w = torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)
    return w.view(torch.float32)


def _div32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Correctly rounded fp32 a / b, as CUDA's `/` is.  torch's vectorised float32 division and sqrt on the CPU are not
    always correctly rounded; through float64 they are, since 53 >= 2 * 24 + 2 bits."""
    return (a.double() / b.double()).to(torch.float32)


def _fma32(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """fp32 fma(a, b, c) via float64 (exact product, one float64 rounding, then fp32)."""
    return (a.double() * b.double() + c.double()).to(torch.float32)


def _params(blob, n: int, C: int):
    return [t.clone() for t in net_torch._split(blob, n, C, "cpu")]


def _bn_scale(g, v):
    """gamma / sqrtf(var + eps), each step correctly rounded in fp32."""
    return _div32(g, torch.sqrt((v + torch.tensor(BN_EPS)).double()).to(torch.float32))


def _fold(k2d, b, g, be, mu, va):
    """Keras [K][O] kernel -> W'[O][K] fp32 and bias' [O] as fold_weights_kernel computes them."""
    s = _bn_scale(g, va)
    W = (k2d * s[None, :]).t().contiguous()
    bias = _fma32(b - mu, s, be)
    return W, bias


def weight_scales(blob, n: int, C: int) -> dict:
    """Per-output-channel weight scales amax_k |W'[o][k]| / 448 (1 for an all-zero channel) of conv3, conv4, fc1."""
    p = _params(blob, n, C)
    out = {}
    for name, base in (("conv3", 12), ("conv4", 18), ("fc1", 24)):
        k = p[base]
        W, _ = _fold(k.reshape(-1, k.shape[-1]), *p[base + 1:base + 6])
        m = W.abs().amax(dim=1)
        out[name] = torch.where(m > 0, _div32(m, torch.tensor(np.float32(E4M3_MAX))), torch.ones_like(m)).numpy()
    return out


def patterns(own, opp, n: int) -> np.ndarray:
    """[B, n, n] 3x3-neighbourhood pattern of every square (0 empty/outside, 1 own, 2 opp; digit t = ky*3+kx)."""
    x = net_torch.boards_from_bits(own, opp, n)
    s = x[..., 0] + 2 * x[..., 1]
    sp = np.pad(s, ((0, 0), (1, 1), (1, 1)))
    pat = np.zeros(s.shape, dtype=np.int64)
    mul = 1
    for t in range(9):
        ky, kx = divmod(t, 3)
        pat += sp[:, ky:ky + n, kx:kx + n].astype(np.int64) * mul
        mul *= 3
    return pat


def _conv3x3(x: torch.Tensor, W: torch.Tensor, pad: int, want_mag: bool):
    """x [B, H, W, Cin], W [O][(ky, kx, ci)] -> (exact sum of products rounded to fp32 [B, OH, OW, O], sum of |products|
    in fp32 or None)."""
    w4 = W.reshape(-1, 3, 3, x.shape[-1]).permute(0, 3, 1, 2)           # OIHW from [o][(ky, kx, ci)]
    xc = x.permute(0, 3, 1, 2)
    acc = F.conv2d(xc.double(), w4.double(), padding=pad).to(torch.float32).permute(0, 2, 3, 1)
    mag = F.conv2d(xc.abs(), w4.abs(), padding=pad).permute(0, 2, 3, 1) if want_mag else None
    return acc, mag


def _wino_conv3(x: torch.Tensor, k: torch.Tensor, s: torch.Tensor, bias: torch.Tensor, rnd, want_mag: bool):
    """conv3 as 1-D Winograd F(2,3) over ky, as wino_weights_kernel, the gather's input transform and oz_wino_kernel
    compute it.  x = act2 [B, n, n, C], k = the Keras kernel [3, 3, C, C] (HWIO), s = the BN scale.
    -> (act3 [B, n-2, n-2, C], the sum of |terms| of each output or None)."""
    B, n, _, C = x.shape
    T = (n - 2) // 2
    g = k * s                                                            # g[ky][kx][ci][co] = W * s in fp32
    U = [rnd(g[0]), rnd((g[0] + g[1] + g[2]) * 0.5), rnd((g[0] - g[1] + g[2]) * 0.5), rnd(g[2])]
    d = [x[:, r:r + 2 * T:2] for r in range(4)]                          # rows 2ty + r: [B, T, n, C]
    V = [rnd(d[0] - d[2]), rnd(d[1] + d[2]), rnd(d[2] - d[1]), rnd(d[1] - d[3])]
    m, mag = [], []
    for e in range(4):  # M_e[b, ty, xo, co] = sum over kx, ci of V_e[b, ty, xo + kx, ci] * U_e[kx, ci, co]
        v = V[e].reshape(B * T, n, C).permute(0, 2, 1)
        u = U[e].permute(2, 1, 0)                                        # [co, ci, kx]
        m.append(F.conv1d(v.double(), u.double()).to(torch.float32).permute(0, 2, 1).reshape(B, T, n - 2, C))
        if want_mag:
            mag.append(F.conv1d(v.abs(), u.abs()).permute(0, 2, 1).reshape(B, T, n - 2, C))
    y0 = rnd(torch.relu(((m[0] + m[1]) + m[2]) + bias))                   # output row 2ty
    y1 = rnd(torch.relu(((m[1] - m[2]) - m[3]) + bias))                   # output row 2ty + 1
    y = torch.stack([y0, y1], dim=2).reshape(B, n - 2, n - 2, C)
    if not want_mag:
        return y, None
    b = bias.abs()
    return y, torch.stack([mag[0] + mag[1] + mag[2] + b, mag[1] + mag[2] + mag[3] + b], dim=2).reshape(B, n - 2, n - 2, C)


@torch.no_grad()
def forward(blob, own, opp, n: int, C: int, scales: dict | None = None, quantize: bool = True, inject: dict | None = None,
            precision: str = "fp8", conv2: str = "table", conv3: str = "direct", magnitudes: dict | None = None):
    """-> (pi [B, n*n], logits [B, n*n], v [B], hidden) as numpy.  hidden[name] is each layer's output [B, rows, channels]
    for name in act1 (conv2="gemm" only), act2, act3, act4, f1 and f2.  The FP8 tower's act2, act3 and act4 are in e4m3
    units of their scales (quantize=True); everything else is in real units.
    precision="bf16" emulates the bf16 tower, with conv2 "table" (the gather) or "gemm" (OZ_NET_CONV2=gemm: act1 is the
    conv1 table row of each square's pattern) and conv3 "direct" or "wino" (OZ_NET_CONV3=wino).
    inject = {name: [B, rows, channels]} passes that value to the next layer instead of the emulation's own, for example
    the device's, so that each layer can be checked on exactly the input the device gave it.  hidden[name] stays the
    emulation's own value, so one call that injects every activation checks every layer.
    magnitudes: a dict, filled for the bf16 tower with M = |bias| + sum |terms| of every output element of act2, act3,
    act4, f1, f2, logits and v: the scale of the fp32 summation error of that element (for the gather's act2, sum |terms|
    is over the nine table entries)."""
    if precision not in ("fp8", "bf16") or conv2 not in ("table", "gemm") or conv3 not in ("direct", "wino"):
        raise ValueError((precision, conv2, conv3))
    fp8 = precision == "fp8"
    if fp8 and (conv2, conv3) != ("table", "direct"):
        raise ValueError("the FP8 tower runs the table gather and the direct conv3 only")
    inject = inject or {}
    want = magnitudes is not None and not fp8
    p = _params(blob, n, C)
    q = _e4m3 if quantize else (lambda t: t)
    bf = _bf16 if quantize else (lambda t: t)
    B = np.asarray(own).size
    hidden = {}

    def out(name, y):
        hidden[name] = y.reshape(B, -1, y.shape[-1]).numpy()
        return torch.as_tensor(np.asarray(inject[name], dtype=np.float32)).reshape(y.shape) if name in inject else y

    # conv1 table rows of the patterns present, fp32 taps in order (conv1_table_kernel)
    pat = patterns(own, opp, n)
    uniq, inv = np.unique(pat, return_inverse=True)
    digits = np.stack([(uniq // 3 ** t) % 3 for t in range(9)], axis=1)     # [U, 9]
    w1 = p[0].reshape(9, 2, C)
    acc = torch.zeros(len(uniq), C)
    for t in range(9):
        d = torch.as_tensor(digits[:, t])
        acc = acc + torch.where((d == 1)[:, None], w1[t, 0][None], torch.zeros(C)) \
                  + torch.where((d == 2)[:, None], w1[t, 1][None], torch.zeros(C))
    s1 = _bn_scale(p[2], p[5])
    table1 = bf(torch.relu(_fma32(acc + p[1] - p[4], s1, p[3])))           # [U, C]
    W2, b2 = _fold(p[6].reshape(9 * C, C), *p[7:12])
    W2 = bf(W2)
    if conv2 == "table":
        # conv1∘conv2 table: T[u][t][co] = W2'[co][t*C:(t+1)*C] . table1[u]
        T = torch.einsum("uc,otc->uto", table1.double(), W2.reshape(C, 9, C).double()).to(torch.float32)  # [U, 9, C]
        if quantize:
            Te = T.clone()
            Te[..., 0::2] = _bf16(T[..., 0::2])
            Te[..., 1::2] = _pair_fused(T[..., 0::2], T[..., 1::2])
            T = Te
        # gather: bias, then taps in order; an off-board neighbour adds the zero row
        Tb = torch.as_tensor(T)[torch.as_tensor(inv.reshape(B, n, n))]      # [B, n, n, 9, C]
        Tp = F.pad(Tb, (0, 0, 0, 0, 1, 1, 1, 1))                           # zero squares around the board
        acc = b2.expand(B, n, n, C).clone()
        mag = b2.abs().expand(B, n, n, C).clone()
        for t in range(9):
            ky, kx = divmod(t, 3)
            # output (y, x) reads tap t of the square (y + ky - 1, x + kx - 1) = padded (y + ky, x + kx)
            acc = acc + Tp[:, ky:ky + n, kx:kx + n, t, :]
            mag = mag + Tp[:, ky:ky + n, kx:kx + n, t, :].abs()
    else:
        # conv1 gather (act1 = table1 row of the square's pattern), then conv2 as an implicit GEMM with zero padding
        x = out("act1", table1[torch.as_tensor(inv.reshape(B, n, n))])
        acc, mag = _conv3x3(x, W2, 1, want)
        acc = acc + b2
        if want:
            mag = mag + b2.abs()
    if fp8 and quantize:
        sa = np.asarray(scales["act"], dtype=np.float32)
        inv_sa2 = torch.tensor(np.float32(1.0) / sa[0])
        x = _e4m3(torch.relu(acc) * inv_sa2)
    else:
        x = bf(torch.relu(acc))
    if want:
        magnitudes["act2"] = mag.reshape(B, n * n, C).numpy()
    x = out("act2", x)
    # conv3, conv4, fc1
    for li, (name, base) in enumerate((("conv3", 12), ("conv4", 18), ("fc1", 24))):
        k = p[base]
        key = ("act3", "act4", "f1")[li]
        W, bias = _fold(k.reshape(-1, k.shape[-1]), *p[base + 1:base + 6])
        if not fp8:
            if name == "conv3" and conv3 == "wino":
                y, mag = _wino_conv3(x, k, _bn_scale(p[base + 2], p[base + 5]), bias, bf, want)
            else:
                if name == "fc1":
                    xf = x.reshape(B, -1)
                    accl = (xf.double() @ bf(W).double().t()).to(torch.float32)
                    mag = xf.abs() @ bf(W).abs().t() if want else None
                else:
                    accl, mag = _conv3x3(x, bf(W), 0, want)
                y = bf(torch.relu(accl + bias))
                if want:
                    mag = mag + bias.abs()
            if want:
                magnitudes[key] = mag.reshape(B, -1, mag.shape[-1]).numpy()
            x = out(key, y)
            continue
        if quantize:
            sw = torch.as_tensor(np.asarray(scales[name], dtype=np.float32))
            Wq = _e4m3(_div32(W, sw[:, None]))
            sa_in = torch.tensor(sa[li])
            sa_out = torch.tensor(sa[li + 1] if li < 2 else np.float32(1.0))
            alpha, beta = _div32(sa_in * sw, sa_out), _div32(bias, sa_out)
        else:
            Wq, alpha, beta = W, torch.ones_like(bias), bias
        if name == "fc1":
            accl = (x.reshape(B, -1).double() @ Wq.double().t()).to(torch.float32)
            x = out(key, bf(torch.relu(_fma32(accl, alpha, beta))))
        else:
            accl, _ = _conv3x3(x, Wq, 0, False)
            x = out(key, q(torch.relu(_fma32(accl, alpha, beta))))
    # fc2 and heads: bf16 weights and activations, fp32 accumulation
    f1 = x
    W6, b6 = _fold(p[30], *p[31:36])
    f2 = out("f2", bf(torch.relu((f1.double() @ bf(W6).double().t()).to(torch.float32) + b6)))
    Wp, bp, Wv, bv = p[36], p[37], p[38], p[39]
    logits = (f2.double() @ bf(Wp).double()).to(torch.float32) + bp
    vpre = (f2.double() @ bf(Wv).double()).to(torch.float32).reshape(-1) + bv
    if want:
        magnitudes["f2"] = (f1.abs() @ bf(W6).abs().t() + b6.abs()).reshape(B, 1, -1).numpy()
        magnitudes["logits"] = (f2.abs() @ bf(Wp).abs() + bp.abs()).numpy()
        magnitudes["v"] = ((f2.abs() @ bf(Wv).abs()).reshape(-1) + bv.abs()).numpy()
    pi = torch.softmax(logits, dim=1)
    return pi.numpy(), logits.numpy(), torch.tanh(vpre).numpy(), hidden
