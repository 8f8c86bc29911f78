"""Host emulation of the FP8 tower (DESIGN.md 13) in torch on the CPU.

It follows the device pipeline step by step and reproduces every rounding it makes, given the device's scales
(Engine.fp8_scales):

- conv1 table: fp32 taps in order, BN fold, ReLU, bf16.
- conv1∘conv2 table: the per-tap products table1 . W2'^T.  Even channels are rounded to bf16.  Odd channels use the fused
  pair encoding of pack_pair_fused (oz_net.cu).
- the gather: bias, then taps 0..8 added in order in fp32, then act2 = e4m3(relu(acc) * (1 / sa_2)).
- conv3, conv4: e4m3 x e4m3 products (exact) summed, then e4m3(relu(fma(acc, alpha, beta))), with alpha and beta
  computed in fp32 exactly as the device computes them.
- fc1: the same with a bf16 output.
- fc2 and the heads: bf16 weights, fp32 accumulation, the bf16 f2.

The sums of exact products are taken in float64.  The device sums in fp32 in the tensor core's order, so the two agree up
to that summation order.  That difference is far below an e4m3 step, so it flips a rounding only where a value sits
almost exactly on a rounding boundary.

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


@torch.no_grad()
def forward(blob, own, opp, n: int, C: int, scales: dict | None = None, quantize: bool = True, inject: dict | None = None):
    """-> (pi [B, n*n], logits [B, n*n], v [B], hidden) as numpy.  hidden = [act2, act3, act4] ([B, rows, C]) in e4m3
    units of their scales (quantize=True) or in real units (quantize=False).
    inject = {"act2" | "act3" | "act4": [B, rows, C]} replaces the emulation's own value of that activation, for example
    with the device's, so that each layer can be checked on exactly the input the device gave it."""
    inject = inject or {}
    p = _params(blob, n, C)
    q = _e4m3 if quantize else (lambda t: t)
    bf = _bf16 if quantize else (lambda t: t)
    B = np.asarray(own).size
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
    # conv1∘conv2 table: T[u][t][co] = W2'[co][t*C:(t+1)*C] . table1[u]
    W2, b2 = _fold(p[6].reshape(9 * C, C), *p[7:12])
    W2 = bf(W2).reshape(C, 9, C)
    T = torch.einsum("uc,otc->uto", table1.double(), W2.double()).to(torch.float32)  # [U, 9, C]
    if quantize:
        Te = T.clone()
        Te[..., 0::2] = _bf16(T[..., 0::2])
        Te[..., 1::2] = _pair_fused(T[..., 0::2], T[..., 1::2])
        T = Te
    # gather: taps in order; an off-board neighbour adds the zero row
    Tb = torch.as_tensor(T)[torch.as_tensor(inv.reshape(B, n, n))]          # [B, n, n, 9, C]
    Tp = F.pad(Tb, (0, 0, 0, 0, 1, 1, 1, 1))                               # zero squares around the board
    acc = b2.expand(B, n, n, C).clone()
    for t in range(9):
        ky, kx = divmod(t, 3)
        # output (y, x) reads tap t of the square (y + ky - 1, x + kx - 1) = padded (y + ky, x + kx)
        acc = acc + Tp[:, ky:ky + n, kx:kx + n, t, :]
    if quantize:
        sa = np.asarray(scales["act"], dtype=np.float32)
        inv_sa2 = torch.tensor(np.float32(1.0) / sa[0])
        x = _e4m3(torch.relu(acc) * inv_sa2)
    else:
        x = torch.relu(acc)
    if "act2" in inject:
        x = torch.as_tensor(np.asarray(inject["act2"], dtype=np.float32)).reshape(x.shape)
    hidden = [x.reshape(B, n * n, C).numpy()]
    # conv3, conv4, fc1
    for li, (name, base) in enumerate((("conv3", 12), ("conv4", 18), ("fc1", 24))):
        k = p[base]
        W, bias = _fold(k.reshape(-1, k.shape[-1]), *p[base + 1:base + 6])
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
            f1 = bf(torch.relu(_fma32(accl, alpha, beta)))
        else:
            w4 = Wq.reshape(-1, 3, 3, C).permute(0, 3, 1, 2).double()       # OIHW from [o][(ky, kx, ci)]
            accl = F.conv2d(x.permute(0, 3, 1, 2).double(), w4).to(torch.float32).permute(0, 2, 3, 1)
            y = torch.relu(_fma32(accl, alpha, beta))
            x = q(y)
            key = "act3" if name == "conv3" else "act4"
            if key in inject:
                x = torch.as_tensor(np.asarray(inject[key], dtype=np.float32)).reshape(x.shape)
            hidden.append(x.reshape(B, -1, C).numpy())
    # fc2 and heads: bf16 weights and activations, fp32 accumulation
    W6, b6 = _fold(p[30], *p[31:36])
    f2 = bf(torch.relu((f1.double() @ bf(W6).double().t()).to(torch.float32) + b6))
    Wp, bp, Wv, bv = p[36], p[37], p[38], p[39]
    logits = (f2.double() @ bf(Wp).double()).to(torch.float32) + bp
    vpre = (f2.double() @ bf(Wv).double()).to(torch.float32).reshape(-1) + bv
    pi = torch.softmax(logits, dim=1)
    return pi.numpy(), logits.numpy(), torch.tanh(vpre).numpy(), hidden
