"""Float64 restatement of the tensor-core coupling network of the Glow prior, one launch at a time, and the gates that
hold each launch to it.

  * ``k_nn_tc4`` (csrc/nn_tc.cu; ASEP_PREC_BF16 / FP16) and ``k_nn_tcx`` (csrc/nn_tcx.cu; BF16X2 / FP16X2 / FP16X3):
    ShiftAndLogScaleConvNet (conv3x3 -> ReLU -> BN -> conv1x1 -> ReLU -> BN -> conv3x3) and its data gradient as three
    GEMMs per 128-pixel tile, the per-tap stage-3 outputs G in a tiled layout, col2im by the gather kernels;
  * ``k_wgrad_tc`` (csrc/wgrad_tc.cu): out[512, ldo] += A^T B over the pixels, split-K over the grid.

Weights.  ``TcNet`` restates GlowModel::prepare + nn_tc_prepare + build_stage_set: the BatchNorm fold g' =
float32(gamma / sqrt(var + 1e-3)) (float64 arithmetic), b' = float32(beta - g' mu); the float32 products g1'.K2 and
g2'.K3 that the tile images hold; their RN to bf16 or fp16; the residual images rn(w - rn(w)) of the three-product mode;
its x256 weight scale and 1/256 on the accumulators; bias2 = c2 + b1'.K2 and const3[tap] = b2'.K3[tap] summed in float64
in the host's order and stored as float32.

Which products each mode forms (from the kernels):
  * stage 1 is the im2col of the source as a split pair [x_hi | x_lo] against [W1 ; W1]: bf16 pairs and bf16 W1, except
    the FP16X3 forward, where x is split into fp16 pairs against fp16 W1 with the residual image [W1_lo ; 0]
    (x_hi . W1_lo only);
  * forward hidden activations: one bf16 word (BF16), one fp16 word (FP16), (hi, lo) pairs of bf16 (BF16X2) or fp16
    (FP16X2, FP16X3); stage-2/3 weights fp16 in the three fp16 modes, bf16 otherwise; FP16X3 adds hi . w_lo per GEMM;
  * the data gradient always runs on bf16 weights (bf16 residuals in FP16X3) with ReLU masks instead of bias + ReLU,
    one bf16 word per gradient in the one-product kernel, bf16 pairs in the split kernel;
  * the split kernel writes G as two K-split parts (hidden units 0-255 and 256-511 of the second layer), the gather
    adds them.

Gates.  Stage outputs are accumulated in fp32 in TMEM: one K = 16 tensor-core instruction after another into the same
accumulator, each adding its 16 exact products.  Along the path of any term there are at most ``steps`` accumulator
roundings plus at most 4 inside one instruction plus 1 in the epilogue (bias add, fma with the 1/256, or nothing), each
off by at most 2^-23 of the running magnitude (round-to-nearest gives 2^-24; 2^-23 also admits truncation), so
|got - ref| <= tau(steps) * A with tau(steps) = (steps + 5) * 2^-23 and A the sum of the magnitudes of the terms
(``acc_tau``).  Stages whose input the kernel hands out exactly (the bf16 dumps of the BF16 forward and of every
one-product backward) are checked this way, stage by stage.  Rounding to the activation format is monotone, so each bf16
dump must lie between the roundings of relu(ref - tau A) and relu(ref + tau A) (``bracket_violations``); a mask bit must
equal ref > 0 wherever |ref| > tau A.

Where the intermediates are not handed out (FP16, BF16X2, FP16X2, FP16X3 forward; the split-precision backward) G and
out are held to the magnitude chain (``chain_bounds``): with the activation unit u (2^-11 fp16, 2^-17 bf16 pairs, 2^-22
fp16 pairs) and eps the absolute error of an fp16 subnormal (2^-25; 0 for bf16), ReLU being 1-Lipschitz,
  e1 = (tau1 + 2u) m1 + eps,                        m1 = |W1||x| + |b1|
  d2 = (1 + tau2) |W2| e1 + tau2 m2,               m2 = |W2| m1 + |b2|
  e2 = (1 + u) d2 + u m2 + eps
  eG = (1 + tau3) |W3| e2 + tau3 |W3| m2            per G element
  eR = sum over the in-bounds taps of eG + 2^-20 m3, m3 = sum_tap (|W3| m2 + |const3|) + |c3|  (the gather: <= 11 fp32
                                                                                                  additions)
and every element must satisfy |got - ref| <= the bound.  Given its masks the data gradient is linear (the masks zero
the same elements in both), so its chain is the same with the masks applied and no biases.  Reported ratios are
|got - ref| / A (staged) or |got - ref| / bound (chain); the gates are tau and 1.  Worst ratios observed on a B200 are
listed next to each gate in ``WORST_OBSERVED``.

What the chain cannot see: a defect whose effect is a sum of rounding-sized errors of random sign.  Dropping the lo
word of the fp16 pairs in the forward (2^-11 per activation, summed over 512 hidden units with random signs: about
2^-16.5 of m2) stays under the worst-case accumulation term tau2 m2; the bf16 pairs' lo word (2^-9) does not.  In the
split-precision data gradient, which hands out no masks or dumps, a missing lo word or residual image is damped the
same way (its random-sign errors pass through |W| in the bound): there only the stage-1 defects, the layouts and the
tile hand-overs are caught.  The forward's masks catch a missing residual image of stage 1.

``emulate`` is a CPU restatement of each kernel's arithmetic (its operand roundings, float64 sums rounded to fp32 once
per stage): it must pass every gate, and with a planted defect it must not (tests/test_oracle_coupling_tc.py).
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

from .glow_oracle import BN_EPS

HID = 512                # hidden width of the tensor-core kernels
TILE = 128               # pixels per tile
U23 = 2.0 ** -23
GATHER_TAU = 2.0 ** -20  # the col2im sums: <= 9 taps x (part + const3) + c3 -> at most 11 fp32 additions of 2^-24 each
MODES = ("bf16", "fp16", "bf16x2", "fp16x2", "fp16x3")

# Worst ratio observed per gate over tests/test_gpu_coupling_tc.py (`pytest -m gpu ... -s`) on an NVIDIA B200 at a
# 1000 W power limit.  Staged gates: |got - ref| / A against tau(steps) (4.4e-6 for the 32-step stage 3); chain gates and
# the weight gradient: |got - ref| / bound against 1.  Every bracket, mask and bitwise-gather count was 0.
WORST_OBSERVED: Dict[str, float] = {
    "k_nn_tc4<fwd> bf16 G (staged)": 3.2e-7, "k_nn_tc4<bwd> bf16 G (staged)": 3.2e-7,
    "k_nn_tc4<bwd> fp16 G (staged)": 2.8e-7,
    "k_nn_tc4<fwd> fp16 G (chain)": 7.5e-4, "k_nn_tc4<fwd> fp16 out (chain)": 2.5e-4,
    "k_nn_tcx<fwd> bf16x2 G (chain)": 5.6e-4, "k_nn_tcx<fwd> fp16x2 G (chain)": 7.3e-4,
    "k_nn_tcx<fwd> fp16x3 G (chain)": 7.9e-4, "k_nn_tcx<fwd> out (chain, any mode)": 1.5e-4,
    "k_nn_tcx<bwd> bf16x2 G (chain)": 1.9e-3, "k_nn_tcx<bwd> fp16x2 G (chain)": 1.9e-3,
    "k_nn_tcx<bwd> fp16x3 G (chain)": 2.1e-3, "k_nn_tcx<bwd> out (chain, any mode)": 4.4e-4,
    "k_wgrad_tc (/ wgrad_tau)": 1.6e-1,
}


def spec(mode: str) -> dict:
    """What each precision mode forms (from nn_tc_prepare / nn_tc.cu / nn_tcx.cu)."""
    if mode not in MODES:
        raise ValueError(mode)
    pairs = mode in ("bf16x2", "fp16x2", "fp16x3")
    f16 = mode in ("fp16", "fp16x2", "fp16x3")
    x3 = mode == "fp16x3"
    return {"pairs": pairs, "f16": f16, "x3": x3, "f16_s1": x3, "wscale": 256.0 if x3 else 1.0, "nparts": 2 if pairs else 1}


def act_unit(mode: str, backward: bool) -> tuple:
    """(u, eps) of the hidden activations / gradients the kernel hands to the next GEMM."""
    s = spec(mode)
    if backward:
        return (2.0 ** -17 if s["pairs"] else 2.0 ** -9), 0.0
    if s["pairs"]:
        return (2.0 ** -22, 2.0 ** -25) if s["f16"] else (2.0 ** -17, 0.0)
    return (2.0 ** -11, 2.0 ** -25) if s["f16"] else (2.0 ** -9, 0.0)


def acc_tau(steps: int) -> float:
    """Gate of one fp32 TMEM accumulation over `steps` K = 16 instructions (module docstring)."""
    return (steps + 5) * U23


# ------------------------------------------------------------------ 16-bit formats
def rn(t, half: bool) -> torch.Tensor:
    """fp32 -> bf16 (half = False) or fp16 round-to-nearest-even, returned as fp32 values."""
    t = torch.as_tensor(t, dtype=torch.float32)
    return t.to(torch.float16 if half else torch.bfloat16).float()


def split(t, half: bool) -> tuple:
    """(hi, lo) = (rn(t), rn(t - hi)): the pair words of ``split_pair`` / the residual images (t - hi is exact)."""
    t = torch.as_tensor(t, dtype=torch.float32)
    hi = rn(t, half)
    return hi, rn(t - hi, half)


# ------------------------------------------------------------------ weights
def fold_bn(params, pre: str, name: str) -> tuple:
    """Inference-mode BatchNorm as GlowModel::prepare folds it: (g', b') float32 from float64 arithmetic."""
    g = {k: np.asarray(params[f"{pre}nn/{name}/{k}"], np.float32).astype(np.float64)
         for k in ("gamma", "beta", "moving_mean", "moving_variance")}
    gg = g["gamma"] / np.sqrt(g["moving_variance"] + BN_EPS)
    return torch.from_numpy(gg.astype(np.float32)), torch.from_numpy((g["beta"] - gg * g["moving_mean"]).astype(np.float32))


def _seq_sum(init: np.ndarray, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """float64 init + sum_k a[k] * b[k] added in k order (the host loops of nn_tc_prepare), as float32."""
    acc = init.astype(np.float64).copy()
    a, b = a.astype(np.float64), b.astype(np.float64)
    for k in range(a.shape[0]):
        acc = acc + a[k] * b[k]
    return acc.astype(np.float32)


class TcNet:
    """The weights one coupling network of a prepared model multiplies by in one precision mode.

    For each direction ``w[d]`` (d = "fwd" / "bwd") holds the three stages as [K, N] float32 tensors (hi, lo) -- lo is
    None outside FP16X3 -- and ``scale``, the factor on every accumulator (1/256 in the FP16X3 forward).  ``raw`` keeps
    the float32 weights before rounding (k1 [9Ch, F], g1'.K2 [F, F], g2'.K3 [F, 9C])."""

    def __init__(self, params, pre: str, C: int, mode: str):
        s = spec(mode)
        self.C, self.mode, self.spec = C, mode, s
        Ch = C // 2
        f32 = lambda n: torch.as_tensor(np.asarray(params[pre + n], np.float32))  # noqa: E731
        k1 = f32("nn/conv1/kernel").reshape(9 * Ch, HID)            # [tap*Ch + ci, n]
        k2 = f32("nn/conv2/kernel").reshape(HID, HID)               # [in, out]
        k3 = f32("nn/conv3/kernel").reshape(9, HID, C)              # [tap, k, c]
        g1, b1 = fold_bn(params, pre, "bn1")
        g2, b2 = fold_bn(params, pre, "bn2")
        w2 = g1[:, None] * k2                                       # float32 products g1'[k] K2[k][n]
        w3 = g2[None, :, None] * k3                                 # g2'[k] K3[tap][k][c]
        self.raw = {"k1": k1, "w2": w2, "w3": w3.permute(1, 0, 2).reshape(HID, 9 * C)}
        ws = s["wscale"]

        def stage(w, half, scale=1.0):
            v = w * scale                                           # exact: a power of two
            hi, lo = split(v, half)
            return hi, (lo if s["x3"] else None)

        self.w = {
            "fwd": {"s1": stage(k1, s["f16_s1"], ws), "s2": stage(w2, s["f16"], ws),
                    "s3": stage(self.raw["w3"], s["f16"], ws), "scale": 1.0 / ws},
            "bwd": {"s1": stage(w3.permute(0, 2, 1).reshape(9 * C, HID), False),     # [tap*C + c, n] = g2'[n] K3[tap][n][c]
                    "s2": stage(w2.T.contiguous(), False),                           # [k, n] = g1'[n] K2[n][k]
                    "s3": stage(k1.T.contiguous(), False), "scale": 1.0},            # [k, tap*Ch + ci] = K1[tap][ci][k]
        }
        c2 = np.asarray(params[pre + "nn/conv2/bias"], np.float32)
        self.b1 = f32("nn/conv1/bias")
        self.b2 = torch.from_numpy(_seq_sum(c2, b1.numpy(), k2.numpy()))
        k3n = k3.numpy()
        self.const3 = torch.from_numpy(np.stack([_seq_sum(np.zeros(C), b2.numpy(), k3n[t]) for t in range(9)]).reshape(-1))
        self.c3 = f32("nn/conv3/bias")
        self.g2, self.bo2 = g2, b2
        self.g1, self.bo1 = g1, b1
        self.n3p = {"fwd": _pad16(9 * C), "bwd": _pad16(9 * Ch)}

    def to(self, device) -> "TcNet":
        mv = lambda t: None if t is None else t.to(device)  # noqa: E731
        for d in self.w.values():
            for k in ("s1", "s2", "s3"):
                d[k] = (mv(d[k][0]), mv(d[k][1]))
        for k in ("b1", "b2", "const3", "c3"):
            setattr(self, k, getattr(self, k).to(device))
        return self

    def k1_steps(self, backward: bool) -> int:
        src = self.C if backward else self.C // 2
        return (2 * 9 * src + 15) // 16

    def steps(self, backward: bool) -> dict:
        """K = 16 instructions accumulated into each output of each stage (stage 3: per K-split part in the split
        kernel)."""
        s = self.spec
        x3 = s["x3"]
        k1 = self.k1_steps(backward) * (2 if x3 else 1)
        if not s["pairs"]:
            return {"s1": k1, "s2": 32, "s3": 32}
        return {"s1": k1, "s2": 64 + (32 if x3 else 0), "s3": 32 + (16 if x3 else 0)}

    def fp32_net(self, xb: torch.Tensor):
        """The network on the float32 weights before any 16-bit rounding, in float64: (tanh(r[:C/2]), r[C/2:]), the
        form of GlowOracle.nn."""
        N, H, W, Ch = xb.shape
        C = 2 * Ch
        x = im2col(torch.cat([torch.zeros_like(xb), xb], -1), C, False)
        a1 = torch.relu(x.double() @ self.raw["k1"].double() + self.b1.double())
        a2 = torch.relu(a1 @ self.raw["w2"].double() + self.b2.double())
        G = a2 @ self.raw["w3"].double()
        r = gather_fwd([G.reshape(N * H * W, 9 * C)], self.const3.double(), self.c3.double(), N, H, W, C, exact=True)
        return torch.tanh(r[..., :Ch]), r[..., Ch:]


def _pad16(n: int) -> int:
    return (n + 15) // 16 * 16


# ------------------------------------------------------------------ layouts
def im2col(src: torch.Tensor, C: int, backward: bool, tap_sign: Optional[int] = None, src_off: Optional[int] = None,
           swap_dxdy: bool = False) -> torch.Tensor:
    """Stage-1 rows [M, 9*src_ch] (column tap*src_ch + ci): forward reads channels C/2.. of pixel p + off(tap), the data
    gradient all C channels of p - off(tap); off(tap) = (tap // 3 - 1, tap % 3 - 1), zero outside the image.  The
    keyword arguments plant the defects of tests/test_oracle_coupling_tc.py."""
    N, H, W, _ = src.shape
    sign = tap_sign if tap_sign is not None else (-1 if backward else 1)
    off = src_off if src_off is not None else (0 if backward else C // 2)
    ch = C if backward else C // 2
    x = F.pad(src[..., off:off + ch], (0, 0, 1, 1, 1, 1))
    cols = []
    for tap in range(9):
        dy, dx = (tap // 3 - 1) * sign, (tap % 3 - 1) * sign
        if swap_dxdy:
            dy, dx = dx, dy
        cols.append(x[:, 1 + dy:1 + dy + H, 1 + dx:1 + dx + W, :])
    return torch.cat(cols, -1).reshape(N * H * W, 9 * ch)


def tile_g(rows: torch.Tensor) -> torch.Tensor:
    """[Mp, n3p] (Mp a multiple of 128) -> the flat tiled layout [tile][n3p/4][128 rows][4]."""
    Mp, n3p = rows.shape
    return rows.reshape(Mp // TILE, TILE, n3p // 4, 4).permute(0, 2, 1, 3).reshape(-1)


def untile_g(flat: torch.Tensor, n3p: int) -> torch.Tensor:
    """Inverse of ``tile_g``."""
    t = flat.reshape(-1, n3p // 4, TILE, 4)
    return t.permute(0, 2, 1, 3).reshape(-1, n3p)


def pack_masks(bits: torch.Tensor) -> torch.Tensor:
    """ReLU bits [M, 512] (bool) -> int32 [M, 16]: word ch*8 + panel holds columns 64*panel + 32*ch + i in bit i."""
    M = bits.shape[0]
    b = bits.reshape(M, 8, 2, 32).permute(0, 2, 1, 3).to(torch.int64)           # [M, ch, panel, i]
    w = (b << torch.arange(32, device=bits.device)).sum(-1).reshape(M, 16)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)


def unpack_masks(words: torch.Tensor) -> torch.Tensor:
    """Inverse of ``pack_masks``."""
    M = words.shape[0]
    w = words.to(torch.int64) & 0xFFFFFFFF
    b = (w.reshape(M, 2, 8, 1) >> torch.arange(32, device=words.device)) & 1     # [M, ch, panel, i]
    return b.permute(0, 2, 1, 3).reshape(M, HID).bool()


def _tap_shift(G: torch.Tensor, N: int, H: int, W: int, dy: int, dx: int) -> tuple:
    """(values of G at pixel p + (dy, dx), in-bounds mask) as [N, H, W, cols]."""
    g = G.reshape(N, H, W, -1)
    gp = F.pad(g, (0, 0, 1, 1, 1, 1))
    ok = torch.zeros((1, H + 2, W + 2, 1), dtype=torch.bool, device=G.device)
    ok[:, 1:H + 1, 1:W + 1] = True
    sl = (slice(None), slice(1 + dy, 1 + dy + H), slice(1 + dx, 1 + dx + W))
    return gp[sl], ok[sl]


def gather_fwd(parts, const3, c3, N: int, H: int, W: int, C: int, exact: bool = False) -> torch.Tensor:
    """col2im of the forward in the gather kernels' float32 order: acc = c3; acc += (G0 [+ G1]) + const3 over the
    in-bounds taps p + off(tap).  parts: [M(+), n3p] rows per K-split part; exact = True: the same sums in float64."""
    dt = torch.float64 if exact else torch.float32
    M = N * H * W
    acc = c3.to(dt).expand(N, H, W, C).clone()
    for tap in range(9):
        dy, dx = tap // 3 - 1, tap % 3 - 1
        t = None
        for G in parts:
            v, ok = _tap_shift(G[:M, tap * C:(tap + 1) * C].to(dt), N, H, W, dy, dx)
            t = v if t is None else t + v
        t = t + const3[tap * C:(tap + 1) * C].to(dt)
        acc = torch.where(ok, acc + t, acc)
    return acc


def gather_bwd(parts, N: int, H: int, W: int, Ch: int, exact: bool = False) -> torch.Tensor:
    """col2im of the data gradient: gxb[p] = sum over the in-bounds taps of (G0' [+ G1'])[p - off(tap)][tap*Ch + ci],
    in the float32 order of k_gather_vec."""
    dt = torch.float64 if exact else torch.float32
    M = N * H * W
    acc = torch.zeros((N, H, W, Ch), dtype=dt, device=parts[0].device)
    for tap in range(9):
        dy, dx = tap // 3 - 1, tap % 3 - 1
        t = None
        for G in parts:
            v, ok = _tap_shift(G[:M, tap * Ch:(tap + 1) * Ch].to(dt), N, H, W, -dy, -dx)
            t = v if t is None else t + v
        acc = torch.where(ok, acc + t, acc)
    return acc


# ------------------------------------------------------------------ stage arithmetic
def _gemm(hi, lo, w, scale, absolute=False) -> torch.Tensor:
    """float64 [hi | lo] . [W_hi ; W_hi] + hi . W_lo, times the accumulator scale (absolute: of the magnitudes)."""
    f = (lambda t: t.double().abs()) if absolute else (lambda t: t.double())  # noqa: E731
    whi, wlo = w
    out = f(hi) @ f(whi)
    if lo is not None:
        out = out + f(lo) @ f(whi)
    if wlo is not None:
        out = out + f(hi) @ f(wlo)
    return out * scale


def stage1_operand(net: TcNet, src: torch.Tensor, backward: bool, **defect) -> tuple:
    """(x_hi, x_lo) of the stage-1 rows: split pairs of the im2col, fp16 in the FP16X3 forward, bf16 otherwise."""
    x = im2col(src.float(), net.C, backward, **defect)
    return split(x, net.spec["f16_s1"] and not backward)


def stage_ref(net: TcNet, backward: bool, stage: str, hi, lo, bias=None) -> tuple:
    """(ref, A) of one stage given the kernel's own operand words: float64 sum and sum of magnitudes (bias included)."""
    d = net.w["bwd" if backward else "fwd"]
    ref = _gemm(hi, lo, d[stage], d["scale"])
    A = _gemm(hi, lo, d[stage], d["scale"], absolute=True)
    if bias is not None:
        ref = ref + bias.double()
        A = A + bias.double().abs()
    return ref, A


def g_parts_ref(net: TcNet, backward: bool, hi, lo) -> list:
    """(ref, A) of stage 3 per K-split part (hidden units 256 q .. 256 q + 255 in the split kernel; one part else)."""
    d = net.w["bwd" if backward else "fwd"]
    whi, wlo = d["s3"]
    if net.spec["nparts"] == 1:
        return [stage_ref(net, backward, "s3", hi, lo)]
    out = []
    for q in range(2):
        ks = slice(256 * q, 256 * q + 256)
        w = (whi[ks], None if wlo is None else wlo[ks])
        out.append((_gemm(hi[:, ks], None if lo is None else lo[:, ks], w, d["scale"]),
                    _gemm(hi[:, ks], None if lo is None else lo[:, ks], w, d["scale"], absolute=True)))
    return out


# ------------------------------------------------------------------ CPU emulation of the kernels
DEFECTS = ("drop_k1", "drop_k2", "drop_k3", "tap_sign", "swap_dxdy", "read_xa", "no_x_lo", "no_h_lo", "no_w_lo",
           "no_inv_scale", "swap_mask_words", "stale_tile", "unwritten_tail_row")


def emulate(net: TcNet, src: torch.Tensor, backward: bool, masks=None, dumps: bool = True, defect: Optional[str] = None,
            drop_step: int = 1) -> dict:
    """What one launch writes, computed on the CPU with the kernel's operand roundings and float64 sums rounded to fp32
    once per stage: dump1 / dump2 (bf16 values as fp32, one-product modes), mask1 / mask2 (int32 words, forward), G
    ([nparts, flat] tiled; rows past M computed from zero stage-1 rows as the kernel does) and out.  ``masks`` (the
    backward's input): (mask1, mask2) int32 words.  ``defect`` plants one of ``DEFECTS``."""
    s = net.spec
    d = net.w["bwd" if backward else "fwd"]
    N, H, W, C = src.shape
    M = N * H * W
    Mp = (M + TILE - 1) // TILE * TILE
    kw = {}
    if defect == "tap_sign":
        kw["tap_sign"] = 1 if backward else -1
    if defect == "swap_dxdy":
        kw["swap_dxdy"] = True
    if defect == "read_xa":
        kw["src_off"] = 0
    xh, xl = stage1_operand(net, src, backward, **kw)
    pad = lambda t: F.pad(t, (0, 0, 0, Mp - M))  # noqa: E731
    xh, xl = pad(xh), pad(xl)
    if defect == "no_x_lo":
        xl = torch.zeros_like(xl)
    w = {k: d[k] for k in ("s1", "s2", "s3")}
    if defect == "no_w_lo":
        w = {k: (v[0], None) for k, v in w.items()}
    scale = 1.0 if defect == "no_inv_scale" else d["scale"]

    def acc(hi, lo, stage, drop):
        whi, wlo = w[stage]
        if drop:                                    # one 16-wide K step of this stage never issued
            k0 = 16 * drop_step
            hi = hi.clone(); hi[:, k0:k0 + 16] = 0
            if lo is not None:
                lo = lo.clone(); lo[:, k0:k0 + 16] = 0
        return _gemm(hi, lo, (whi, wlo), 1.0)

    half_act = s["f16"] and not backward
    mk_in = None
    if backward:
        mk_in = [F.pad(unpack_masks(m), (0, 0, 0, Mp - M)) for m in masks]

    def epilogue(a, bias, mask_in):
        """fp32 accumulator -> (stage-2/3 operand hi, lo or None, mask bits, bf16 dump)."""
        if backward:
            f = torch.where(mask_in, a.float(), torch.zeros((), dtype=torch.float32))
            bits = None
        else:
            f = (a * scale + bias.double()).float()           # acc + b (one product) / fmaf(acc, scale, b) (split)
            bits = f > 0
            f = torch.relu(f)
        if s["pairs"]:
            hi, lo = split(f, half_act)
            if defect == "no_h_lo":
                lo = torch.zeros_like(lo)
            return hi, lo, bits, None
        hi = rn(f, half_act)
        return hi, None, bits, rn(hi, False)

    a1 = acc(xh, xl, "s1", defect == "drop_k1").float().double()
    h1, l1, m1, dump1 = epilogue(a1, net.b1, mk_in[1] if backward else None)
    a2 = acc(h1, l1, "s2", defect == "drop_k2").float().double()
    h2, l2, m2, dump2 = epilogue(a2, net.b2, mk_in[0] if backward else None)
    parts = []
    if s["nparts"] == 1:
        parts.append((acc(h2, l2, "s3", defect == "drop_k3") * scale).float())
    else:
        for q in range(2):
            ks = slice(256 * q, 256 * q + 256)
            wq = {"s3": (w["s3"][0][ks], None if w["s3"][1] is None else w["s3"][1][ks])}
            whi, wlo = wq["s3"]
            hq, lq = h2[:, ks], None if l2 is None else l2[:, ks]
            if defect == "drop_k3" and q == 0:
                hq = hq.clone(); hq[:, 16 * drop_step:16 * drop_step + 16] = 0
                if lq is not None:
                    lq = lq.clone(); lq[:, 16 * drop_step:16 * drop_step + 16] = 0
            parts.append((_gemm(hq, lq, (whi, wlo), 1.0) * scale).float())
    n3p = net.n3p["bwd" if backward else "fwd"]
    parts = [F.pad(p, (0, n3p - p.shape[1])) for p in parts]
    if defect == "stale_tile" and Mp >= 2 * TILE:           # tile 1 still holds the previous round's rows (tile 0)
        parts = [torch.cat([p[:TILE], p[:TILE], p[2 * TILE:]]) for p in parts]
    if defect == "unwritten_tail_row":
        parts = [p.clone() for p in parts]
        for p in parts:
            p[M - 1] = float("nan")
    if backward:
        out = gather_bwd(parts, N, H, W, C // 2)
    else:
        out = gather_fwd(parts, net.const3, net.c3, N, H, W, C)
    res = {"G": torch.stack([tile_g(p) for p in parts]), "out": out}
    if not backward:
        mw = [pack_masks(m[:M]) for m in (m1, m2)]
        if defect == "swap_mask_words":
            for m in mw:
                m[:, [2, 3]] = m[:, [3, 2]]
        res["mask1"], res["mask2"] = mw
    if dumps and not s["pairs"]:
        if backward:                     # dump1 = dL/dp2 (stage-1 epilogue), dump2 = dL/dp1
            res["dump1"], res["dump2"] = rn(h1[:M], False), rn(h2[:M], False)
        else:
            res["dump1"], res["dump2"] = dump1[:M], dump2[:M]
    return res


# ------------------------------------------------------------------ gates
def _ratio(got, ref, A) -> float:
    got, ref, A = got.double(), ref.double().to(got.device), A.double().to(got.device)
    r = (got - ref).abs() / A.clamp_min(1e-300)
    r = torch.where(torch.isnan(got), torch.full_like(r, float("inf")), r)
    return float(r.max()) if r.numel() else 0.0


def bracket_violations(dump, ref, A, tau, backward: bool, half: bool = False) -> int:
    """Elements of a bf16 dump outside [rn(f(ref - tau A)), rn(f(ref + tau A))], f = relu (forward) or the identity
    (backward, where the masks have zeroed the same elements in ref): rounding is monotone.  half: the activations
    were fp16 first (rn_bf16(rn_fp16(.)) is monotone as well)."""
    f = (lambda t: t) if backward else torch.relu  # noqa: E731

    def r16(t):
        t = t.float()
        return rn(rn(t, True), False) if half else rn(t, False)

    lo, hi = r16(f(ref - tau * A)), r16(f(ref + tau * A))
    d = dump.float().to(lo.device)
    return int(((d < lo) | (d > hi) | torch.isnan(d)).sum())


def mask_violations(words, ref, bound) -> int:
    """Mask bits that differ from ref > 0 where |ref| exceeds the error bound of the pre-activation."""
    bits = unpack_masks(words.to(ref.device))
    return int(((bits != (ref > 0)) & (ref.abs() > bound)).sum())


def chain_bounds(net: TcNet, backward: bool, x_hi, x_lo, masks=None) -> dict:
    """Float64 reference and error bound of every G part and of out when the intermediates are not handed out (module
    docstring).  masks: (bits1, bits2) [Mp, 512] bool of the backward."""
    d = net.w["bwd" if backward else "fwd"]
    st = net.steps(backward)
    t1, t2, t3 = acc_tau(st["s1"]), acc_tau(st["s2"]), acc_tau(st["s3"])
    u, eps = act_unit(net.mode, backward)
    eff = lambda w: w[0].double() + (0 if w[1] is None else w[1].double())  # noqa: E731
    W2, W3 = eff(d["s2"]) * d["scale"], eff(d["s3"]) * d["scale"]
    b1 = None if backward else net.b1
    b2 = None if backward else net.b2
    ref1, m1 = stage_ref(net, backward, "s1", x_hi, x_lo, b1)
    k1 = masks[1].double() if backward else None
    k2 = masks[0].double() if backward else None
    a1 = ref1 * k1 if backward else torch.relu(ref1)
    e1 = (t1 + 2 * u) * m1 + eps
    if backward:
        e1, m1 = e1 * k1, m1 * k1
    ref2 = a1 @ W2 + (0 if b2 is None else b2.double())
    m2 = m1 @ W2.abs() + (0 if b2 is None else b2.double().abs())
    d2 = (1 + t2) * (e1 @ W2.abs()) + t2 * m2
    a2 = ref2 * k2 if backward else torch.relu(ref2)
    e2 = (1 + u) * d2 + u * m2 + eps
    if backward:
        e2, m2 = e2 * k2, m2 * k2
    out = {"ref1": ref1, "A1": m1, "ref2": ref2, "m2": m2, "d2": d2, "parts": []}
    ks = [slice(0, HID)] if net.spec["nparts"] == 1 else [slice(0, 256), slice(256, HID)]
    for k in ks:
        out["parts"].append((a2[:, k] @ W3[k], (1 + t3) * (e2[:, k] @ W3[k].abs()) + t3 * (m2[:, k] @ W3[k].abs()),
                             m2[:, k] @ W3[k].abs()))
    return out


def check_launch(net: TcNet, src: torch.Tensor, backward: bool, res: dict, masks=None) -> list:
    """Every gate of one launch: [(gate name, value, limit)], each passing when value <= limit.  res: what the launch
    wrote (``emulate`` or the kernel): G [nparts, flat], out, and mask1 / mask2 / dump1 / dump2 where they exist.
    masks: the backward's input words (mask1, mask2)."""
    s = net.spec
    N, H, W, C = src.shape
    M = N * H * W
    n3p = net.n3p["bwd" if backward else "fwd"]
    dev = src.device
    xh, xl = stage1_operand(net, src, backward)
    st = net.steps(backward)
    t1, t2, t3 = acc_tau(st["s1"]), acc_tau(st["s2"]), acc_tau(st["s3"])
    parts = [untile_g(res["G"][q], n3p)[:M] for q in range(s["nparts"])]
    ncols = 9 * C // 2 if backward else 9 * C
    gates = []
    bits = [unpack_masks(m.to(dev)) for m in masks] if backward else None
    exact = "dump1" in res and "dump2" in res and (backward or net.mode == "bf16")   # intermediates handed out exactly
    if exact:
        # staged: each stage from the kernel's own input words
        b1 = None if backward else net.b1
        ref1, A1 = stage_ref(net, backward, "s1", xh, xl, b1)
        if backward:
            ref1, A1 = ref1 * bits[1], A1 * bits[1]
        gates.append(("stage 1 dump outside its bracket", bracket_violations(res["dump1"], ref1, A1, t1, backward), 0))
        d1 = res["dump1"].to(dev).float()
        b2 = None if backward else net.b2
        ref2, A2 = stage_ref(net, backward, "s2", d1, None, b2)
        if backward:
            ref2, A2 = ref2 * bits[0], A2 * bits[0]
        gates.append(("stage 2 dump outside its bracket", bracket_violations(res["dump2"], ref2, A2, t2, backward), 0))
        if not backward:
            gates.append(("mask1 bits", mask_violations(res["mask1"], ref1, t1 * A1), 0))
            gates.append(("mask2 bits", mask_violations(res["mask2"], ref2, t2 * A2), 0))
        d2 = res["dump2"].to(dev).float()
        for q, (ref, A) in enumerate(g_parts_ref(net, backward, d2, None)):
            gates.append((f"G part {q} |got-ref|/A", _ratio(parts[q][:, :ncols], ref, A), t3))
    else:
        cb = chain_bounds(net, backward, xh, xl, [b[:M] for b in bits] if backward else None)
        if not backward and "mask1" in res:
            gates.append(("mask1 bits", mask_violations(res["mask1"], cb["ref1"], t1 * cb["A1"]), 0))
            gates.append(("mask2 bits", mask_violations(res["mask2"], cb["ref2"], cb["d2"]), 0))
        if "dump1" in res:            # FP16 forward: the stage-1 input is exact, its dump is rn_bf16(rn_fp16(.))
            gates.append(("stage 1 dump outside its bracket",
                          bracket_violations(res["dump1"], cb["ref1"], cb["A1"], t1, False, half=True), 0))
        for q, (ref, bound, _) in enumerate(cb["parts"]):
            gates.append((f"G part {q} |got-ref|/bound", _ratio(parts[q][:, :ncols], ref, bound), 1.0))
        if backward:
            eo = gather_bwd([p[1] for p in cb["parts"]], N, H, W, C // 2, exact=True)
            mo = gather_bwd([p[2] for p in cb["parts"]], N, H, W, C // 2, exact=True)
            ro = gather_bwd([p[0] for p in cb["parts"]], N, H, W, C // 2, exact=True)
        else:
            z = torch.zeros_like(net.const3, dtype=torch.float64)
            eo = gather_fwd([p[1] for p in cb["parts"]], z, z[:C], N, H, W, C, exact=True)
            mo = gather_fwd([p[2] for p in cb["parts"]], net.const3.double().abs(), net.c3.double().abs(), N, H, W, C,
                            exact=True)
            ro = gather_fwd([p[0] for p in cb["parts"]], net.const3, net.c3, N, H, W, C, exact=True)
        if res.get("out") is not None:
            gates.append(("out |got-ref|/bound", _ratio(res["out"], ro, eo + GATHER_TAU * mo), 1.0))
    if res.get("out") is not None:
        # the col2im of the kernel's own G, restated in float32 in the gather kernels' order: bitwise
        g = gather_bwd(parts, N, H, W, C // 2) if backward else gather_fwd(parts, net.const3, net.c3, N, H, W, C)
        o = res["out"].to(dev)
        gates.append(("out != gather(G) (elements)", int((g.view(torch.int32) != o.float().contiguous().view(torch.int32)).sum()), 0))
    return gates


def failed(gates: list) -> list:
    return [g for g in gates if not (g[1] <= g[2])]


# ------------------------------------------------------------------ weight gradient
def wgrad_split(P: int, ldb: int, sms: int = 148) -> tuple:
    """(slices, 64-pixel tiles per slice) of the split-K partition of wgrad_tc (host side of wgrad_tc.cu)."""
    ntiles = (ldb + min(256, ldb) - 1) // min(256, ldb)
    kt = (P + 63) // 64
    splits = min(max(1, sms // (4 * ntiles)), kt)
    per = (kt + splits - 1) // splits
    return (kt + per - 1) // per, per


def wgrad_tau(P: int, ldb: int, sms: int = 148) -> float:
    """Gate of one wgrad_tc call: a CTA accumulates 4 K = 16 instructions per 64-pixel tile of its slice in TMEM (plus <= 4
    roundings inside one), then every slice is added to out with an fp32 atomic: at most 4 * per + 4 + slices + 1
    roundings of 2^-23 each (in any order of the atomics)."""
    slices, per = wgrad_split(P, ldb, sms)
    return (4 * per + 4 + slices + 1) * U23


def wgrad_ref(A, B, out0, n_valid: int, drop_slice: Optional[int] = None, sms: int = 148) -> tuple:
    """(ref, scale) of out[:, :n_valid] after out0 += A^T B: float64, and |out0| + |A|^T |B|.  drop_slice plants the
    defect of a split-K slice that never adds its part (its pixels left out of the sum)."""
    _, per = wgrad_split(A.shape[0], B.shape[1], sms)
    A, B = A.double(), B.double()[:, :n_valid]
    if drop_slice is not None:
        keep = torch.ones(A.shape[0], dtype=torch.bool, device=A.device)
        keep[drop_slice * per * 64:(drop_slice + 1) * per * 64] = False
        A, B = A[keep], B[keep]
    o = out0.double()[:, :n_valid]
    return o + A.T @ B, o.abs() + A.abs().T @ B.abs()


# ------------------------------------------------------------------ operands
def melspec_config(K: int = 2):
    """The level shapes of the melspec model (48x32 C=4, 24x16 C=8, 12x8 C=16) at n_filters = 512."""
    from audiosourcesep_b200.config import GlowConfig
    return GlowConfig(H=96, W=64, C=1, L=3, K=K, n_filters=HID, minval=0.0, maxval=1.0)


def near_kink_params(cfg, seed: int) -> dict:
    """Perturbed Glow parameters with the hidden biases and BatchNorm offsets near zero, so that a large share of the
    ReLUs sit close to their kink (mask bits and rounding brackets are exercised where they are hardest)."""
    from audiosourcesep_b200.weights import init_glow_params
    p = init_glow_params(cfg, seed=seed, mode="perturbed")
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    for name in list(p):
        if name.endswith(("nn/conv1/bias", "nn/conv2/bias", "bn1/beta", "bn2/beta", "bn1/moving_mean", "bn2/moving_mean")):
            p[name] = rng.normal(0.0, 1e-3, p[name].shape).astype(np.float32)
    return p


def random_masks(M: int, seed: int, device=None) -> tuple:
    """Two int32 mask arrays [M, 16] with uniformly random bits (every bit pattern and word position)."""
    gen = torch.Generator().manual_seed(seed)
    w = torch.randint(-2 ** 31, 2 ** 31, (2, M, HID // 32), generator=gen, dtype=torch.int64).to(torch.int32)
    return w[0].to(device), w[1].to(device)
