"""Float64 restatement of the tensor-core convolutions of the score networks, and the gates that hold each launch to it.

  * ``k_conv_tc`` / ``k_conv_tc_sw`` (csrc/conv_tc.cu): Keras ``Conv2D(padding='same')``, stride 1, dilated, NHWC x HWIO,
    plus bias and up to two residual tensors -> ``conv_same``;
  * the data gradient (the same kernel on the transposed, flipped tile image) -> ``conv_data_grad``, the true adjoint;
  * ``k_conv_wgrad_tc`` (csrc/conv_wgrad_tc.cu) -> ``conv_wgrad``;
  * the bf16 tile images of ``conv_tc_prepare`` / ``k_build_conv_image`` -> ``tile_image``.

Everything is torch float64 and runs on the device of its inputs (CPU here, the GPU in the per-launch tests: a different
implementation from the kernels under test).  The tests feed the kernels exactly representable bf16 operands, so the
reference is exact up to float64 rounding and the only expected difference is the kernels' fp32 accumulation.

Gates: an element is accepted when |got - ref| <= tau * A with A the sum of the magnitudes of every term of that element
(``conv_same_abs`` etc. plus |bias| + |add| + |add2|).  Scaling by A instead of |ref| keeps the gate meaningful where
the terms cancel, and makes it a bound on the accumulation itself: a sum of n fp32 additions is off by at most about
n * 2^-24 * A.  tests/test_oracle_conv.py checks that each gate rejects the defects a kernel is likely to have (a
dropped 16-wide K step, a wrong border tap, swapped channels, a missing split-K slice, a missing split-bf16 pass).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

U32 = 2.0 ** -24        # unit roundoff of fp32

# bf16 x bf16 products accumulated in fp32 (TMEM): |got - ref| <= TAU_FWD * A per output element, for the forward and
# the data-gradient launches.  Calibrated on a B200 (1000 W power limit) over the whole per-launch matrix of
# tests/test_gpu_conv_tc.py: worst observed ratio 5.8e-7 (k_conv_tc), 5.1e-7 (k_conv_tc_sw), 5.5e-7 (data gradient);
# the gate is 13x that and 32x under 2^-12.
TAU_FWD = 2.0 ** -17
# the weight gradient (fp32 TMEM accumulation over a pixel slice + fp32 atomics over the split-K slices): worst observed
# ratio on the same B200 1.1e-7; the gate is 17x that.
TAU_WGRAD = 2.0 ** -19
# split-bf16 (three passes hi.hi + lo.hi + hi.lo of the unrounded fp32 operands): with x = hi + lo + r, |lo| <= 2^-8 |x|,
# |r| <= 2^-16 |x| (bf16 keeps 8 significant bits), every product is off by at most |lo_x lo_w| + |r_x w| + |x r_w| <=
# 3 * 2^-16 |x w|; one 2^-16 more covers the fp32 accumulation of the three passes.  (Worst observed on the B200:
# 2.2e-6, forward and data gradient.)
TAU_X3 = 4.0 * 2.0 ** -16
# instance-norm statistics: the epilogue sums `out` in fp32 inside a tile (the plain kernel: 8 pixels per lane, two
# shuffles, four warps -- at most 13 roundings on any term; the swapped kernel: 256 pixels per thread) and adds the tile
# sums in float64, so each (image, channel) sum is off by at most depth * 2^-24 * sum |term|.
STATS_DEPTH_PLAIN = 16
STATS_DEPTH_SWAPPED = 256


# ------------------------------------------------------------------ bf16
def bf16_rn(a) -> torch.Tensor:
    """fp32 -> bf16 round-to-nearest-even (``__float2bfloat16``), returned as the fp32 value of the bf16 number.
    Overflow rounds to +-inf, subnormals are kept, NaN becomes the quiet NaN 0x7FC0."""
    a = torch.as_tensor(a, dtype=torch.float32)
    u = a.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    r = torch.where(torch.isnan(a), torch.full_like(r, 0x7FC0), r)
    bits = r << 16
    bits = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32)
    return bits.view(torch.float32).reshape(a.shape)


def split_bf16(a) -> tuple:
    """(hi, lo) of the split-bf16 mode: hi = bf16(a), lo = bf16(a - hi) (the fp32 difference is exact)."""
    a = torch.as_tensor(a, dtype=torch.float32)
    hi = bf16_rn(a)
    return hi, bf16_rn(a - hi)


# ------------------------------------------------------------------ convolutions (NHWC x HWIO, float64)
def _f64(t, device=None) -> torch.Tensor:
    t = torch.as_tensor(t)
    return t.to(device=device if device is not None else t.device, dtype=torch.float64)


def _taps(ksize: int, dil: int, H: int, W: int):
    """(ty, tx, row slice, column slice) of every tap into the input padded by dil * (ksize // 2) on each side."""
    for ty in range(ksize):
        for tx in range(ksize):
            yield ty, tx, slice(ty * dil, ty * dil + H), slice(tx * dil, tx * dil + W)


def _pad(x: torch.Tensor, p: int) -> torch.Tensor:
    return F.pad(x, (0, 0, p, p, p, p)) if p else x


def conv_same(x, k, dil: int = 1) -> torch.Tensor:
    """Keras Conv2D(padding='same', dilation_rate=dil), stride 1: x [N,H,W,Cin], k [ks,ks,Cin,Cout] -> [N,H,W,Cout]."""
    x = _f64(x)
    k = _f64(k, x.device)
    N, H, W, _ = x.shape
    ks = k.shape[0]
    xp = _pad(x, dil * (ks // 2))
    out = torch.zeros((N, H, W, k.shape[3]), dtype=torch.float64, device=x.device)
    for ty, tx, rs, cs in _taps(ks, dil, H, W):
        out += xp[:, rs, cs, :] @ k[ty, tx]
    return out


def conv_same_abs(x, k, dil: int = 1) -> torch.Tensor:
    """A = sum over taps and input channels of |x * w| for every output element (the scale of the forward gates)."""
    return conv_same(_f64(x).abs(), _f64(k).abs(), dil)


def conv_data_grad(g, k, dil: int = 1) -> torch.Tensor:
    """Adjoint of ``conv_same`` in x: <conv_same(x, k), g> = <x, conv_data_grad(g, k)>; g [N,H,W,Cout] -> [N,H,W,Cin].
    Written as the scatter of every output gradient back to the inputs it read, not as a convolution."""
    g = _f64(g)
    k = _f64(k, g.device)
    N, H, W, _ = g.shape
    ks = k.shape[0]
    p = dil * (ks // 2)
    dxp = torch.zeros((N, H + 2 * p, W + 2 * p, k.shape[2]), dtype=torch.float64, device=g.device)
    for ty, tx, rs, cs in _taps(ks, dil, H, W):
        dxp[:, rs, cs, :] += g @ k[ty, tx].T
    return dxp[:, p:p + H, p:p + W, :]


def conv_data_grad_abs(g, k, dil: int = 1) -> torch.Tensor:
    return conv_data_grad(_f64(g).abs(), _f64(k).abs(), dil)


def conv_wgrad(x, g, ksize: int, dil: int = 1) -> torch.Tensor:
    """Weight gradient of ``conv_same``: dk[ty,tx,ci,co] = sum_p x[p + dil*(ty-h, tx-h)][ci] * g[p][co], h = ksize // 2
    (taps outside the image contribute nothing); x [N,H,W,Cin], g [N,H,W,Cout] -> [ks,ks,Cin,Cout]."""
    x = _f64(x)
    g = _f64(g, x.device)
    N, H, W, Cin = x.shape
    Cout = g.shape[3]
    xp = _pad(x, dil * (ksize // 2))
    g2 = g.reshape(-1, Cout)
    dk = torch.zeros((ksize, ksize, Cin, Cout), dtype=torch.float64, device=x.device)
    for ty, tx, rs, cs in _taps(ksize, dil, H, W):
        dk[ty, tx] = xp[:, rs, cs, :].reshape(-1, Cin).T @ g2
    return dk


def conv_wgrad_abs(x, g, ksize: int, dil: int = 1) -> torch.Tensor:
    return conv_wgrad(_f64(x).abs(), _f64(g).abs(), ksize, dil)


def transpose_kernel(k) -> torch.Tensor:
    """The kernel of the data gradient as an ordinary HWIO kernel: K'[tap'][co][ci] = K[taps-1-tap'][ci][co]."""
    k = torch.as_tensor(k)
    return torch.flip(k, dims=(0, 1)).transpose(2, 3).contiguous()


# ------------------------------------------------------------------ tile images
def swizzle_index(rows: int) -> np.ndarray:
    """Offset of element (r, c) of one [rows x 64] SWIZZLE_128B block: r*64 + (((c>>3) ^ (r&7))<<3) + (c&7)."""
    r = np.arange(rows)[:, None]
    c = np.arange(64)[None, :]
    return r * 64 + (((c >> 3) ^ (r & 7)) << 3) + (c & 7)


def tile_image(kernel, transposed: bool = False, lo: bool = False) -> torch.Tensor:
    """The bf16 tile image of an fp32 HWIO kernel (``conv_tc_prepare`` / ``k_build_conv_image``), flat, on the CPU:
    for every (tap, 64-channel panel of the contraction dimension) one [rows x 64] block, rows = the output channels of
    the image.  ``transposed``: the image of the data gradient (``transpose_kernel``); ``lo``: bf16(v - bf16(v))."""
    k = torch.as_tensor(kernel, dtype=torch.float32).cpu()
    if transposed:
        k = transpose_kernel(k)
    ks, _, ci, co = k.shape
    if ci % 64:
        raise ValueError(f"the contraction extent {ci} is not a multiple of 64")
    hi, low = split_bf16(k)
    v = (low if lo else hi).reshape(ks * ks, ci // 64, 64, co)           # [tap, panel, c, r]
    blocks = v.permute(0, 1, 3, 2).reshape(ks * ks * (ci // 64), co * 64)  # [tap*panel][r*64 + c], unswizzled
    img = torch.empty_like(blocks)
    img[:, torch.as_tensor(swizzle_index(co).reshape(-1))] = blocks
    return img.reshape(-1).to(torch.bfloat16)


def untile_image(img, ksize: int, cin: int, cout: int) -> torch.Tensor:
    """Inverse of ``tile_image`` for an image whose contraction extent is ``cin`` and row count ``cout`` -> fp32 HWIO."""
    b = torch.as_tensor(img).float().cpu().reshape(ksize * ksize * (cin // 64), cout, 8, 8)   # [block, r, chunk slot, 8]
    r = torch.arange(cout)
    out = torch.empty_like(b)
    for c in range(8):
        out[:, :, c, :] = b[:, r, torch.as_tensor(c) ^ (r & 7), :]
    return out.reshape(ksize * ksize, cin // 64, cout, 64).permute(0, 1, 3, 2).reshape(ksize, ksize, cin, cout)


# ------------------------------------------------------------------ gates
def gate_ratio(got, ref, scale) -> float:
    """max |got - ref| / scale over all elements (scale > 0): what a tau gate compares with tau."""
    got, ref, scale = _f64(got), _f64(ref), _f64(scale)
    return float(((got - ref.to(got.device)).abs() / scale.to(got.device).clamp_min(1e-300)).max())


def stats_ref(out) -> torch.Tensor:
    """float64 per-(image, channel) sum and sum of squares of an NHWC tensor -> [N, C, 2]."""
    o = _f64(out)
    return torch.stack([o.sum(dim=(1, 2)), (o * o).sum(dim=(1, 2))], dim=-1)


def stats_scale(out) -> torch.Tensor:
    """The magnitudes the statistics gate scales with: sum |o| and sum o^2 per (image, channel) -> [N, C, 2]."""
    o = _f64(out)
    return torch.stack([o.abs().sum(dim=(1, 2)), (o * o).sum(dim=(1, 2))], dim=-1)


def wgrad_splits(sms: int, ksize: int, cin: int, cout: int, k_tiles: int) -> tuple:
    """(slices, pixel tiles per slice) of the split-K partition of ``conv_wgrad_tc`` (conv_wgrad_tc.cu host side):
    k_tiles tiles of 64 pixels over about 2 CTAs per SM."""
    n_mma = cout if cout <= 256 else cout // 2
    mtiles, ntiles = (cin + 127) // 128, cout // n_mma
    splits = max(1, (2 * sms) // (ksize * ksize * mtiles * ntiles))
    splits = min(splits, k_tiles)
    per = (k_tiles + splits - 1) // splits
    return (k_tiles + per - 1) // per, per


# ------------------------------------------------------------------ operands
def operands(seed: int, N: int, H: int, W: int, cin: int, cout: int, ksize: int, device=None) -> dict:
    """Seeded fp32 operands of one convolution: x ~ N(0, 1) [N,H,W,cin] (normalised activations), the HWIO kernel ~
    N(0, 1/(ksize^2 cin)) (He-like), bias, two residual tensors [N,H,W,cout] and an output gradient g ~ N(0, 1)."""
    gen = torch.Generator().manual_seed(seed)
    t = lambda *s, scale=1.0: (torch.randn(*s, generator=gen) * scale).to(device=device, dtype=torch.float32)  # noqa: E731
    return {"x": t(N, H, W, cin), "k": t(ksize, ksize, cin, cout, scale=(ksize * ksize * cin) ** -0.5),
            "bias": t(cout, scale=0.5), "add": t(N, H, W, cout), "add2": t(N, H, W, cout), "g": t(N, H, W, cout)}
