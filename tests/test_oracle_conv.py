"""CPU checks of the float64 convolution oracle (oracle/conv_oracle.py) and of the gates tests/test_gpu_conv_tc.py holds
the tensor-core convolutions to: each gate accepts what fp32 accumulation can produce and rejects the defects such a
kernel is likely to have."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import conv_oracle as co


def _torch_conv(x, k, dil):
    """torch's float64 conv2d in NHWC / HWIO with Keras 'same' padding (odd kernels, stride 1)."""
    p = dil * (k.shape[0] // 2)
    y = F.conv2d(x.permute(0, 3, 1, 2), k.permute(3, 2, 0, 1), padding=p, dilation=dil)
    return y.permute(0, 2, 3, 1)


@pytest.mark.parametrize("ksize,dil", [(1, 1), (3, 1), (3, 2), (3, 4)])
def test_conv_same_matches_torch_conv2d(ksize, dil):
    gen = torch.Generator().manual_seed(ksize * 10 + dil)
    x = torch.randn(2, 12, 8, 5, generator=gen, dtype=torch.float64)       # 12 x 8 with dilation 4: taps leave the image
    k = torch.randn(ksize, ksize, 5, 7, generator=gen, dtype=torch.float64)
    assert torch.allclose(co.conv_same(x, k, dil), _torch_conv(x, k, dil), rtol=1e-13, atol=1e-13)
    a = co.conv_same_abs(x, k, dil)
    assert torch.allclose(a, _torch_conv(x.abs(), k.abs(), dil), rtol=1e-13, atol=1e-13)
    assert bool((a >= co.conv_same(x, k, dil).abs() - 1e-12).all())


@pytest.mark.parametrize("ksize,dil", [(1, 1), (3, 1), (3, 2), (3, 4)])
def test_data_grad_is_the_adjoint_and_the_flipped_transposed_convolution(ksize, dil):
    gen = torch.Generator().manual_seed(7 + dil)
    x = torch.randn(2, 8, 16, 6, generator=gen, dtype=torch.float64)
    g = torch.randn(2, 8, 16, 4, generator=gen, dtype=torch.float64)
    k = torch.randn(ksize, ksize, 6, 4, generator=gen, dtype=torch.float64)
    dx = co.conv_data_grad(g, k, dil)
    lhs = float((co.conv_same(x, k, dil) * g).sum())
    rhs = float((x * dx).sum())
    assert abs(lhs - rhs) <= 1e-12 * (abs(lhs) + 1.0)
    # what the training step runs: the forward convolution with the transposed, flipped kernel
    assert torch.allclose(co.conv_same(g, co.transpose_kernel(k), dil), dx, rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize("ksize,dil", [(1, 1), (3, 1), (3, 2), (3, 4)])
def test_conv_wgrad_matches_autograd(ksize, dil):
    gen = torch.Generator().manual_seed(3 + dil)
    x = torch.randn(2, 8, 8, 5, generator=gen, dtype=torch.float64)
    g = torch.randn(2, 8, 8, 3, generator=gen, dtype=torch.float64)
    k = torch.randn(ksize, ksize, 5, 3, generator=gen, dtype=torch.float64, requires_grad=True)
    (_torch_conv(x, k, dil) * g).sum().backward()
    assert torch.allclose(co.conv_wgrad(x, g, ksize, dil), k.grad, rtol=1e-13, atol=1e-13)


def test_bf16_rn_matches_torch_cast():
    f32 = np.float32
    bits = np.array([0x3F808000, 0x3F818000, 0x3F80C000, 0x3F807FFF,   # ties to even (down, up), above and below a tie
                     0xBF808000, 0xBF818000,                              # negative ties
                     0x00000001, 0x00008000, 0x00018000, 0x007FFFFF,      # subnormals, incl. ties and the largest
                     0x80008000, 0x7F7FFFFF, 0x7F7F8000, 0xFF7FFFFF,      # overflow to +-inf, a tie at the top binade
                     0x7F800000, 0xFF800000, 0x00000000, 0x80000000], dtype=np.uint32)
    rng = np.random.default_rng(0)
    vals = np.concatenate([bits.view(f32), rng.standard_normal(4096).astype(f32) * f32(1e3),
                           rng.integers(0, 2 ** 32, 4096, dtype=np.uint64).astype(np.uint32).view(f32)])
    vals = vals[~np.isnan(vals)]
    t = torch.from_numpy(vals)
    ours = co.bf16_rn(t)
    want = t.to(torch.bfloat16).float()
    assert torch.equal(ours.view(torch.int32), want.view(torch.int32))
    assert torch.isnan(co.bf16_rn(torch.tensor([float("nan")]))).all()
    assert float(co.bf16_rn(torch.tensor([1.0 + 2.0 ** -8]))) == 1.0                  # tie -> even
    assert float(co.bf16_rn(torch.tensor([1.0 + 3 * 2.0 ** -8]))) == 1.0 + 2.0 ** -6  # tie -> even (up)
    normal = t[len(bits):len(bits) + 4096]
    hi, lo = co.split_bf16(normal)
    assert torch.equal(lo, co.bf16_rn(normal - hi)) and torch.equal(hi + lo, normal.to(torch.bfloat16).float() + lo)


@pytest.mark.parametrize("transposed,lo", [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("ksize,cin,cout", [(3, 64, 128), (1, 192, 384), (3, 128, 192)])
def test_tile_image_unswizzles_to_the_kernel(ksize, cin, cout, transposed, lo):
    k = co.operands(1, 1, 2, 2, cin, cout, ksize)["k"]
    img = co.tile_image(k, bool(transposed), bool(lo))
    assert img.dtype == torch.bfloat16 and img.numel() == k.numel()
    kk = co.transpose_kernel(k) if transposed else k
    hi, low = co.split_bf16(kk)
    ci, ro = (cout, cin) if transposed else (cin, cout)
    assert torch.equal(co.untile_image(img, ksize, ci, ro), low if lo else hi)
    # element (r, c) of block 0 sits at r*64 + (((c>>3) ^ (r&7))<<3) + (c&7): spot-check against the kernel directly
    for r, c in [(0, 0), (1, 0), (7, 9), (9, 63), (ro - 1, 17)]:
        off = r * 64 + (((c >> 3) ^ (r & 7)) << 3) + (c & 7)
        assert float(img[off]) == float((low if lo else hi)[0, 0, c, r])


# ------------------------------------------------------------------ gate sensitivity
def _bf(t):
    return co.bf16_rn(t).double()


def _fwd(seed, N, H, W, cin, cout, ksize, dil):
    op = co.operands(seed, N, H, W, cin, cout, ksize)
    x, k = _bf(op["x"]), _bf(op["k"])
    return x, k, co.conv_same(x, k, dil), co.conv_same_abs(x, k, dil)


def _defects(x, k, ref, dil):
    """The forward defects a gate must reject: (name, perturbed reference)."""
    ks, cin = k.shape[0], k.shape[2]
    N, H, W, _ = x.shape
    out = []
    kd = torch.zeros_like(k)                                  # the last 16-wide K step (highest tap, last 16 channels)
    kd[ks - 1, ks - 1, cin - 16:, :] = k[ks - 1, ks - 1, cin - 16:, :]
    out.append(("drop_k16", ref - co.conv_same(x, kd, dil)))
    bad = ref.clone()                                         # tap (dy = +dil, dx = -dil) of the top-right pixel
    ty, tx = (ks - 1, 0) if ks == 3 else (0, 0)
    bad[0, 0, W - 1, :] -= x[0, ty * dil - dil * (ks // 2), W - 1 + tx * dil - dil * (ks // 2), :] @ k[ty, tx]
    out.append(("border_tap", bad))
    bad = ref.clone()                                         # channels 3 and 70 of one interior pixel swapped
    bad[N - 1, H // 2, W // 2, [3, 70]] = ref[N - 1, H // 2, W // 2, [70, 3]]
    out.append(("swap_channels", bad))
    return out


@pytest.mark.parametrize("dil", [1, 4])
def test_forward_gate_rejects_kernel_defects_at_the_largest_k(dil):
    """K = taps * Cin = 3456 (Cin = 384, the widest NCSN layer): every defect moves some element by more than
    TAU_FWD * A, while an fp32 evaluation of the same products stays inside the gate."""
    x, k, ref, A = _fwd(0, 1, 16, 32, 384, 128, 3, dil)
    f32 = _torch_conv(x.float(), k.float(), dil)                # fp32 accumulation of the same products
    assert co.gate_ratio(f32, ref, A) <= co.TAU_FWD
    for name, bad in _defects(x, k, ref, dil):
        assert co.gate_ratio(bad, ref, A) > 4 * co.TAU_FWD, name


def test_forward_gate_rejects_the_out_bf16_rounding():
    """out_bf16 is compared bitwise; the fp32 output must not pass if it were only bf16-accurate."""
    x, k, ref, A = _fwd(1, 1, 8, 32, 192, 128, 3, 2)
    assert co.gate_ratio(co.bf16_rn(ref.float()), ref, A) > 4 * co.TAU_FWD


def test_data_gradient_gate_rejects_defects():
    """The data gradient runs the forward kernel on the transposed image: Cin' = Cout = 384, Cout' = Cin = 192."""
    op = co.operands(2, 1, 16, 32, 192, 384, 3)
    g, k = _bf(op["g"]), _bf(op["k"])
    kt = co.transpose_kernel(k)
    ref, A = co.conv_data_grad(g, k, 2), co.conv_data_grad_abs(g, k, 2)
    for name, bad in _defects(g, kt, ref, 2):
        assert co.gate_ratio(bad, ref, A) > 4 * co.TAU_FWD, name


def _x3(seed, N, H, W, cin, cout, dil):
    op = co.operands(seed, N, H, W, cin, cout, 3)
    x, k = op["x"], op["k"]
    (xh, xl), (kh, kl) = co.split_bf16(x), co.split_bf16(k)
    ref, A = co.conv_same(x, k, dil), co.conv_same_abs(x, k, dil)
    parts = [co.conv_same(xh, kl, dil), co.conv_same(xl, kh, dil), co.conv_same(xh, kh, dil)]
    return x, k, ref, A, parts


def test_split_bf16_gate_holds_the_three_products_and_rejects_a_missing_pass():
    x, k, ref, A, parts = _x3(3, 1, 16, 32, 192, 192, 2)
    assert co.gate_ratio(sum(parts), ref, A) <= co.TAU_X3 / 2        # the operand error alone, in float64
    for i, name in enumerate(["no_hi_lo", "no_lo_hi"]):
        assert co.gate_ratio(sum(p for j, p in enumerate(parts) if j != i), ref, A) > 2 * co.TAU_X3, name
    for name, bad in _defects(x.double(), k.double(), ref, 2):
        assert co.gate_ratio(bad, ref, A) > 4 * co.TAU_X3, name


def test_split_bf16_gate_rejects_defects_at_the_largest_k():
    x, k, ref, A, parts = _x3(4, 1, 8, 32, 384, 128, 1)
    assert co.gate_ratio(sum(parts), ref, A) <= co.TAU_X3 / 2
    for name, bad in _defects(x.double(), k.double(), ref, 1):
        assert co.gate_ratio(bad, ref, A) > 4 * co.TAU_X3, name


# the largest weight-gradient problem of tests/test_gpu_conv_tc.py: 30 x 96 x 64 pixels
WGRAD_LARGEST = (30, 96, 64)


def test_wgrad_gate_rejects_defects_at_the_largest_pixel_count():
    N, H, W = WGRAD_LARGEST
    op = co.operands(5, N, H, W, 64, 128, 3)
    x, g = _bf(op["x"]), _bf(op["g"])
    ref, A = co.conv_wgrad(x, g, 3, 4), co.conv_wgrad_abs(x, g, 3, 4)
    xf, gf = x.reshape(-1, 64), g.reshape(-1, 128)
    f32 = xf.float().T @ gf.float()                           # fp32 accumulation of the centre tap's products
    assert co.gate_ratio(f32, ref[1, 1], A[1, 1]) <= co.TAU_WGRAD
    defects = {
        # one 16-pixel K step of the centre tap missing (the pixel range is the reduction)
        "drop_k16": ref[1, 1] - xf[4096:4112].T @ gf[4096:4112],
        # the last 64-pixel tile (the ragged end of the last split-K slice) missing from the centre tap
        "drop_last_tile": ref[1, 1] - xf[-64:].T @ gf[-64:],
        # one border pixel's contribution to one off-centre tap missing (pixel (0, 0, W-1) reads x at (4, W-5))
        "border_tap": ref[2, 0] - torch.outer(x[0, 4, W - 5], g[0, 0, W - 1]),
    }
    for name, bad in defects.items():
        tap = (1, 1) if name != "border_tap" else (2, 0)
        assert co.gate_ratio(bad, ref[tap], A[tap]) > 4 * co.TAU_WGRAD, name
    bad = ref.clone()
    bad[0, 0, 5, [3, 70]] = ref[0, 0, 5, [70, 3]]
    assert co.gate_ratio(bad, ref, A) > 4 * co.TAU_WGRAD


def test_stats_gate_rejects_a_wrong_column_group_and_a_missing_tile():
    x, k, ref, _ = _fwd(6, 2, 8, 32, 64, 384, 1, 1)
    out = ref.float()
    st, scale = co.stats_ref(out), co.stats_scale(out)
    tol = co.STATS_DEPTH_SWAPPED * co.U32                     # the looser of the two kernels' gates
    bad = st.clone()
    bad[:, 192:, :] = st[:, :192, :]                          # the second column group (Cout = 384) gets the first's sums
    assert co.gate_ratio(bad, st, scale) > 4 * tol
    o2 = out.clone()
    o2[1, :4] = 0                                             # one 128-pixel tile of image 1 missing from the sums
    assert co.gate_ratio(co.stats_ref(o2), st, scale) > 4 * tol


def test_wgrad_split_partition_matches_the_host_logic():
    # 148 SMs: Cin = 192 (two M tiles), Cout = 384 (two N tiles), 3 x 3 -> 296 // 36 = 8 slices
    assert co.wgrad_splits(148, 3, 192, 384, 100) == (8, 13)
    assert co.wgrad_splits(148, 1, 64, 128, 3) == (3, 1)
    assert co.wgrad_splits(148, 3, 384, 384, 5) == (5, 1)
