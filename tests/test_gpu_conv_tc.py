"""The tensor-core convolutions of the score networks one launch at a time against the float64 oracle
(oracle/conv_oracle.py): k_conv_tc / k_conv_tc_sw (forward and, on the transposed image, data gradient),
k_conv_wgrad_tc (weight gradient) and the two tile-image builders.

Operands are exact bf16 values, so the reference is exact and the only expected difference is fp32 accumulation: every
element must satisfy |got - ref| <= tau * A with A the sum of the magnitudes of its terms.  The gates and the defects
they reject are checked on the CPU in tests/test_oracle_conv.py.  Run with -s to see the worst ratio per kernel."""
import itertools

import pytest
import torch

from audiosourcesep_b200 import _lib, ops
from oracle import conv_oracle as co

pytestmark = pytest.mark.gpu

ERR_BAD_DTYPE, ERR_BAD_SHAPE, ERR_UNSUPPORTED = -3, -2, -9
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    for name, r in sorted(WORST.items()):
        print(f"\n{name}: worst |got - ref| / A = {r:.3e}")


def _record(name, r):
    WORST[name] = max(WORST.get(name, 0.0), r)
    return r


def _dev():
    return torch.device("cuda", _lib.init())


def _ops(seed, N, H, W, cin, cout, ksize):
    return co.operands(seed, N, H, W, cin, cout, ksize, device=_dev())


def _bf(t):
    return t.to(torch.bfloat16)


def _bits(t):
    return t.contiguous().view(torch.int16)


def _swapped(cout, H, W, mode):
    return mode != "plain" and cout == 128 and 256 % W == 0 and H % (256 // W) == 0


def _mode(monkeypatch, mode):
    # conv_tc_forward reads ASEP_CONV_NO_SWAP on every call
    if mode == "plain":
        monkeypatch.setenv("ASEP_CONV_NO_SWAP", "1")
    else:
        monkeypatch.delenv("ASEP_CONV_NO_SWAP", raising=False)


def _check_stats(st, out, swapped, name):
    depth = co.STATS_DEPTH_SWAPPED if swapped else co.STATS_DEPTH_PLAIN
    r = _record(name, co.gate_ratio(st, co.stats_ref(out), co.stats_scale(out)))
    assert r <= depth * co.U32, f"instance-norm statistics off by {r:.3e} of sum |o| (gate {depth} * 2^-24)"


# ------------------------------------------------------------------ forward
CINS, COUTS = (64, 128, 192, 256, 384), (128, 192, 256, 384)


def _fwd_cases():
    c = []   # (cin, cout, ksize, dil, H, W, N, mode); mode: "sw" / "plain" for Cout = 128, "-" otherwise
    add = lambda *a: c.extend([a + ("sw",), a + ("plain",)] if a[1] == 128 else [a + ("-",)])  # noqa: E731
    for cin, cout in itertools.product(CINS, COUTS):              # every (Cin, Cout) pair, 3 x 3
        add(cin, cout, 3, 1, 8, 64, 2)
    for cout, cin in zip(COUTS, (192, 128, 384, 192)):            # 1 x 1 and dilation 2 / 4 at every Cout
        add(cin, cout, 1, 1, 16, 32, 2)
        add(cin, cout, 3, 2, 16, 32, 2)
        add(cin, cout, 3, 4, 16, 32, 2)                           # W = 32: 4-row tiles, dy = +-4 boxes wholly outside
    add(384, 384, 3, 4, 48, 32, 2)                                # v1 half resolution
    add(256, 256, 3, 4, 48, 32, 2)                                # v2 half resolution
    add(128, 128, 3, 2, 64, 8, 2)                                 # the supported narrow / wide widths
    add(192, 384, 3, 4, 64, 8, 1)
    add(256, 256, 3, 4, 32, 16, 2)
    add(128, 192, 3, 1, 16, 16, 1)
    add(128, 128, 3, 1, 4, 128, 2)
    add(384, 384, 3, 4, 8, 128, 1)
    add(64, 256, 1, 1, 4, 128, 1)
    c.append((128, 128, 3, 1, 6, 64, 2, "fallback"))             # H % (256 / W) != 0: the plain form by itself
    c.append((256, 128, 3, 2, 12, 32, 1, "fallback"))
    add(192, 384, 3, 2, 48, 32, 1)                                # N = 1: fewer units than SMs
    add(128, 128, 3, 1, 96, 64, 30)                               # N = 30: >= 3 units per CTA, TMEM phases wrap
    add(192, 192, 3, 1, 96, 64, 30)
    add(192, 384, 3, 2, 96, 64, 30)
    return c


def _fid(c):
    cin, cout, ks, dil, H, W, N, mode = c
    return f"ci{cin}-co{cout}-k{ks}d{dil}-n{N}x{H}x{W}" + ("" if mode == "-" else f"-{mode}")


@pytest.mark.parametrize("case", _fwd_cases(), ids=_fid)
def test_forward_matches_float64(case, monkeypatch):
    """bias + add + add2 + statistics + bf16 copy all on: out within TAU_FWD * A, out_bf16 = bf16_rn(out) bitwise,
    statistics within the fp32 tile-sum bound, a second identical call bitwise equal."""
    cin, cout, ks, dil, H, W, N, mode = case
    _mode(monkeypatch, mode)
    op = _ops(cin + cout + ks + dil + H + N, N, H, W, cin, cout, ks)
    x, kb = _bf(op["x"]), co.bf16_rn(op["k"])
    img = ops.conv_tc_image(op["k"])
    args = dict(bias=op["bias"], add=op["add"], add2=op["add2"], stats=True, out_bf16=True)
    out, st, ob = ops.conv_tc_forward(img, x, ks, cin, cout, dil, **args)
    extra = op["bias"].double() + op["add"].double() + op["add2"].double()
    ref = co.conv_same(x, kb, dil) + extra
    A = co.conv_same_abs(x, kb, dil) + op["bias"].double().abs() + op["add"].double().abs() + op["add2"].double().abs()
    swapped = _swapped(cout, H, W, mode)
    kern = "k_conv_tc_sw" if swapped else "k_conv_tc"
    r = _record(f"forward {kern}", co.gate_ratio(out, ref, A))
    assert r <= co.TAU_FWD, f"{kern}: max |got - ref| / A = {r:.3e} > {co.TAU_FWD:.3e}"
    assert torch.equal(_bits(ob), _bits(_bf(out))), "out_bf16 is not bf16_rn(out)"
    _check_stats(st, out, swapped, f"stats {kern}")
    out2, _, ob2 = ops.conv_tc_forward(img, x, ks, cin, cout, dil, **args)
    assert torch.equal(out2.view(torch.int32), out.view(torch.int32)) and torch.equal(_bits(ob2), _bits(ob))


EPILOGUES = [(b, a, a2, False) for b, a, a2 in itertools.product((0, 1), repeat=3)] + [(0, 1, 0, True), (1, 1, 1, True)]


@pytest.mark.parametrize("epi", EPILOGUES, ids=lambda e: f"bias{e[0]}-add{e[1]}-add2{e[2]}" + ("-alias" if e[3] else ""))
@pytest.mark.parametrize("geom", [(128, 128, "sw"), (128, 128, "plain"), (192, 384, "-")], ids=lambda g: f"co{g[1]}-{g[2]}")
def test_forward_epilogue_combinations(geom, epi, monkeypatch):
    """Every combination of bias / add / add2, and add aliasing out (the split-bf16 passes accumulate in place)."""
    cin, cout, mode = geom
    use_bias, use_add, use_add2, alias = epi
    _mode(monkeypatch, mode)
    N, H, W = 2, 16, 32
    op = _ops(17, N, H, W, cin, cout, 3)
    x, kb = _bf(op["x"]), co.bf16_rn(op["k"])
    img = ops.conv_tc_image(op["k"])
    bias = op["bias"] if use_bias else None
    add = op["add"] if use_add else None
    add2 = op["add2"] if use_add2 else None
    out = None
    if alias:
        out = op["add"].clone()
        add = out
    out, st, ob = ops.conv_tc_forward(img, x, 3, cin, cout, 2, bias=bias, add=add, add2=add2, out=out, stats=True,
                                      out_bf16=True)
    ref, A = co.conv_same(x, kb, 2), co.conv_same_abs(x, kb, 2)
    for used, t in ((use_bias, op["bias"]), (use_add, op["add"]), (use_add2, op["add2"])):
        if used:
            ref, A = ref + t.double(), A + t.double().abs()
    swapped = _swapped(cout, H, W, mode)
    r = _record("forward epilogues", co.gate_ratio(out, ref, A))
    assert r <= co.TAU_FWD, f"max |got - ref| / A = {r:.3e}"
    assert torch.equal(_bits(ob), _bits(_bf(out)))
    _check_stats(st, out, swapped, "stats epilogues")


X3_CASES = [(128, 128, 3, 2, 16, 32, 2, "sw"), (128, 128, 3, 2, 16, 32, 2, "plain"), (192, 192, 3, 1, 32, 64, 2, "-"),
            (384, 384, 3, 4, 48, 32, 2, "-"), (256, 256, 3, 2, 16, 32, 2, "-"), (192, 384, 1, 1, 16, 64, 2, "-"),
            (384, 192, 3, 2, 16, 32, 2, "-")]


@pytest.mark.parametrize("case", X3_CASES, ids=_fid)
def test_split_bf16_composition(case, monkeypatch):
    """The three launches of one ASEP_PREC_BF16X3 convolution (ncsn_model.cu, NcsnModel::conv): lo image x hi x with
    add / add2, then hi image x lo x accumulated in place, then hi x hi with bias and statistics -- against float64 of
    the unrounded fp32 operands."""
    cin, cout, ks, dil, H, W, N, mode = case
    _mode(monkeypatch, mode)
    op = _ops(cin * 3 + cout + dil, N, H, W, cin, cout, ks)
    xh, xl = (_bf(t) for t in co.split_bf16(op["x"]))
    hi, lo = ops.conv_tc_image(op["k"]), ops.conv_tc_image(op["k"], lo=True)
    out, _, _ = ops.conv_tc_forward(lo, xh, ks, cin, cout, dil, add=op["add"], add2=op["add2"])
    ops.conv_tc_forward(hi, xl, ks, cin, cout, dil, add=out, out=out)
    _, st, _ = ops.conv_tc_forward(hi, xh, ks, cin, cout, dil, bias=op["bias"], add=out, out=out, stats=True)
    ref = co.conv_same(op["x"], op["k"], dil) + op["bias"].double() + op["add"].double() + op["add2"].double()
    A = (co.conv_same_abs(op["x"], op["k"], dil) + op["bias"].double().abs() + op["add"].double().abs()
         + op["add2"].double().abs())
    r = _record("split-bf16 forward", co.gate_ratio(out, ref, A))
    assert r <= co.TAU_X3, f"max |got - ref| / A = {r:.3e} > {co.TAU_X3:.3e}"
    _check_stats(st, out, _swapped(cout, H, W, mode), "stats split-bf16")


# ------------------------------------------------------------------ data gradient
NET_PAIRS = [(192, 384, 1), (192, 192, 3), (192, 384, 3), (384, 192, 3), (384, 384, 3),      # v1, ngf = 192
             (128, 256, 1), (128, 128, 3), (128, 256, 3), (256, 128, 3), (256, 256, 3)]      # v2, ngf = 128
DGRAD_CASES = ([(ci, cout, ks, d, "bf16") for ci, cout, ks in NET_PAIRS for d in ((1, 2, 4) if ks == 3 else (1,))]
               + [(ci, cout, ks, 2 if ks == 3 else 1, "x3") for ci, cout, ks in NET_PAIRS])


@pytest.mark.parametrize("case", DGRAD_CASES, ids=lambda c: f"ci{c[0]}-co{c[1]}-k{c[2]}d{c[3]}-{c[4]}")
def test_data_gradient_matches_adjoint(case):
    """The device-built transposed image through the forward kernel (Cin' = Cout, Cout' = Cin) against the true
    adjoint; x3: the three launches of ncsn_train.cu (lo image x hi g, hi x lo g, hi x hi g) against the unrounded g."""
    cin, cout, ks, dil, prec = case
    N, H, W = 2, 16, 32
    op = _ops(cin + 2 * cout + dil, N, H, W, cin, cout, ks)
    t_hi = ops.conv_tc_image(op["k"], transposed=True)
    if prec == "bf16":
        g, kb = _bf(op["g"]), co.bf16_rn(op["k"])
        dx, _, _ = ops.conv_tc_forward(t_hi, g, ks, cout, cin, dil)
        ref, A, tau = co.conv_data_grad(g, kb, dil), co.conv_data_grad_abs(g, kb, dil), co.TAU_FWD
    else:
        t_lo = ops.conv_tc_image(op["k"], transposed=True, lo=True)
        gh, gl = (_bf(t) for t in co.split_bf16(op["g"]))
        dx, _, _ = ops.conv_tc_forward(t_lo, gh, ks, cout, cin, dil)
        ops.conv_tc_forward(t_hi, gl, ks, cout, cin, dil, add=dx, out=dx)
        ops.conv_tc_forward(t_hi, gh, ks, cout, cin, dil, add=dx, out=dx)
        ref, A, tau = co.conv_data_grad(op["g"], op["k"], dil), co.conv_data_grad_abs(op["g"], op["k"], dil), co.TAU_X3
    r = _record(f"data gradient {prec}", co.gate_ratio(dx, ref, A))
    assert r <= tau, f"max |got - ref| / A = {r:.3e} > {tau:.3e}"


# ------------------------------------------------------------------ weight gradient
# (cin, cout, ksize, dil, H, W, N, ragged): ragged = the pixel tiles do not divide evenly over the split-K slices
WGRAD_CASES = [(192, 384, 3, 1, 24, 32, 3, True),    # Cin = 192: half-empty second M tile; Cout = 384: n_mma = 192
               (192, 384, 3, 4, 24, 32, 3, True),
               (128, 128, 3, 2, 64, 8, 11, True),    # W = 8
               (256, 256, 3, 4, 32, 16, 5, True),    # W = 16
               (384, 384, 3, 2, 16, 64, 2, True),    # W = 64
               (64, 192, 3, 1, 16, 64, 5, True),
               (192, 384, 1, 1, 16, 64, 10, True),
               (128, 256, 1, 1, 16, 64, 2, False),
               (192, 192, 3, 2, 32, 32, 2, False),
               (256, 128, 3, 4, 48, 32, 2, False),
               (64, 128, 3, 4, 96, 64, 30, False)]   # the largest pixel count (test_oracle_conv.WGRAD_LARGEST)


@pytest.mark.parametrize("case", WGRAD_CASES, ids=lambda c: f"ci{c[0]}-co{c[1]}-k{c[2]}d{c[3]}-n{c[6]}x{c[4]}x{c[5]}")
def test_weight_gradient_accumulates_into_dk(case):
    cin, cout, ks, dil, H, W, N, ragged = case
    sms = torch.cuda.get_device_properties(_dev()).multi_processor_count
    slices, per = co.wgrad_splits(sms, ks, cin, cout, N * H * W // 64)
    assert ((N * H * W // 64) % per != 0) == ragged, f"split-K partition ({slices} x {per}) on {sms} SMs"
    op = _ops(cin + cout + 5 * dil + N, N, H, W, cin, cout, ks)
    x, g = _bf(op["x"]), _bf(op["g"])
    dk0 = torch.randn(ks, ks, cin, cout, generator=torch.Generator().manual_seed(9)).to(_dev())   # dk is accumulated into
    dk = ops.conv_wgrad_tc(x, g, dk0.clone(), ks, dil)
    ref = dk0.double() + co.conv_wgrad(x, g, ks, dil)
    A = dk0.double().abs() + co.conv_wgrad_abs(x, g, ks, dil)
    r = _record("weight gradient k_conv_wgrad_tc", co.gate_ratio(dk, ref, A))
    assert r <= co.TAU_WGRAD, f"max |got - ref| / A = {r:.3e} > {co.TAU_WGRAD:.3e}"


# ------------------------------------------------------------------ tile images
def _geometries():
    g = {(c[2], c[0], c[1]) for c in _fwd_cases()} | {(c[2], c[0], c[1]) for c in WGRAD_CASES}
    g |= {(ks, ci, cout) for ci, cout, ks in NET_PAIRS}
    return sorted(g)


@pytest.mark.parametrize("tl", [(0, 0), (1, 0), (0, 1), (1, 1)], ids=lambda t: f"t{t[0]}lo{t[1]}")
@pytest.mark.parametrize("geom", _geometries(), ids=lambda g: f"k{g[0]}-ci{g[1]}-co{g[2]}")
def test_tile_images_bitwise(geom, tl):
    """The device builder (every optimizer step) = the host builder (asep_ncsn_prepare) = tile_image, bit for bit."""
    ks, cin, cout = geom
    transposed, lo = tl
    k = _ops(ks * 1000 + cin + cout, 1, 1, 1, cin, cout, ks)["k"]
    k[0, 0, 0, 0] = 1.0 + 2.0 ** -8                      # a tie: rounds to even in both words
    dev = ops.conv_tc_image(k, transposed=bool(transposed), lo=bool(lo))
    assert torch.equal(_bits(dev).cpu(), _bits(co.tile_image(k.cpu(), bool(transposed), bool(lo))))
    if not transposed and not lo:
        assert torch.equal(_bits(ops.conv_tc_image(k.cpu(), on_device=False)), _bits(dev))


# ------------------------------------------------------------------ shapes the kernels do not take
def _expect_error(code, fn):
    n0 = _lib.launch_count()
    with pytest.raises(_lib.AsepError) as e:
        fn()
    assert e.value.code == code, str(e.value)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0, "a kernel was launched before the shape was rejected"


@pytest.mark.parametrize("shape", [(64, 320, 8, 64), (64, 128, 8, 48), (64, 256, 3, 64), (64, 128, 2, 32),
                                   (96, 128, 8, 64)], ids=lambda s: "ci{}-co{}-h{}-w{}".format(*s))
def test_forward_rejects_unsupported_shapes(shape):
    """Cout = 320, W = 48 (does not divide 128), H not a multiple of 128 / W, Cin not a multiple of 64."""
    cin, cout, H, W = shape
    dev = _dev()
    img = torch.zeros(9 * cin * cout, dtype=torch.bfloat16, device=dev)
    x = torch.zeros(1, H, W, cin, dtype=torch.bfloat16, device=dev)
    _expect_error(ERR_UNSUPPORTED, lambda: ops.conv_tc_forward(img, x, 3, cin, cout, 1))


@pytest.mark.parametrize("shape", [(64, 128, 2, 128), (64, 320, 8, 64), (64, 128, 8, 48), (96, 128, 8, 64)],
                         ids=lambda s: "ci{}-co{}-h{}-w{}".format(*s))
def test_weight_gradient_rejects_unsupported_shapes(shape):
    """W = 128 (the weight gradient tiles 64 pixels), Cout = 320, W = 48, Cin not a multiple of 64."""
    cin, cout, H, W = shape
    dev = _dev()
    x = torch.zeros(1, H, W, cin, dtype=torch.bfloat16, device=dev)
    g = torch.zeros(1, H, W, cout, dtype=torch.bfloat16, device=dev)
    dk = torch.zeros(3, 3, cin, cout, device=dev)
    _expect_error(ERR_UNSUPPORTED, lambda: ops.conv_wgrad_tc(x, g, dk, 3, 1))


def test_entry_points_check_dtypes_and_shapes():
    dev = _dev()
    lib = _lib.load()
    img = torch.zeros(9 * 64 * 128, dtype=torch.bfloat16, device=dev)
    x = torch.zeros(1, 8, 64, 64, dtype=torch.bfloat16, device=dev)
    out = torch.zeros(1, 8, 64, 128, device=dev)

    def fwd(img=img, x=x, out=out, stats=None, cout=128):
        d = [_lib.dl(t) for t in (img, x, out, stats)]
        _lib.check(lib.asep_conv_tc_forward(d[0].ptr, None, 3, 64, cout, 1, d[1].ptr, None, None, d[2].ptr, d[3].ptr,
                                            None, _lib.stream_ptr()))

    _expect_error(ERR_BAD_DTYPE, lambda: fwd(x=x.float()))
    _expect_error(ERR_BAD_DTYPE, lambda: fwd(img=img.float()))
    _expect_error(ERR_BAD_DTYPE, lambda: fwd(stats=torch.zeros(1, 128, 2, device=dev)))
    _expect_error(ERR_BAD_SHAPE, lambda: fwd(out=torch.zeros(1, 8, 64, 192, device=dev)))
    _expect_error(ERR_BAD_SHAPE, lambda: fwd(img=img[:-64]))
    _expect_error(ERR_BAD_SHAPE, lambda: fwd(stats=torch.zeros(1, 128, 3, dtype=torch.float64, device=dev)))
    _expect_error(ERR_UNSUPPORTED, lambda: ops.conv_tc_image(torch.zeros(3, 3, 96, 128)))
    _expect_error(ERR_BAD_SHAPE, lambda: ops.conv_wgrad_tc(x, _bf(out), torch.zeros(3, 3, 64, 192, device=dev), 3, 1))


def test_empty_batch_launches_nothing():
    dev = _dev()
    op = _ops(1, 1, 8, 64, 64, 128, 3)
    img = ops.conv_tc_image(op["k"])
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    x = torch.zeros(0, 8, 64, 64, dtype=torch.bfloat16, device=dev)
    out, st, ob = ops.conv_tc_forward(img, x, 3, 64, 128, 1, bias=op["bias"], stats=True, out_bf16=True)
    dk = torch.ones(3, 3, 64, 128, device=dev)
    ops.conv_wgrad_tc(x, torch.zeros(0, 8, 64, 128, dtype=torch.bfloat16, device=dev), dk, 3, 1)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0
    assert out.shape == (0, 8, 64, 128) and st.shape == (0, 128, 2) and bool((dk == 1).all())
