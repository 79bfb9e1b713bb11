"""The tensor-core coupling network of the Glow prior one launch at a time against the float64 oracle
(oracle/coupling_tc_oracle.py): k_nn_tc4 (BF16 / FP16) and k_nn_tcx (BF16X2 / FP16X2 / FP16X3), forward and data
gradient, at the three levels of the melspec model, from one tile to 42 rounds of 148 tiles; k_wgrad_tc at the shapes of
the training step; the argument checks of both entry points; the level widths the kernels refuse.

The BF16 forward and every one-product data gradient hand out their intermediates (bf16 dumps): each stage is checked
from the kernel's own input and every dump must lie in the rounding bracket of its float64 reference.  The other modes
are held to the magnitude chain.  The gates and the defects they reject are checked on the CPU in
tests/test_oracle_coupling_tc.py.  Run with -s to see the worst ratio per kernel, mode and gate."""
import pytest
import torch

from audiosourcesep_b200 import GlowConfig, _lib, ops
from audiosourcesep_b200.glow import Glow
from audiosourcesep_b200.weights import init_glow_params
from oracle import coupling_tc_oracle as ct

pytestmark = pytest.mark.gpu

ERR_BAD_ARG, ERR_BAD_SHAPE, ERR_BAD_DTYPE, ERR_UNSUPPORTED = -1, -2, -3, -9
PREC = {"bf16": _lib.PREC_BF16, "fp16": _lib.PREC_FP16, "bf16x2": _lib.PREC_BF16X2, "fp16x2": _lib.PREC_FP16X2,
        "fp16x3": _lib.PREC_FP16X3}
CFG = ct.melspec_config()
PARAMS = ct.near_kink_params(CFG, seed=11)
WORST = {}
_MODELS, _NETS = {}, {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    for name, r in sorted(WORST.items()):
        print(f"\n{name}: worst {r:.3e}")


def _dev():
    return torch.device("cuda", _lib.init())


def _model(mode):
    if mode not in _MODELS:
        _MODELS[mode] = Glow(CFG, PARAMS, precision=PREC[mode])
    return _MODELS[mode]


def _net(mode, block, step):
    key = (mode, block, step)
    if key not in _NETS:
        _NETS[key] = ct.TcNet(PARAMS, f"b{block}/s{step}/", CFG.level_shape(block)[2], mode).to(_dev())
    return _NETS[key]


def _kernel(mode, backward):
    if ct.spec(mode)["pairs"]:
        return "k_nn_tcx" + ("<bwd>" if backward else "<fwd>")
    return "k_nn_tc4" + ("<bwd>" if backward else "<fwd>")


def _buffers(mode, block, N, backward, masks_out, dumps, out=True):
    """Sentinel-filled outputs of one launch."""
    Hb, Wb, C = CFG.level_shape(block)
    M = N * Hb * Wb
    dev = _dev()
    net = _net(mode, block, 0)
    n3p = net.n3p["bwd" if backward else "fwd"]
    b = {"G": torch.full((ct.spec(mode)["nparts"], (M + 127) // 128 * 128 * n3p), float("nan"), device=dev)}
    if masks_out:
        b["mask1"] = torch.full((M, 16), 0x5A5A5A5A, dtype=torch.int32, device=dev)
        b["mask2"] = torch.full((M, 16), 0x5A5A5A5A, dtype=torch.int32, device=dev)
    if dumps:
        b["dump1"] = torch.full((M, 512), float("nan"), dtype=torch.bfloat16, device=dev)
        b["dump2"] = torch.full((M, 512), float("nan"), dtype=torch.bfloat16, device=dev)
    if out:
        b["out"] = torch.full((N, Hb, Wb, C // 2 if backward else C), float("nan"), device=dev)
    return b


def _run(mode, block, step, backward, src, masks=None, masks_out=False, dumps=False, out=True):
    b = _buffers(mode, block, src.shape[0], backward, masks_out, dumps, out)
    m1, m2 = masks if masks is not None else (b.get("mask1"), b.get("mask2"))
    ops.glow_coupling_tc(_model(mode), block, step, backward, src, b["G"], mask1=m1, mask2=m2, dump1=b.get("dump1"),
                         dump2=b.get("dump2"), out=b.get("out"))
    torch.cuda.synchronize()
    return b


def _src(block, N, seed, backward):
    Hb, Wb, C = CFG.level_shape(block)
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(N, Hb, Wb, C, generator=g) * (1.0 if backward else 0.7)).to(_dev())


def _check(mode, block, step, backward, src, res, masks=None):
    gates = ct.check_launch(_net(mode, block, step), src, backward, res, masks=masks)
    kern = _kernel(mode, backward)
    for name, value, limit in gates:
        key = f"{kern} {mode} {name} (gate {limit:.3g})"
        WORST[key] = max(WORST.get(key, 0.0), float(value))
    bad = ct.failed(gates)
    assert not bad, f"{kern} {mode} block {block} N {src.shape[0]}: {bad}"


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _same(a, b):
    for k in a:
        assert torch.equal(_bits(a[k]), _bits(b[k])), f"{k} differs between two identical calls"


# (block, N): one tile per level, a ragged M (288 rows), two rounds with a short second one (156 tiles), three rounds
SHAPES = [(0, 1), (1, 1), (2, 1), (2, 3), (0, 13), (1, 30), (2, 30), (0, 30)]


@pytest.mark.parametrize("block,N", SHAPES, ids=[f"b{b}-n{n}" for b, n in SHAPES])
@pytest.mark.parametrize("mode", ct.MODES)
def test_forward_and_data_gradient(mode, block, N):
    """Forward with masks (and dumps in the one-product modes), forward without masks, data gradient on the forward's
    masks and on random masks: every gate, sentinels overwritten, a second call bitwise equal."""
    one = not ct.spec(mode)["pairs"]
    step = N % 2
    x = _src(block, N, 100 * block + N, False)
    fwd = _run(mode, block, step, False, x, masks_out=True, dumps=one)
    _check(mode, block, step, False, x, fwd)
    _same(fwd, _run(mode, block, step, False, x, masks_out=True, dumps=one))
    plain = _run(mode, block, step, False, x)                        # the kernel instantiated without mask output
    assert torch.equal(_bits(plain["G"]), _bits(fwd["G"])) and torch.equal(_bits(plain["out"]), _bits(fwd["out"]))
    M = x.shape[0] * x.shape[1] * x.shape[2]
    gr = _src(block, N, 7 + N, True)
    for masks in ((fwd["mask1"], fwd["mask2"]), ct.random_masks(M, N, _dev())):
        bwd = _run(mode, block, step, True, gr, masks=masks, dumps=one)
        _check(mode, block, step, True, gr, bwd, masks=masks)
        _same(bwd, _run(mode, block, step, True, gr, masks=masks, dumps=one))


@pytest.mark.parametrize("backward", [False, True], ids=["fwd", "bwd"])
def test_many_rounds(backward):
    """Block 0 at N = 512: 6144 tiles, 42 rounds of 148 CTAs, staged and exact (BF16)."""
    mode, block, N = "bf16", 0, 512
    x = _src(block, N, 1, False)
    fwd = _run(mode, block, 0, False, x, masks_out=True, dumps=not backward)
    if not backward:
        _check(mode, block, 0, False, x, fwd)
        return
    gr = _src(block, N, 2, True)
    masks = (fwd["mask1"], fwd["mask2"])
    bwd = _run(mode, block, 0, True, gr, masks=masks, dumps=True)
    _check(mode, block, 0, True, gr, bwd, masks=masks)


# ------------------------------------------------------------------ weight gradient
WG = [(P, ldb, nv) for P in (1, 40, 63, 64, 65, 640, 46080) for ldb, nv in ((64, 18), (64, 36), (128, 72), (192, 144),
                                                                            (512, 512))]


@pytest.mark.parametrize("P,ldb,n_valid", WG, ids=[f"p{p}-ldb{l}-n{n}" for p, l, n in WG])
def test_wgrad_matches_float64(P, ldb, n_valid):
    dev = _dev()
    g = torch.Generator().manual_seed(P + ldb)
    A = torch.relu(torch.randn(P, 512, generator=g)).to(torch.bfloat16).to(dev)
    B = torch.randn(P, ldb, generator=g).to(torch.bfloat16)
    B[:, n_valid:] = 0
    B = B.to(dev)
    ldo = n_valid + 3
    out0 = torch.randn(512, ldo, generator=g).to(dev)
    out0[:, n_valid:] = 12345.0
    out = out0.clone()
    ops.glow_wgrad_tc(A, B, n_valid, out)
    torch.cuda.synchronize()
    ref, scale = ct.wgrad_ref(A, B, out0, n_valid)
    r = ct._ratio(out[:, :n_valid], ref, scale)
    tau = ct.wgrad_tau(P, ldb)
    key = "k_wgrad_tc |got-ref|/(tau A) (gate 1)"
    WORST[key] = max(WORST.get(key, 0.0), r / tau)
    assert r <= tau, (r, tau)
    assert torch.equal(out[:, n_valid:], out0[:, n_valid:])


# ------------------------------------------------------------------ argument checks
def _status(fn):
    n0 = _lib.launch_count()
    with pytest.raises(_lib.AsepError) as e:
        fn()
    assert _lib.launch_count() == n0, "a rejected call launched something"
    return e.value.code


def test_coupling_tc_rejects_before_launch():
    dev = _dev()
    block, N = 2, 1
    b = _buffers("bf16", block, N, False, True, True)
    bx = _buffers("bf16x2", block, N, True, False, False)
    x = _src(block, N, 0, False)
    call = lambda mode, **kw: ops.glow_coupling_tc(_model(mode), kw.pop("block", block), kw.pop("step", 0),  # noqa: E731
                                                  kw.pop("backward", False), kw.pop("src", x), kw.pop("G", b["G"]), **kw)
    m32 = Glow(CFG, PARAMS, precision=_lib.PREC_FP32)
    assert _status(lambda: ops.glow_coupling_tc(m32, block, 0, False, x, b["G"])) == ERR_UNSUPPORTED
    assert _status(lambda: call("bf16", block=3)) == ERR_BAD_ARG
    assert _status(lambda: call("bf16", step=2)) == ERR_BAD_ARG
    assert _status(lambda: call("bf16", step=-1)) == ERR_BAD_ARG
    assert _status(lambda: call("bf16x2", G=bx["G"], dump1=b["dump1"])) == ERR_UNSUPPORTED
    assert _status(lambda: call("bf16", backward=True, mask1=b["mask1"])) == ERR_BAD_ARG
    assert _status(lambda: call("bf16", mask1=b["mask1"])) == ERR_BAD_ARG
    assert _status(lambda: call("bf16", src=x[..., :8].contiguous())) == ERR_BAD_SHAPE
    assert _status(lambda: call("bf16", G=b["G"][:, :-16].contiguous())) == ERR_BAD_SHAPE
    assert _status(lambda: call("bf16x2", G=b["G"])) == ERR_BAD_SHAPE                  # one part where there are two
    assert _status(lambda: call("bf16", out=torch.empty(N, 12, 8, 8, device=dev))) == ERR_BAD_SHAPE
    assert _status(lambda: call("bf16", mask1=b["mask1"][:, :8].contiguous(), mask2=b["mask2"])) == ERR_BAD_SHAPE
    assert _status(lambda: call("bf16", dump1=torch.empty(96, 256, dtype=torch.bfloat16, device=dev))) == ERR_BAD_SHAPE
    assert _status(lambda: call("bf16", src=x.double())) == ERR_BAD_DTYPE
    assert _status(lambda: call("bf16", mask1=b["mask1"].float(), mask2=b["mask2"])) == ERR_BAD_DTYPE
    assert _status(lambda: call("bf16", dump1=b["dump1"].float())) == ERR_BAD_DTYPE
    call("bf16", mask1=b["mask1"], mask2=b["mask2"], dump1=b["dump1"], dump2=b["dump2"], out=b["out"])   # the valid call


def test_wgrad_tc_rejects_before_launch():
    dev = _dev()
    A = torch.zeros(64, 512, dtype=torch.bfloat16, device=dev)
    out = torch.zeros(512, 512, device=dev)
    B = lambda ldb: torch.zeros(64, ldb, dtype=torch.bfloat16, device=dev)  # noqa: E731
    for ldb in (96, 320, 384):
        assert _status(lambda: ops.glow_wgrad_tc(A, B(ldb), 18, out)) == ERR_UNSUPPORTED
    assert _status(lambda: ops.glow_wgrad_tc(A, B(64), 65, out)) == ERR_BAD_ARG
    assert _status(lambda: ops.glow_wgrad_tc(A, B(64), 0, out)) == ERR_BAD_ARG
    assert _status(lambda: ops.glow_wgrad_tc(A, B(64), 18, out[:, :16].contiguous())) == ERR_BAD_SHAPE
    assert _status(lambda: ops.glow_wgrad_tc(A[:32].contiguous(), B(64), 18, out)) == ERR_BAD_SHAPE
    assert _status(lambda: ops.glow_wgrad_tc(A.float(), B(64), 18, out)) == ERR_BAD_DTYPE
    assert _status(lambda: ops.glow_wgrad_tc(A, B(64), 18, out.double())) == ERR_BAD_DTYPE


# ------------------------------------------------------------------ level widths
def test_unsupported_level_width_refused_at_prepare():
    """C = 3: level widths 12 and 24, outside the tensor-core kernels (4, 8, 16): refused at prepare in every
    tensor-core precision before anything is launched; the fp32 path keeps reporting its own unsupported width."""
    cfg = GlowConfig(H=32, W=16, C=3, L=2, K=1, n_filters=512)
    p = init_glow_params(cfg, seed=1)
    for mode, prec in PREC.items():
        code = _status(lambda: Glow(cfg, p, precision=prec))
        assert code == ERR_UNSUPPORTED, mode
    m = Glow(cfg, p, precision=_lib.PREC_FP32)
    x = torch.rand(1, 32, 16, 3, device=_dev())
    with pytest.raises(_lib.AsepError) as e:
        m.log_prob(x)
    assert e.value.code == ERR_UNSUPPORTED and "channel count" in str(e.value)
