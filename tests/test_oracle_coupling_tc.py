"""The float64 oracle of the tensor-core coupling network (oracle/coupling_tc_oracle.py) checked on the CPU: a CPU
emulation of every mode's arithmetic passes every gate, each defect a kernel is likely to have fails its gate, the
layouts round-trip, and the fp32-weight network is the Glow oracle's ShiftAndLogScaleConvNet."""
import numpy as np
import pytest
import torch

from oracle import coupling_tc_oracle as ct
from oracle.glow_oracle import GlowOracle

CFG = ct.melspec_config()
PARAMS = ct.near_kink_params(CFG, seed=5)
N, H, W = 2, 12, 8          # 192 pixels: two tiles, the second one ragged
BLOCK_OF_C = {4: 0, 8: 1, 16: 2}


def _net(C, mode, step=0):
    return ct.TcNet(PARAMS, f"b{BLOCK_OF_C[C]}/s{step}/", C, mode)


def _src(C, seed, backward=False):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, H, W, C, generator=g) * (1.0 if backward else 0.7)


def _launch(net, backward, seed=0, defect=None, random_masks=False):
    C = net.C
    masks = None
    if backward:
        if random_masks:
            masks = ct.random_masks(N * H * W, seed)
        else:
            fwd = ct.emulate(net, _src(C, seed), False)
            masks = (fwd["mask1"], fwd["mask2"])
    src = _src(C, seed + 1, backward) if backward else _src(C, seed)
    res = ct.emulate(net, src, backward, masks=masks, defect=defect)
    return ct.check_launch(net, src, backward, res, masks=masks)


@pytest.mark.parametrize("C", [4, 8, 16])
@pytest.mark.parametrize("backward", [False, True], ids=["fwd", "bwd"])
@pytest.mark.parametrize("mode", ct.MODES)
def test_emulation_passes_every_gate(mode, backward, C):
    gates = _launch(_net(C, mode), backward, seed=C)
    assert not ct.failed(gates), ct.failed(gates)
    names = [g[0] for g in gates]
    assert any(n.startswith("G part") for n in names) and "out != gather(G) (elements)" in names
    if backward:
        assert not ct.failed(_launch(_net(C, mode), True, seed=C, random_masks=True))


# (defect, mode, backward): every defect on a mode where it can occur; each must fail at least one gate
PLANTED = [
    ("drop_k1", "bf16", False), ("drop_k2", "bf16", False), ("drop_k3", "bf16", False),
    ("drop_k1", "bf16", True), ("drop_k2", "bf16", True), ("drop_k3", "bf16", True),
    ("drop_k1", "fp16x3", False), ("drop_k2", "bf16x2", False), ("drop_k3", "fp16x2", True),
    ("tap_sign", "bf16", False), ("tap_sign", "bf16", True), ("swap_dxdy", "bf16", False), ("swap_dxdy", "fp16", True),
    ("read_xa", "bf16", False), ("read_xa", "fp16x3", False),
    ("no_x_lo", "bf16", False), ("no_x_lo", "bf16", True), ("no_x_lo", "fp16x3", False),
    ("no_h_lo", "bf16x2", False), ("no_w_lo", "fp16x3", False),
    ("no_inv_scale", "fp16x3", False),
    ("swap_mask_words", "bf16", False), ("swap_mask_words", "fp16x2", False),
    ("stale_tile", "bf16", False), ("stale_tile", "bf16x2", True),
    ("unwritten_tail_row", "bf16", False), ("unwritten_tail_row", "fp16x3", True),
]


@pytest.mark.parametrize("defect,mode,backward", PLANTED, ids=[f"{d}-{m}-{'bwd' if b else 'fwd'}" for d, m, b in PLANTED])
def test_planted_defect_fails_its_gate(defect, mode, backward):
    assert defect in ct.DEFECTS
    C = 8
    gates = _launch(_net(C, mode), backward, seed=3, defect=defect)
    assert ct.failed(gates), f"{defect} passed every gate: {gates}"


def test_fp32_weight_network_equals_glow_oracle():
    o = GlowOracle(CFG, PARAMS)
    for b in range(3):
        Hb, Wb, C = CFG.level_shape(b)
        net = ct.TcNet(PARAMS, f"b{b}/s1/", C, "bf16")
        xb = torch.randn(1, Hb, Wb, C // 2, generator=torch.Generator().manual_seed(b), dtype=torch.float64).float()
        ls, t = net.fp32_net(xb)
        ls0, t0 = o.nn(xb.double(), f"b{b}/s1/")
        # the only difference: the float32 rounding of the folded BatchNorm and of the products g'.K (2^-24 each)
        scale = float(t0.abs().max())
        assert float((t - t0).abs().max()) <= 1e-5 * scale
        assert float((ls - ls0).abs().max()) <= 1e-5 * max(1.0, float(ls0.abs().max()))


def test_weights_follow_prepare():
    """bf16 / fp16 tile-image weights, the x256 three-product scale and its residuals, the transposed backward sets."""
    net = _net(8, "fp16x3")
    w = net.w["fwd"]
    k1 = net.raw["k1"]
    assert torch.equal(w["s1"][0], k1.mul(256).half().float())
    assert torch.equal(w["s1"][1], (k1.mul(256) - w["s1"][0]).half().float())
    assert w["scale"] == 1 / 256
    assert net.w["bwd"]["scale"] == 1.0
    assert torch.equal(net.w["bwd"]["s3"][0], k1.T.bfloat16().float())
    assert torch.equal(net.w["bwd"]["s2"][0], net.raw["w2"].T.bfloat16().float())
    b = _net(8, "bf16")
    assert b.w["fwd"]["s2"][1] is None and torch.equal(b.w["fwd"]["s2"][0], b.raw["w2"].bfloat16().float())
    assert _net(8, "fp16").w["fwd"]["s1"][0].equal(k1.bfloat16().float())     # stage 1 stays bf16 in FP16
    assert net.n3p == {"fwd": 80, "bwd": 48}


def test_mask_pack_roundtrip():
    gen = torch.Generator().manual_seed(0)
    bits = torch.rand(37, 512, generator=gen) > 0.5
    w = ct.pack_masks(bits)
    assert w.dtype == torch.int32 and w.shape == (37, 16)
    assert torch.equal(ct.unpack_masks(w), bits)
    one = torch.zeros(1, 512, dtype=torch.bool)
    one[0, 64 * 3 + 32 + 5] = True                     # panel 3, second 32 columns, bit 5 -> word 1*8 + 3
    assert ct.pack_masks(one)[0].tolist() == [0] * 11 + [1 << 5] + [0] * 4
    words = ct.random_masks(5, 1)[0]
    assert torch.equal(ct.pack_masks(ct.unpack_masks(words)), words)


def test_g_tile_roundtrip():
    rows = torch.arange(256 * 48, dtype=torch.float32).reshape(256, 48)
    flat = ct.tile_g(rows)
    # element (p, col) sits at (p >> 7) * 128 n3p + (col >> 2) * 512 + (p & 127) * 4 + (col & 3)   (g_index of nn_tc)
    p, col = 200, 37
    assert float(flat[(p >> 7) * 128 * 48 + (col >> 2) * 512 + (p & 127) * 4 + (col & 3)]) == float(rows[p, col])
    assert torch.equal(ct.untile_g(flat, 48), rows)


def test_gather_restatement_matches_float64():
    """The float32 col2im restatement equals the float64 sums up to its own 11 roundings."""
    g = torch.Generator().manual_seed(4)
    C = 8
    parts = [torch.randn(N * H * W, 80, generator=g) for _ in range(2)]
    const3, c3 = torch.randn(72, generator=g), torch.randn(C, generator=g)
    r32 = ct.gather_fwd(parts, const3, c3, N, H, W, C)
    r64 = ct.gather_fwd(parts, const3, c3, N, H, W, C, exact=True)
    m = ct.gather_fwd([p.abs() for p in parts], const3.abs(), c3.abs(), N, H, W, C, exact=True)
    assert float(((r32.double() - r64).abs() / m).max()) <= ct.GATHER_TAU
    # border: the corner pixel sums the four in-bounds taps only
    ref = c3[0] + sum(parts[0][0 + dy * W + dx, tap * C] + parts[1][0 + dy * W + dx, tap * C] + const3[tap * C]
                      for tap, (dy, dx) in ((4, (0, 0)), (5, (0, 1)), (7, (1, 0)), (8, (1, 1))))
    assert abs(float(r64[0, 0, 0, 0]) - float(ref)) < 1e-5


def _wgrad_emulate(A, B, out0, n_valid, drop_slice=None):
    """fp32 per-slice sums added to out0 in fp32, as the kernel's atomics do."""
    slices, per = ct.wgrad_split(A.shape[0], B.shape[1])
    out = out0.clone()
    for s in range(slices):
        if s == drop_slice:
            continue
        rows = slice(s * per * 64, (s + 1) * per * 64)
        out[:, :n_valid] += (A[rows].double().T @ B[rows, :n_valid].double()).float()
    return out


@pytest.mark.parametrize("P,ldb,n_valid", [(1, 64, 18), (640, 128, 72), (46080, 64, 36), (4000, 512, 512)])
def test_wgrad_gate(P, ldb, n_valid):
    g = torch.Generator().manual_seed(P)
    A = torch.randn(P, 512, generator=g).bfloat16().float()
    B = torch.randn(P, ldb, generator=g).bfloat16().float()
    out0 = torch.randn(512, ldb, generator=g)
    tau = ct.wgrad_tau(P, ldb)
    ref, scale = ct.wgrad_ref(A, B, out0, n_valid)
    got = _wgrad_emulate(A, B, out0, n_valid)
    assert ct._ratio(got[:, :n_valid], ref, scale) <= tau
    slices, _ = ct.wgrad_split(P, ldb)
    if slices > 1:     # one split-K slice dropped
        bad = _wgrad_emulate(A, B, out0, n_valid, drop_slice=slices - 1)
        assert ct._ratio(bad[:, :n_valid], ref, scale) > tau
    assert ct.wgrad_split(46080, 64) == (36, 20)
    assert ct.wgrad_split(46080, 512) == (18, 40)


def test_wgrad_split_defect_slice_rows():
    """The dropped-slice reference leaves out exactly the pixels of that slice."""
    A = torch.ones(640, 512)
    B = torch.ones(640, 64)
    slices, per = ct.wgrad_split(640, 64)
    ref, _ = ct.wgrad_ref(A, B, torch.zeros(512, 64), 64, drop_slice=0)
    assert float(ref[0, 0]) == 640 - per * 64
    np.testing.assert_equal(slices * per * 64 >= 640, True)
