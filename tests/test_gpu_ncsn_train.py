"""GPU parity tests of the NCSN denoising-score-matching train step (train_ncsn.py:26-57) vs the float64 autograd oracle."""
import numpy as np
import pytest
import torch

from audiosourcesep_b200 import NCSNConfig
from audiosourcesep_b200.weights import init_ncsn_params
from oracle import basis_oracle as bo
from oracle import train_ncsn_oracle as to
from oracle.train_oracle import adam_update

pytestmark = pytest.mark.gpu


def _cfg(version):
    # the reference widths (192 / 128 filters) on a 32 x 32 patch: every layer shape class of the 96 x 64 networks
    # (full / half resolution, dilation 1 / 2 / 4, 1x1 shortcut, pooled and up-sampled branches) at 1/6 of the cost
    if version == "v1":
        return NCSNConfig(version="v1", H=32, W=32, ngf=192, num_classes=10, sigma1=1.0, sigmaL=0.01)
    return NCSNConfig(version="v2", H=32, W=32, ngf=128, num_classes=12, sigma1=1.0, sigmaL=0.01)


def _setup(version, precision, n=3, seed=5):
    from audiosourcesep_b200 import _lib
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    cfg = _cfg(version)
    params = init_ncsn_params(cfg, seed=seed, mode="perturbed")
    sig = bo.get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, cfg.progression)
    model = ScoreModel(cfg, params, sigmas=sig, precision={"bf16": _lib.PREC_BF16, "x3": _lib.PREC_BF16X3}[precision])
    model.enable_training()
    rng = np.random.default_rng(11)
    x = rng.random((n, cfg.H, cfg.W, 1)).astype(np.float32)
    z = rng.standard_normal((n, cfg.H, cfg.W, 1)).astype(np.float32)
    idx = np.array([cfg.num_classes - 1, cfg.num_classes // 2, 2][:n], dtype=np.int32)   # one level per SAMPLE (general path)
    return cfg, params, sig, model, x, z, idx


@pytest.mark.parametrize("version", ["v1", "v2"])
def test_dsm_gradients_match_autograd_oracle_split_bf16(version):
    """Parity mode (three split-bf16 products in all three GEMMs of every convolution): loss and the gradient of every
    parameter tensor against torch autograd in float64."""
    cfg, params, sig, model, x, z, idx = _setup(version, "x3")
    gb = 6                                                   # global batch larger than the local one (data-parallel scaling)
    loss_ref, g_ref = to.dsm_loss_and_grads(cfg, params, sig, x, z, idx, gb)
    grads, loss = model.train_grads(torch.as_tensor(x), torch.as_tensor(z), torch.as_tensor(idx), gb)
    got = model.unflatten(grads)
    assert abs(loss.item() - loss_ref) <= 2e-4 * abs(loss_ref), (loss.item(), loss_ref)
    total = np.sqrt(sum(float(np.sum(g ** 2)) for g in g_ref.values()))
    rows = []
    for name, want in g_ref.items():
        err = float(np.linalg.norm(got[name] - want))
        rows.append((err / max(float(np.linalg.norm(want)), 1e-3 * total / np.sqrt(len(g_ref))), name, float(np.linalg.norm(want))))
    rows.sort(reverse=True)
    for r in rows[:8]:
        print(f"[{version}] rel err {r[0]:.3e}  |g| {r[2]:.3e}  {r[1]}")
    flat_err = np.sqrt(sum(float(np.sum((got[n] - g_ref[n]) ** 2)) for n in g_ref)) / total
    print(f"[{version}] whole-gradient relative error {flat_err:.3e}, loss {loss.item():.6f} vs {loss_ref:.6f}")
    assert np.all(np.isfinite(grads.cpu().numpy()))
    if version == "v1":
        assert rows[0][0] <= 5e-4, rows[:5]
        assert flat_err <= 2e-4
    else:
        # v2 routes gradients through 5x5 MAX pooling (score_network_v2.py:15-25): the arg-max of a window flips when two
        # taps differ by less than the forward arithmetic's error, so two correct implementations disagree by far more
        # than their forward error (torch fp32 vs torch fp64 autograd on this very case: 7.5e-5 whole gradient, 4.4e-4
        # worst tensor, against 1.3e-6 / 2.7e-6 for v1).  Every tensor DOWNSTREAM of the last max-pool must be tight;
        # the rest is bounded loosely.
        after_last_pool = [r for r in rows if r[1].startswith(("end_conv", "normalizer", "refine4/RCU_output", "refine4/CRP/conv_2"))]
        assert len(after_last_pool) >= 10 and max(r[0] for r in after_last_pool) <= 5e-4, after_last_pool[:5]
        assert rows[0][0] <= 3e-2, rows[:5]
        assert flat_err <= 1.5e-2


@pytest.mark.parametrize("version", ["v1", "v2"])
def test_dsm_gradients_throughput_mode(version):
    """One bf16 product per GEMM: the whole-gradient direction stays within a few percent of the float64 oracle."""
    cfg, params, sig, model, x, z, idx = _setup(version, "bf16")
    loss_ref, g_ref = to.dsm_loss_and_grads(cfg, params, sig, x, z, idx, 3)
    grads, loss = model.train_grads(torch.as_tensor(x), torch.as_tensor(z), torch.as_tensor(idx), 3)
    got = model.unflatten(grads)
    total = np.sqrt(sum(float(np.sum(g ** 2)) for g in g_ref.values()))
    flat_err = np.sqrt(sum(float(np.sum((got[n] - g_ref[n]) ** 2)) for n in g_ref)) / total
    print(f"[{version}] bf16 whole-gradient relative error {flat_err:.3e}, loss {loss.item():.5f} vs {loss_ref:.5f}")
    assert abs(loss.item() - loss_ref) <= 5e-2 * abs(loss_ref)
    assert flat_err <= (1e-1 if version == "v1" else 2e-1)       # (v2: max-pool routing, see the parity-mode test)


def test_adam_trajectory_and_inference_after_update():
    """Two Keras-Adam steps on the flat vector follow the float32 numpy restatement fed with the CUDA gradients; the
    tile images are rebuilt on the device, so the score network evaluates with the UPDATED weights and the loss of
    the same batch goes down."""
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    from audiosourcesep_b200 import _lib
    cfg, params, sig, model, x, z, idx = _setup("v2", "x3")
    lr = 2e-5        # (Adam moves every weight by ~lr per step whatever the gradient scale: 1e-3 overshoots these random nets)
    opt = dict(kind="adam", lr=lr, beta1=0.9, beta2=0.999, eps=1e-7)
    theta = model.get_flat().cpu().numpy()
    m = np.zeros_like(theta)
    v = np.zeros_like(theta)
    losses = []
    for t in (1, 2, 3):
        grads, loss = model.train_grads(torch.as_tensor(x), torch.as_tensor(z), torch.as_tensor(idx), 3)
        losses.append(loss.item())
        theta, m, v = adam_update(theta, grads.cpu().numpy(), m, v, t, lr=lr)
        model.apply_gradients(grads, opt)
        got = model.get_flat().cpu().numpy()
        assert np.max(np.abs(got - theta)) <= 1e-6 * max(1.0, float(np.max(np.abs(theta)))), t
    print("losses", losses)
    assert losses[2] < losses[0]
    # a fresh inference handle holding the trained weights gives the same score as the training handle
    model.sync_host()
    fresh = ScoreModel(cfg, model.variables, sigmas=sig, precision=_lib.PREC_BF16X3)
    xs = torch.as_tensor(x)
    a = model.score(xs, torch.as_tensor(idx)).cpu().numpy()
    b = fresh.score(xs, torch.as_tensor(idx)).cpu().numpy()
    assert np.linalg.norm(a - b) <= 1e-5 * np.linalg.norm(b)
    # set_flat round trip (data-parallel broadcast / checkpoint restore)
    model.set_flat(torch.as_tensor(theta))
    assert np.array_equal(model.get_flat().cpu().numpy(), theta)


def test_dsm_gradients_at_the_reference_patch_size():
    """The v1 network of configs/melspec_ncsnv1.yml (96 x 64 patches, 192 filters, 10 noise levels) in the parity mode:
    whole-gradient and worst-tensor error against float64 autograd at the size every config uses (the 32 x 32 cases above
    cover the layer classes; this one covers the tile counts, the W = 64 / 32 tensor maps and the split-K sizes of the real shape)."""
    from audiosourcesep_b200 import _lib
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    cfg = NCSNConfig(version="v1", H=96, W=64, ngf=192, num_classes=10, sigma1=1.0, sigmaL=0.01)
    params = init_ncsn_params(cfg, seed=7, mode="perturbed")
    sig = bo.get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, cfg.progression)
    model = ScoreModel(cfg, params, sigmas=sig, precision=_lib.PREC_BF16X3)
    model.enable_training()
    rng = np.random.default_rng(3)
    x = rng.random((2, 96, 64, 1)).astype(np.float32)
    z = rng.standard_normal((2, 96, 64, 1)).astype(np.float32)
    idx = np.array([9, 4], dtype=np.int32)
    loss_ref, g_ref = to.dsm_loss_and_grads(cfg, params, sig, x, z, idx, 32)
    grads, loss = model.train_grads(torch.as_tensor(x), torch.as_tensor(z), torch.as_tensor(idx), 32)
    got = model.unflatten(grads)
    total = np.sqrt(sum(float(np.sum(g ** 2)) for g in g_ref.values()))
    flat_err = np.sqrt(sum(float(np.sum((got[n] - g_ref[n]) ** 2)) for n in g_ref)) / total
    worst = max((float(np.linalg.norm(got[n] - g_ref[n])) / max(float(np.linalg.norm(g_ref[n])), 1e-3 * total / np.sqrt(len(g_ref))), n)
                for n in g_ref)
    print(f"[v1 96x64] whole-gradient relative error {flat_err:.3e}, worst tensor {worst[0]:.3e} ({worst[1]}), loss {loss.item():.6f} vs {loss_ref:.6f}")
    assert abs(loss.item() - loss_ref) <= 2e-4 * abs(loss_ref)
    assert flat_err <= 2e-4 and worst[0] <= 1e-3


def test_enable_training_rejects_a_patch_the_weight_gradient_does_not_tile():
    """The forward convolution tiles W up to 128, the weight gradient only up to 64: a W = 128 score network runs
    inference, and enable_training refuses it up front (ASEP_ERR_UNSUPPORTED) instead of the first train step."""
    from audiosourcesep_b200 import _lib
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    cfg = NCSNConfig(version="v2", H=8, W=128, ngf=128, num_classes=4, sigma1=1.0, sigmaL=0.01)
    sig = bo.get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, cfg.progression)
    model = ScoreModel(cfg, init_ncsn_params(cfg, seed=1, mode="perturbed"), sigmas=sig, precision=_lib.PREC_BF16)
    score = model.score(torch.rand(2, cfg.H, cfg.W, 1), 1)
    assert bool(torch.isfinite(score).all())
    with pytest.raises(_lib.AsepError) as e:
        model.enable_training()
    assert e.value.code == -9 and "weight-gradient" in str(e.value)
