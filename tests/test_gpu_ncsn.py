"""GPU parity tests of the NCSN v1 / v2 score networks and of the NCSN-BASIS Langevin loop vs the oracle."""
import numpy as np
import pytest
import torch

from audiosourcesep_b200 import NCSNConfig, synthetic
from audiosourcesep_b200.weights import init_ncsn_params
from oracle import basis_oracle as bo
from oracle.ncsn_oracle import NCSNOracle

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _cfg(version):
    if version == "v1":
        return NCSNConfig(version="v1", ngf=192, num_classes=10, sigma1=1.0, sigmaL=0.01)
    return NCSNConfig(version="v2", ngf=128, num_classes=200, sigma1=30.0, sigmaL=0.01)


def _model(cfg, params, precision=None):
    from audiosourcesep_b200 import _lib
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    sig = bo.get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, cfg.progression)
    return ScoreModel(cfg, params, sigmas=sig, precision=_lib.PREC_BF16 if precision is None else precision), sig


@pytest.mark.parametrize("version", ["v1", "v2"])
@pytest.mark.parametrize("mode", ["perturbed", "faithful"])
def test_score_network_matches_oracle(version, mode):
    cfg = _cfg(version)
    params = init_ncsn_params(cfg, seed=5, mode=mode)
    model, sig = _model(cfg, params)
    oracle = NCSNOracle(cfg, params, sigmas=sig, dtype=torch.float32)
    x = synthetic.normalise(synthetic.mel_patches_db(2, seed=1)) + 0.05 * np.random.default_rng(0).standard_normal((2, 96, 64, 1)).astype(np.float32)
    idx = np.array([0, cfg.num_classes - 1], dtype=np.int32)
    want = oracle.score(x, idx).numpy()
    got = _np(model(([torch.as_tensor(x), torch.as_tensor(idx)]), training=True))
    assert np.all(np.isfinite(got))
    rel = np.linalg.norm(got - want) / np.linalg.norm(want)
    per_sample = [float(np.linalg.norm(got[i] - want[i]) / np.linalg.norm(want[i])) for i in range(2)]
    print(f"[{version}, {mode}] score relative L2 error = {rel:.3e} (per sample {per_sample})")
    # vs the fp32 restatement: bf16 tensor-core operands through 75 convolutions (the bf16-operand restatement of
    # the same graph differs from the fp32 one by 0.9 % for v1 and 3.0 % for v2 with these weights)
    assert rel <= 5e-2, rel
    # vs the restatement with the SAME arithmetic contract (bf16 operands, exact accumulation): tight
    emu = NCSNOracle(cfg, params, sigmas=sig, dtype=torch.float32, bf16_operands=True).score(x, idx).numpy()
    rel_emu = np.linalg.norm(got - emu) / np.linalg.norm(emu)
    print(f"[{version}, {mode}] vs bf16-operand restatement = {rel_emu:.3e}")
    # two bf16-operand evaluations that differ only in accumulation order already disagree at the level at which
    # each disagrees with fp32 (random-weight RefineNets amplify a 2^-9 operand rounding ~15x), so this is a
    # consistency bound, not a tight one
    assert rel_emu <= 5e-2, rel_emu
    # dict call form (train_ncsn.py:43,52) and determinism
    again = _np(model({"perturbed_X": torch.as_tensor(x), "sigma_idx": torch.as_tensor(idx)}))
    assert np.array_equal(got, again)


def test_ncsn_param_count_known_answer():
    cfg = _cfg("v1")
    params = init_ncsn_params(cfg, seed=0, mode="faithful")
    model, _ = _model(cfg, params)
    assert model.count_params() == 67464769          # trained_ncsn/ncsn_piano_192_32_dB_custom_loop/out.log:35


@pytest.mark.parametrize("version", ["v1", "v2"])
def test_score_network_split_bf16_mode_matches_fp32_oracle(version):
    """ASEP_PREC_BF16X3 (operands as hi + lo bf16 pairs, three tcgen05 products per convolution): the score agrees
    with the fp32 restatement at the level two fp32 evaluation orders agree with each other."""
    from audiosourcesep_b200 import _lib
    cfg = _cfg(version)
    params = init_ncsn_params(cfg, seed=5, mode="perturbed")
    model, sig = _model(cfg, params, _lib.PREC_BF16X3)
    x = synthetic.normalise(synthetic.mel_patches_db(2, seed=1)) + 0.05 * np.random.default_rng(0).standard_normal((2, 96, 64, 1)).astype(np.float32)
    idx = np.array([0, cfg.num_classes - 1], dtype=np.int32)
    want64 = NCSNOracle(cfg, params, sigmas=sig, dtype=torch.float64).score(x, idx).numpy()
    want32 = NCSNOracle(cfg, params, sigmas=sig, dtype=torch.float32).score(x, idx).numpy()
    got = _np(model([torch.as_tensor(x), torch.as_tensor(idx)], training=True))
    rel = np.linalg.norm(got - want64) / np.linalg.norm(want64)
    rel32 = np.linalg.norm(want32 - want64) / np.linalg.norm(want64)
    print(f"[{version}, split-bf16] score relative L2 error vs fp64 = {rel:.3e} (the fp32 restatement itself: {rel32:.3e})")
    assert rel <= max(2e-4, 20 * rel32), (rel, rel32)


@pytest.mark.parametrize("version,sigma_idx,gate,x3", [("v1", 9, 1e-3, False), ("v1", 3, 1e-2, False), ("v2", 199, 1e-3, False),
                                                      ("v2", 120, 1e-2, False), ("v1", 3, 1e-3, True), ("v2", 120, 1e-3, True),
                                                      ("v1", 0, 1e-3, True)])
def test_basis_ncsn_inner_loop_vs_oracle(version, sigma_idx, gate, x3):
    """Per-step Langevin state parity with injected noise for the NCSN priors.  In the throughput mode (one bf16
    product per convolution) the north-star gate (<= 1e-3 relative) is asserted at the annealed end of the schedule;
    at the large-step levels the bf16-operand score error (1-3 % with random weights) times eta exceeds it, so those
    cases carry a documented looser bound.  The split-bf16 mode meets the gate at every level."""
    from audiosourcesep_b200 import _lib, ops
    cfg = _cfg(version)
    p1, p2 = init_ncsn_params(cfg, seed=11, mode="perturbed"), init_ncsn_params(cfg, seed=12, mode="perturbed")
    prec = _lib.PREC_BF16X3 if x3 else _lib.PREC_BF16
    (m1, sig), (m2, _) = _model(cfg, p1, prec), _model(cfg, p2, prec)
    o1 = NCSNOracle(cfg, p1, sigmas=sig, dtype=torch.float32)
    o2 = NCSNOracle(cfg, p2, sigmas=sig, dtype=torch.float32)
    n_mixed, T = 2, 2
    mixed, _, _ = synthetic.basis_problem(n_mixed)
    x1, x2 = synthetic.langevin_init(n_mixed, seed=4)
    eta, lam, ns = bo.step_constants(sig, sigma_idx)
    rng = np.random.default_rng(3)
    noise = rng.standard_normal((T, 2, n_mixed, 96, 64, 1)).astype(np.float32)
    g, grad_g = bo.mixing_process("melspec", "dB")
    idx = np.full((n_mixed,), sigma_idx, dtype=np.int64)
    a, b = x1.copy(), x2.copy()
    states = [(a.copy(), b.copy())]
    for t in range(T):
        s1 = o1.score(a, idx).numpy().astype(np.float32)
        s2 = o2.score(b, idx).numpy().astype(np.float32)
        a, b = bo.langevin_update(a, b, s1, s2, mixed, noise[t, 0], noise[t, 1], eta, lam, ns, g, grad_g)
        states.append((a.copy(), b.copy()))
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    worst = 0.0
    for t in range(T):
        t1, t2 = torch.as_tensor(states[t][0]).cuda(), torch.as_tensor(states[t][1]).cuda()
        ops.basis_ncsn_inner(m1, m2, torch.as_tensor(mixed), t1, t2, sigma_idx, 1, float(eta), float(lam), float(ns),
                             noise1=torch.as_tensor(noise[t:t + 1, 0]), noise2=torch.as_tensor(noise[t:t + 1, 1]),
                             nan_count=nan)
        for got, want in ((t1, states[t + 1][0]), (t2, states[t + 1][1])):
            worst = max(worst, float(np.linalg.norm(_np(got) - want) / np.linalg.norm(want)))
    print(f"[{version}, sigma_idx={sigma_idx}, {'split-bf16' if x3 else 'bf16'}] worst per-step state relative error = {worst:.3e}")
    assert worst <= gate, worst
    assert nan.item() == 0


def test_anneal_langevin_dynamics_matches_oracle():
    """ncsn/utils.py:17-38 with injected noise: the unconditional sampler is the lambda = 0 case of the fused update."""
    from audiosourcesep_b200.ncsn.utils import anneal_langevin_dynamics
    cfg = _cfg("v1")
    params = init_ncsn_params(cfg, seed=21, mode="perturbed")
    model, sig = _model(cfg, params)
    oracle = NCSNOracle(cfg, params, sigmas=sig, dtype=torch.float32)
    sig_used = sig[-2:]
    rng = np.random.default_rng(5)
    x0 = rng.uniform(0, 1, (2, 96, 64, 1)).astype(np.float32)
    noise = rng.standard_normal((2, 2, 2, 96, 64, 1)).astype(np.float32)

    class Shifted:                       # the sampler labels levels 0..len(sigmas)-1; test the last two levels of the schedule
        def __init__(self, f, off):
            self.f, self.off = f, off

        def __call__(self, inputs, training=True):
            return self.f([inputs[0], inputs[1] + self.off], training=training)

    got = anneal_langevin_dynamics(x0, [96, 64, 1], Shifted(model, 8), 2, sig_used, n_steps_each=2, step_lr=2e-5, noise=noise)
    want = bo.anneal_langevin_dynamics(x0.copy(), lambda x, i: oracle.score(x, np.full((2,), i + 8)).numpy().astype(np.float32),
                                       sig_used, 2, 2e-5, lambda i, s: noise[i][s])
    rel = np.linalg.norm(got - want) / np.linalg.norm(want)
    print(f"annealed Langevin sampler relative state error = {rel:.3e}")
    assert rel <= 1e-3, rel


@pytest.mark.parametrize("version", ["v1", "v2"])
def test_score_is_sample_wise_at_the_bench_size(version):
    """30 segments (n_mixed of run_basis_sep.py:478): the score of a segment may not depend on the other segments of
    the batch (instance norms are per sample, score_network.py:204-207).  The statistics are accumulated with
    double-precision atomics in arrival order, so the comparison is to 1e-5 relative rather than bit-exact."""
    cfg = _cfg(version)
    params = init_ncsn_params(cfg, seed=5, mode="perturbed")
    model, _ = _model(cfg, params)
    x = torch.as_tensor(synthetic.normalise(synthetic.mel_patches_db(30, seed=2))).cuda()
    idx = torch.full((30,), cfg.num_classes - 1, dtype=torch.int32, device="cuda")
    s = model([x, idx], training=True)
    assert torch.isfinite(s).all()
    perm = torch.randperm(30, generator=torch.Generator().manual_seed(1)).cuda()
    s_perm = model([x[perm].contiguous(), idx], training=True)
    rel = float((s_perm - s[perm]).norm() / s.norm())
    s_one = model([x[7:8].contiguous(), idx[:1]], training=True)
    rel1 = float((s_one - s[7:8]).norm() / s[7:8].norm())
    print(f"[{version}] permutation {rel:.2e}, single segment {rel1:.2e}")
    assert rel <= 1e-5 and rel1 <= 1e-5, (rel, rel1)
    assert model([x[:0].contiguous(), idx[:0]], training=True).shape == (0, 96, 64, 1)      # empty batch


@pytest.mark.parametrize("version", ["v1", "v2"])
def test_ncsn_step_graph_replay_equals_eager_launches(version):
    """ops.basis_ncsn_inner replays steps 2..T as one captured CUDA graph (the two score networks as parallel branches):
    same states as eager launches (the instance-norm statistics are accumulated with double atomics, whose order may
    differ in the last bit, hence a 1e-6 bound instead of bit equality)."""
    from audiosourcesep_b200 import ops, _lib
    cfg = _cfg(version)
    m1, sig = _model(cfg, init_ncsn_params(cfg, seed=5, mode="perturbed"))
    m2, _ = _model(cfg, init_ncsn_params(cfg, seed=6, mode="perturbed"))
    mixed, _, _ = synthetic.basis_problem(3)
    x1, x2 = synthetic.langevin_init(3, seed=4)
    T = 4
    outs = []
    try:
        for graphs in (False, True):
            _lib.basis_graphs(graphs)
            t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
            dump = torch.zeros((T, 2, 3, 96, 64, 1), device="cuda")
            for call, level in enumerate((cfg.num_classes - 3, cfg.num_classes - 1)):
                eta, lam, ns = bo.step_constants(sig, level)
                ops.basis_ncsn_inner(m1, m2, torch.as_tensor(mixed), t1, t2, level, T, float(eta), float(lam), float(ns),
                                     seed=11, step0=call * T, per_step=dump)      # same key twice: the second call replays the cached graph from its first step
            outs.append((t1.clone(), t2.clone(), dump.clone()))
    finally:
        _lib.basis_graphs(True)
    for k in range(3):
        a, b = _np(outs[0][k]), _np(outs[1][k])
        assert np.linalg.norm(a - b) <= 1e-6 * np.linalg.norm(a), k
    assert not torch.equal(outs[1][0], torch.as_tensor(x1).cuda())
