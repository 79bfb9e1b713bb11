"""GPU parity tests of the fused Langevin update and the BASIS inner loop vs the oracle."""
import numpy as np
import pytest
import torch

from audiosourcesep_b200 import GlowConfig, synthetic
from audiosourcesep_b200.weights import init_glow_params
from oracle import basis_oracle as bo
from oracle.glow_oracle import GlowOracle

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def test_mixing_db_matches_oracle():
    from audiosourcesep_b200 import ops
    g, grad_g = bo.mixing_process("melspec", "dB")
    rng = np.random.default_rng(0)
    a = rng.uniform(-0.5, 1.5, (3, 8, 4, 1)).astype(np.float32)
    b = rng.uniform(-0.5, 1.5, (3, 8, 4, 1)).astype(np.float32)
    gg, w1, w2 = ops.mixing_db(torch.as_tensor(a), torch.as_tensor(b))
    ga, gb = grad_g(a, b)
    np.testing.assert_allclose(_np(gg), g(a, b), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(_np(w1), ga, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(_np(w2), gb, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("sigma_idx", [0, 4, 9])
def test_langevin_step_matches_oracle_with_injected_noise(sigma_idx):
    from audiosourcesep_b200 import ops
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, sigma_idx)
    g, grad_g = bo.mixing_process("melspec", "dB")
    rng = np.random.default_rng(sigma_idx)
    shp = (4, 96, 64, 1)
    x1, x2, mixed = (rng.uniform(0, 1, shp).astype(np.float32) for _ in range(3))
    s1, s2, n1, n2 = (rng.standard_normal(shp).astype(np.float32) for _ in range(4))
    y1, y2 = bo.langevin_update(x1, x2, s1, s2, mixed, n1, n2, eta, lam, ns, g, grad_g)
    t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.langevin_step(t1, t2, torch.as_tensor(s1), torch.as_tensor(s2), torch.as_tensor(mixed), float(eta), float(lam),
                      float(ns), n1=torch.as_tensor(n1), n2=torch.as_tensor(n2), nan_count=nan)
    for got, want in ((t1, y1), (t2, y2)):
        rel = np.linalg.norm(_np(got) - want) / np.linalg.norm(want)
        assert rel <= 1e-5, rel                      # gate: per-step state relative error <= 1e-3
    assert nan.item() == 0
    # NaN flag (the reference's --debug asserts, run_basis_sep.py:183-191)
    bad = torch.full(shp, float("nan"), device="cuda")
    ops.langevin_step(t1, t2, bad, torch.as_tensor(s2), torch.as_tensor(mixed), float(eta), float(lam), float(ns),
                      n1=torch.as_tensor(n1), n2=torch.as_tensor(n2), nan_count=nan)
    assert nan.item() > 0


def test_philox_noise_is_standard_normal_and_shard_invariant():
    from audiosourcesep_b200 import ops
    n = 30 * 6144
    full = ops.philox_normal((n,), seed=7, step=3, stream_id=1)
    v = _np(full).astype(np.float64)
    assert abs(v.mean()) < 0.01 and abs(v.std() - 1.0) < 0.01
    assert abs(((v - v.mean()) ** 3).mean()) < 0.03 and abs((v ** 4).mean() - 3.0) < 0.08
    # sharding segments over ranks gives the same draws (elem_offset = global index of the shard)
    half = n // 2
    lo = ops.philox_normal((half,), seed=7, step=3, stream_id=1, elem_offset=0)
    hi = ops.philox_normal((n - half,), seed=7, step=3, stream_id=1, elem_offset=half)
    assert torch.equal(torch.cat([lo, hi]), full)
    other = ops.philox_normal((n,), seed=7, step=4, stream_id=1)
    assert abs(np.corrcoef(v, _np(other))[0, 1]) < 0.01
    assert not torch.equal(ops.philox_normal((n,), seed=7, step=3, stream_id=2), full)


@pytest.mark.parametrize("weights,sigma_idx", [("faithful", 0), ("faithful", 9), ("perturbed", 6), ("perturbed", 9)])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_basis_glow_inner_loop_vs_oracle(precision, weights, sigma_idx):
    """Langevin steps with two Glow priors and injected noise.  Gate: per-step state relative error
    <= 1e-3 (each CUDA step starts from the oracle's previous state); the free-running drift over the
    T steps is reported and loosely bounded.

    ``faithful`` = the reference's random init (zero conv3, ActNorm initialised from a minibatch) at the
    largest and smallest step size; ``perturbed`` = non-trivial couplings.  With perturbed random weights
    and the largest step sizes (eta = 0.2) one update moves the state by more than its own norm and the
    piecewise-constant ReLU gradient makes ANY two arithmetics diverge (fp32 vs fp64 already differ by
    5e-4 per step there), so the perturbed cases use the annealed end of the schedule."""
    from audiosourcesep_b200 import ops, _lib
    from audiosourcesep_b200.glow import Glow
    # BASIS states are normalised [0,1]: SpecPreprocessing(minval=0, maxval=1) (SURVEY.md App. B)
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=3, n_filters=512, minval=0.0, maxval=1.0)
    prec = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}[precision]
    p1, p2 = init_glow_params(cfg, seed=2, mode=weights), init_glow_params(cfg, seed=3, mode=weights)
    if weights == "faithful":
        p1.update(GlowOracle(cfg, p1).init_actnorm(synthetic.normalise(synthetic.mel_patches_db(8, seed=9))))
        p2.update(GlowOracle(cfg, p2).init_actnorm(synthetic.normalise(synthetic.mel_patches_db(8, seed=10))))
    o1, o2 = GlowOracle(cfg, p1), GlowOracle(cfg, p2)
    m1, m2 = Glow(cfg, p1, precision=prec), Glow(cfg, p2, precision=prec)
    n_mixed = 3
    T = 1 if (weights == "faithful" and sigma_idx == 0) else 3   # eta = 0.2 on an untrained Gaussian score diverges within 2 steps
    mixed, _, _ = synthetic.basis_problem(n_mixed)
    x1, x2 = synthetic.langevin_init(n_mixed, seed=4)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, sigma_idx)
    rng = np.random.default_rng(3)
    noise = rng.standard_normal((T, 2, n_mixed, 96, 64, 1)).astype(np.float32)
    g, grad_g = bo.mixing_process("melspec", "dB")
    a, b = x1.copy(), x2.copy()
    states = [(a.copy(), b.copy())]
    for t in range(T):
        s1 = o1.grad_log_prob(a)[0].numpy().astype(np.float32)
        s2 = o2.grad_log_prob(b)[0].numpy().astype(np.float32)
        a, b = bo.langevin_update(a, b, s1, s2, mixed, noise[t, 0], noise[t, 1], eta, lam, ns, g, grad_g)
        states.append((a.copy(), b.copy()))
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    worst = 0.0
    for t in range(T):     # synchronised: one CUDA step from the oracle's state
        t1, t2 = torch.as_tensor(states[t][0]).cuda(), torch.as_tensor(states[t][1]).cuda()
        ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), t1, t2, 1, float(eta), float(lam), float(ns),
                             noise1=torch.as_tensor(noise[t:t + 1, 0]), noise2=torch.as_tensor(noise[t:t + 1, 1]),
                             nan_count=nan)
        for got, want in ((t1, states[t + 1][0]), (t2, states[t + 1][1])):
            rel = float(np.linalg.norm(_np(got) - want) / np.linalg.norm(want))
            worst = max(worst, rel)
    print(f"[{precision}, {weights}, sigma_idx={sigma_idx}] worst per-step state relative error = {worst:.3e}")
    assert worst <= 1e-3, worst
    assert nan.item() == 0
    nan.zero_()
    # free-running T steps inside the library, with the per-step dump
    t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
    dump = torch.empty((T, 2, n_mixed, 96, 64, 1), device="cuda")
    ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), t1, t2, T, float(eta), float(lam), float(ns),
                         noise1=torch.as_tensor(noise[:, 0]), noise2=torch.as_tensor(noise[:, 1]),
                         per_step=dump, nan_count=nan)
    drift = max(float(np.linalg.norm(_np(dump[T - 1, k]) - states[T][k]) / np.linalg.norm(states[T][k])) for k in range(2))
    print(f"[{precision}, {weights}, sigma_idx={sigma_idx}] free-running drift after {T} steps = {drift:.3e}")
    if not (weights == "faithful" and sigma_idx == 0):   # eta = 0.2 on an untrained linear-Gaussian score is an unstable iteration
        assert drift <= 5e-3
    assert torch.equal(dump[T - 1, 0], t1) and torch.equal(dump[T - 1, 1], t2)


def test_same_prior_for_both_sources_keeps_two_score_tensors():
    """model1 and model2 are just callables in the reference (run_basis_sep.py:166-175): passing ONE handle for both
    sources must give the same result as two handles holding the same weights."""
    from audiosourcesep_b200 import ops, _lib
    from audiosourcesep_b200.glow import Glow
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=2, n_filters=512, minval=0.0, maxval=1.0)
    p = init_glow_params(cfg, seed=2, mode="perturbed")
    ma, mb = Glow(cfg, p, precision=_lib.PREC_BF16), Glow(cfg, p, precision=_lib.PREC_BF16)
    mixed, _, _ = synthetic.basis_problem(3)
    x1, x2 = synthetic.langevin_init(3, seed=4)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 8)
    outs = []
    for m1, m2 in ((ma, mb), (ma, ma)):
        t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
        ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), t1, t2, 2, float(eta), float(lam), float(ns), seed=3)
        outs.append((t1.clone(), t2.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert not torch.equal(outs[1][0], torch.as_tensor(x1).cuda())


def test_device_sigma_loop_equals_the_host_loop():
    """ops.basis_run (the whole sigma x T loop inside the library, run_basis_sep.py:217-260) gives bit-identical
    states and per-level snapshots to one ops.basis_glow_inner call per noise level."""
    from audiosourcesep_b200 import ops, _lib
    from audiosourcesep_b200.glow import Glow
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=2, n_filters=512, minval=0.0, maxval=1.0)
    m1 = Glow(cfg, init_glow_params(cfg, seed=2, mode="perturbed"), precision=_lib.PREC_BF16)
    m2 = Glow(cfg, init_glow_params(cfg, seed=3, mode="perturbed"), precision=_lib.PREC_BF16)
    mixed, _, _ = synthetic.basis_problem(3)
    x1, x2 = synthetic.langevin_init(3, seed=4)
    sig = bo.get_sigmas(0.05, 0.01, 4, "logarithmic")
    T = 2
    consts = [bo.step_constants(sig, i) for i in range(len(sig))]
    a1, a2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
    host_snaps = []
    for i, (eta, lam, ns) in enumerate(consts):
        ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), a1, a2, T, float(eta), float(lam), float(ns), seed=9, step0=i * T)
        host_snaps.append((a1.clone(), a2.clone()))
    b1, b2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
    snaps = torch.empty((len(sig), 2) + tuple(b1.shape), device="cuda")
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.basis_run(m1, m2, torch.as_tensor(mixed), b1, b2, T, [c[0] for c in consts], [c[1] for c in consts],
                  [c[2] for c in consts], seed=9, snapshots=snaps, nan_count=nan)
    assert torch.equal(a1, b1) and torch.equal(a2, b2) and nan.item() == 0
    for i, (s1, s2) in enumerate(host_snaps):
        assert torch.equal(snaps[i, 0], s1) and torch.equal(snaps[i, 1], s2)
    # one pair of priors per noise level (the per-sigma fine-tuned models of run_basis_sep.py:228-234), all resident
    c1, c2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
    ops.basis_run([m1] * len(sig), [m2] * len(sig), torch.as_tensor(mixed), c1, c2, T, [c[0] for c in consts],
                  [c[1] for c in consts], [c[2] for c in consts], seed=9)
    assert torch.equal(c1, a1) and torch.equal(c2, a2)



@pytest.mark.parametrize("same_handle", [False, True])
def test_glow_step_graph_replay_equals_eager_launches(same_handle):
    """Steps 2..T of ops.basis_glow_inner are replays of ONE captured CUDA graph (both scores as parallel branches when
    the priors are two handles, per-step scalars in device memory): states and the per-step dump must equal those of
    eager launches, for in-kernel Philox noise and across two consecutive calls that reuse the cached graph."""
    from audiosourcesep_b200 import ops, _lib
    from audiosourcesep_b200.glow import Glow
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=2, n_filters=512, minval=0.0, maxval=1.0)
    m1 = Glow(cfg, init_glow_params(cfg, seed=2, mode="perturbed"), precision=_lib.PREC_BF16)
    m2 = m1 if same_handle else Glow(cfg, init_glow_params(cfg, seed=3, mode="perturbed"), precision=_lib.PREC_BF16)
    mixed, _, _ = synthetic.basis_problem(3)
    x1, x2 = synthetic.langevin_init(3, seed=4)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    T = 5
    outs = []
    try:
        for graphs in (False, True):
            _lib.basis_graphs(graphs)
            t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
            dump = torch.zeros((T, 2, 3, 96, 64, 1), device="cuda")
            n0 = _lib.launch_count()
            for call, level in enumerate((7, 9)):          # second call: other step constants, same cached graph
                eta, lam, ns = bo.step_constants(sig, level)
                ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), t1, t2, T, float(eta), float(lam), float(ns), seed=11,
                                     step0=call * T, per_step=dump)      # same key twice: the second call replays the cached graph from its first step
            outs.append((t1.clone(), t2.clone(), dump.clone(), _lib.launch_count() - n0))
    finally:
        _lib.basis_graphs(True)
    for k in range(3):
        assert torch.equal(outs[0][k], outs[1][k]), k
    assert outs[0][3] > 0 and abs(outs[1][3] - outs[0][3]) <= 0.05 * outs[0][3]   # replayed launches are counted like eager ones
    assert not torch.equal(outs[1][0], torch.as_tensor(x1).cuda())
