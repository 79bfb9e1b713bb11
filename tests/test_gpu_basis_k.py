"""GPU tests of BASIS with K sources: the K-source fused update, the K-source step runner and graphs, the stacked C ABI,
and run_basis_sep / melspec_inversion_basis with three sources."""
import os
import wave

import numpy as np
import pytest
import torch

from audiosourcesep_b200 import GlowConfig, NCSNConfig, synthetic
from audiosourcesep_b200.weights import init_glow_params, init_ncsn_params
from oracle import basis_k_oracle as bko
from oracle import basis_oracle as bo
from oracle.glow_oracle import GlowOracle

pytestmark = pytest.mark.gpu

SHP = (3, 96, 64, 1)


def _np(t):
    return t.detach().cpu().numpy()


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


def _glow_cfg(K=2):
    return GlowConfig(H=96, W=64, C=1, L=3, K=K, n_filters=512, minval=0.0, maxval=1.0)


def _glows(n, precision, K=2, mode="perturbed"):
    from audiosourcesep_b200.glow import Glow
    cfg = _glow_cfg(K)
    return [Glow(cfg, init_glow_params(cfg, seed=2 + k, mode=mode), precision=precision) for k in range(n)]


def _ncsn_v2(n, precision, seeds=(11, 12, 13)):
    from audiosourcesep_b200.ncsn.score_model import ScoreModel
    cfg = NCSNConfig(version="v2", ngf=128, num_classes=200, sigma1=30.0, sigmaL=0.01)
    sig = bo.get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, cfg.progression)
    params = [init_ncsn_params(cfg, seed=seeds[k], mode="perturbed") for k in range(n)]
    return cfg, sig, params, [ScoreModel(cfg, p, sigmas=sig, precision=precision) for p in params]


def _problem(K, n=3):
    rng = np.random.default_rng(K)
    xs = np.stack([rng.uniform(0, 1, (n, 96, 64, 1)).astype(np.float32) for _ in range(K)])
    gts = [synthetic.mel_patches_db(n, k) for k in range(K)]
    return synthetic.normalise(synthetic.mixture_db(*gts)), xs


@pytest.mark.parametrize("K", [2, 3, 5])
def test_mixing_db_k_matches_oracle(K):
    from audiosourcesep_b200 import ops
    g, grad_g = bo.mixing_process("melspec", "dB")
    rng = np.random.default_rng(K)
    x = rng.uniform(-0.5, 1.5, (K, 3, 8, 4, 1)).astype(np.float32)
    gg, w = ops.mixing_db_k(torch.as_tensor(x))
    np.testing.assert_allclose(_np(gg), g(*x), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(_np(w), np.stack(grad_g(*x)), rtol=1e-5, atol=1e-6)
    if K == 2:
        g2, w1, w2 = ops.mixing_db(torch.as_tensor(x[0]), torch.as_tensor(x[1]))
        assert torch.equal(gg, g2) and torch.equal(w[0], w1) and torch.equal(w[1], w2)


@pytest.mark.parametrize("K", [3, 8])
def test_langevin_step_k_matches_oracle_with_injected_noise(K):
    from audiosourcesep_b200 import ops
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 6)
    g, grad_g = bo.mixing_process("melspec", "dB")
    rng = np.random.default_rng(K)
    x = rng.uniform(0, 1, (K,) + SHP).astype(np.float32)
    mixed = rng.uniform(0, 1, SHP).astype(np.float32)
    s, z = (rng.standard_normal((K,) + SHP).astype(np.float32) for _ in range(2))
    want = bko.langevin_update_k(list(x), list(s), mixed, list(z), eta, lam, ns, g, grad_g)
    t = torch.as_tensor(x).cuda()
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.langevin_step_k(t, torch.as_tensor(s), torch.as_tensor(mixed), float(eta), float(lam), float(ns),
                        noise=torch.as_tensor(z), nan_count=nan)
    for k in range(K):
        assert _rel(_np(t[k]), want[k]) <= 1e-5, k
    assert nan.item() == 0
    bad = torch.as_tensor(s).cuda()
    bad[K - 1, 0, 0, 0, 0] = float("nan")                # any source sets the flag
    ops.langevin_step_k(t, bad, torch.as_tensor(mixed), float(eta), float(lam), float(ns), noise=torch.as_tensor(z),
                        nan_count=nan)
    assert nan.item() > 0


@pytest.mark.parametrize("injected", [True, False])
def test_langevin_step_k2_is_bitwise_the_two_source_step(injected):
    from audiosourcesep_b200 import ops
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 3)
    rng = np.random.default_rng(1)
    x = rng.uniform(0, 1, (2,) + SHP).astype(np.float32)
    mixed = rng.uniform(0, 1, SHP).astype(np.float32)
    s, z = (torch.as_tensor(rng.standard_normal((2,) + SHP).astype(np.float32)).cuda() for _ in range(2))
    a1, a2 = torch.as_tensor(x[0]).cuda(), torch.as_tensor(x[1]).cuda()
    ops.langevin_step(a1, a2, s[0], s[1], torch.as_tensor(mixed), float(eta), float(lam), float(ns),
                      n1=z[0] if injected else None, n2=z[1] if injected else None, seed=7, step=12, elem_offset=4096)
    b = torch.as_tensor(x).cuda()
    ops.langevin_step_k(b, s, torch.as_tensor(mixed), float(eta), float(lam), float(ns), noise=z if injected else None,
                        seed=7, step=12, elem_offset=4096)
    assert torch.equal(b[0], a1) and torch.equal(b[1], a2)


def test_philox_stream_of_source_k_is_stream_k_plus_1():
    from audiosourcesep_b200 import ops
    K = 5
    x = torch.zeros((K,) + SHP, device="cuda")
    ops.langevin_step_k(x, torch.zeros_like(x), torch.zeros(SHP), 0.0, 0.0, 1.0, seed=3, step=17, elem_offset=8192)
    for k in range(K):
        assert torch.equal(x[k], ops.philox_normal(SHP, seed=3, step=17, stream_id=k + 1, elem_offset=8192)), k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_three_glow_priors_vs_oracle(precision):
    """Per-step parity of K = 3 Glow priors with injected noise (each CUDA step starts from the oracle's state), the
    free-running drift over T steps and the per-step dump, in the shape of the two-source test."""
    from audiosourcesep_b200 import ops, _lib
    K, T, n = 3, 3, 3
    prec = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}[precision]
    cfg = _glow_cfg(3)
    params = [init_glow_params(cfg, seed=2 + k, mode="perturbed") for k in range(K)]
    from audiosourcesep_b200.glow import Glow
    models = [Glow(cfg, p, precision=prec) for p in params]
    oracles = [GlowOracle(cfg, p) for p in params]
    mixed, x0 = _problem(K, n)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 9)
    noise = np.random.default_rng(3).standard_normal((T, K, n, 96, 64, 1)).astype(np.float32)
    g, grad_g = bo.mixing_process("melspec", "dB")
    states = [list(x0)]
    for t in range(T):
        ss = [o.grad_log_prob(x)[0].numpy().astype(np.float32) for o, x in zip(oracles, states[-1])]
        states.append(bko.langevin_update_k(states[-1], ss, mixed, list(noise[t]), eta, lam, ns, g, grad_g))
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    worst = 0.0
    for t in range(T):
        x = torch.as_tensor(np.stack(states[t])).cuda()
        ops.basis_glow_inner_k(models, torch.as_tensor(mixed), x, 1, float(eta), float(lam), float(ns),
                               noise=torch.as_tensor(noise[t:t + 1]), nan_count=nan)
        worst = max(worst, max(_rel(_np(x[k]), states[t + 1][k]) for k in range(K)))
    print(f"[{precision}] K = 3 worst per-step state relative error = {worst:.3e}")
    assert worst <= 1e-3 and nan.item() == 0
    x = torch.as_tensor(x0).cuda()
    dump = torch.empty((T, K, n, 96, 64, 1), device="cuda")
    ops.basis_glow_inner_k(models, torch.as_tensor(mixed), x, T, float(eta), float(lam), float(ns),
                           noise=torch.as_tensor(noise), per_step=dump, nan_count=nan)
    drift = max(_rel(_np(dump[T - 1, k]), states[T][k]) for k in range(K))
    print(f"[{precision}] K = 3 free-running drift after {T} steps = {drift:.3e}")
    assert drift <= 5e-3
    assert torch.equal(dump[T - 1], x)


def test_three_ncsn_v2_score_networks_vs_oracle():
    from audiosourcesep_b200 import ops, _lib
    from oracle.ncsn_oracle import NCSNOracle
    K, T, n, sigma_idx = 3, 2, 2, 120
    cfg, sig, params, models = _ncsn_v2(K, _lib.PREC_BF16X3)
    oracles = [NCSNOracle(cfg, p, sigmas=sig, dtype=torch.float32) for p in params]
    mixed, x0 = _problem(K, n)
    eta, lam, ns = bo.step_constants(sig, sigma_idx)
    noise = np.random.default_rng(3).standard_normal((T, K, n, 96, 64, 1)).astype(np.float32)
    g, grad_g = bo.mixing_process("melspec", "dB")
    idx = np.full((n,), sigma_idx, dtype=np.int64)
    states = [list(x0)]
    for t in range(T):
        ss = [o.score(x, idx).numpy().astype(np.float32) for o, x in zip(oracles, states[-1])]
        states.append(bko.langevin_update_k(states[-1], ss, mixed, list(noise[t]), eta, lam, ns, g, grad_g))
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    worst = 0.0
    for t in range(T):
        x = torch.as_tensor(np.stack(states[t])).cuda()
        ops.basis_ncsn_inner_k(models, torch.as_tensor(mixed), x, sigma_idx, 1, float(eta), float(lam), float(ns),
                               noise=torch.as_tensor(noise[t:t + 1]), nan_count=nan)
        worst = max(worst, max(_rel(_np(x[k]), states[t + 1][k]) for k in range(K)))
    print(f"NCSN v2 split-bf16, K = 3: worst per-step state relative error = {worst:.3e}")
    assert worst <= 1e-3 and nan.item() == 0


def test_k2_entry_points_are_bitwise_the_two_source_ones():
    from audiosourcesep_b200 import ops, _lib
    mixed, x0 = _problem(2)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 8)
    T = 4
    for models in (_glows(2, _lib.PREC_BF16), ):
        for pair in ((models[0], models[1]), (models[0], models[0])):
            a1, a2 = torch.as_tensor(x0[0]).cuda(), torch.as_tensor(x0[1]).cuda()
            d2 = torch.zeros((T, 2) + SHP, device="cuda")
            ops.basis_glow_inner(pair[0], pair[1], torch.as_tensor(mixed), a1, a2, T, float(eta), float(lam), float(ns),
                                 seed=5, step0=2, per_step=d2)
            b = torch.as_tensor(x0).cuda()
            dk = torch.zeros((T, 2) + SHP, device="cuda")
            ops.basis_glow_inner_k(list(pair), torch.as_tensor(mixed), b, T, float(eta), float(lam), float(ns), seed=5,
                                   step0=2, per_step=dk)
            assert torch.equal(b[0], a1) and torch.equal(b[1], a2) and torch.equal(dk, d2)
        L = 3
        consts = [bo.step_constants(sig, 7 + i) for i in range(L)]
        cs = [[c[j] for c in consts] for j in range(3)]
        a1, a2 = torch.as_tensor(x0[0]).cuda(), torch.as_tensor(x0[1]).cuda()
        s2 = torch.zeros((L, 2) + SHP, device="cuda")
        ops.basis_run(models[0], models[1], torch.as_tensor(mixed), a1, a2, 3, *cs, seed=4, snapshots=s2)
        b = torch.as_tensor(x0).cuda()
        sk = torch.zeros((L, 2) + SHP, device="cuda")
        ops.basis_run_k(models, torch.as_tensor(mixed), b, 3, *cs, seed=4, snapshots=sk)
        assert torch.equal(b[0], a1) and torch.equal(b[1], a2) and torch.equal(sk, s2)
    # score networks: the instance-norm statistics are accumulated with double atomics whose order may differ in the last
    # bit between two runs of the same entry point, so the bound is the one of the NCSN graph-replay test
    cfg, nsig, _, nets = _ncsn_v2(2, _lib.PREC_BF16X3)
    consts = [bo.step_constants(nsig, i) for i in range(3)]
    cs = [[c[j] for c in consts] for j in range(3)]
    a1, a2 = torch.as_tensor(x0[0]).cuda(), torch.as_tensor(x0[1]).cuda()
    s2 = torch.zeros((3, 2) + SHP, device="cuda")
    ops.basis_run(nets[0], nets[1], torch.as_tensor(mixed), a1, a2, 3, *cs, seed=4, snapshots=s2)
    b = torch.as_tensor(x0).cuda()
    sk = torch.zeros((3, 2) + SHP, device="cuda")
    ops.basis_run_k(nets, torch.as_tensor(mixed), b, 3, *cs, seed=4, snapshots=sk)
    assert _rel(_np(sk), _np(s2)) <= 1e-6 and _rel(_np(b[0]), _np(a1)) <= 1e-6 and _rel(_np(b[1]), _np(a2)) <= 1e-6
    e, l_, n_ = bo.step_constants(nsig, 150)
    a1, a2 = torch.as_tensor(x0[0]).cuda(), torch.as_tensor(x0[1]).cuda()
    d2 = torch.zeros((T, 2) + SHP, device="cuda")
    ops.basis_ncsn_inner(nets[0], nets[1], torch.as_tensor(mixed), a1, a2, 150, T, float(e), float(l_), float(n_), seed=5,
                         per_step=d2)
    b = torch.as_tensor(x0).cuda()
    dk = torch.zeros((T, 2) + SHP, device="cuda")
    ops.basis_ncsn_inner_k(nets, torch.as_tensor(mixed), b, 150, T, float(e), float(l_), float(n_), seed=5, per_step=dk)
    assert _rel(_np(dk), _np(d2)) <= 1e-6


def test_device_sigma_loop_k_equals_one_inner_call_per_level():
    from audiosourcesep_b200 import ops, _lib
    K = 3
    models = _glows(K, _lib.PREC_BF16)
    mixed, x0 = _problem(K)
    sig = bo.get_sigmas(0.05, 0.01, 4, "logarithmic")
    T = 2
    consts = [bo.step_constants(sig, i) for i in range(len(sig))]
    cs = [[c[j] for c in consts] for j in range(3)]
    a = torch.as_tensor(x0).cuda()
    host = []
    for i, (eta, lam, ns) in enumerate(consts):
        ops.basis_glow_inner_k(models, torch.as_tensor(mixed), a, T, float(eta), float(lam), float(ns), seed=9, step0=i * T)
        host.append(a.clone())
    b = torch.as_tensor(x0).cuda()
    snaps = torch.empty((len(sig),) + tuple(b.shape), device="cuda")
    nan = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.basis_run_k(models, torch.as_tensor(mixed), b, T, *cs, seed=9, snapshots=snaps, nan_count=nan)
    assert torch.equal(a, b) and nan.item() == 0
    for i, h in enumerate(host):
        assert torch.equal(snaps[i], h)
    c = torch.as_tensor(x0).cuda()                       # one set of K priors per noise level, all resident
    ops.basis_run_k([models] * len(sig), torch.as_tensor(mixed), c, T, *cs, seed=9)
    assert torch.equal(c, a)


@pytest.mark.parametrize("handles", ["abc", "aab"])
def test_k3_step_graph_replay_equals_eager_launches(handles):
    from audiosourcesep_b200 import ops, _lib
    pool = _glows(2 if handles == "aab" else 3, _lib.PREC_BF16)
    models = [pool[0], pool[0], pool[1]] if handles == "aab" else pool
    mixed, x0 = _problem(3)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    T = 5
    outs = []
    try:
        for graphs in (False, True):
            _lib.basis_graphs(graphs)
            x = torch.as_tensor(x0).cuda()
            dump = torch.zeros((T, 3) + SHP, device="cuda")
            n0 = _lib.launch_count()
            for call, level in enumerate((7, 9)):          # second call: other step constants, same cached graph
                eta, lam, ns = bo.step_constants(sig, level)
                ops.basis_glow_inner_k(models, torch.as_tensor(mixed), x, T, float(eta), float(lam), float(ns), seed=11,
                                       step0=call * T, per_step=dump)
            outs.append((x.clone(), dump.clone(), _lib.launch_count() - n0))
    finally:
        _lib.basis_graphs(True)
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert outs[0][2] > 0 and abs(outs[1][2] - outs[0][2]) <= 0.05 * outs[0][2]
    assert not torch.equal(outs[1][0], torch.as_tensor(x0).cuda())


def test_k3_shards_equal_one_call():
    from audiosourcesep_b200 import ops, _lib
    models = _glows(3, _lib.PREC_BF16)
    mixed, x0 = _problem(3)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 8)
    full = torch.as_tensor(x0).cuda()
    ops.basis_glow_inner_k(models, torch.as_tensor(mixed), full, 3, float(eta), float(lam), float(ns), seed=2, step0=6)
    seg = 96 * 64
    parts = []
    for lo, hi in ((0, 1), (1, 3)):
        x = torch.as_tensor(np.ascontiguousarray(x0[:, lo:hi])).cuda()
        ops.basis_glow_inner_k(models, torch.as_tensor(mixed[lo:hi]), x, 3, float(eta), float(lam), float(ns), seed=2,
                               step0=6, elem_offset=lo * seg)
        parts.append(x)
    assert torch.equal(torch.cat(parts, 1), full)


def test_bad_arguments_raise_before_any_launch():
    from audiosourcesep_b200 import ops, _lib
    models = _glows(3, _lib.PREC_BF16)
    mixed, x0 = _problem(3)
    mx = torch.as_tensor(mixed)

    def rejects(fn, error=_lib.AsepError):
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        with pytest.raises(error):
            fn()
        assert _lib.launch_count() == n0

    x = torch.as_tensor(x0).cuda()
    rejects(lambda: ops.basis_glow_inner_k(models[:1], mx, x[:1].contiguous(), 2, 1e-5, 1.0, 1e-3))
    rejects(lambda: ops.basis_glow_inner_k([models[0]] * 9, mx, torch.zeros((9,) + SHP, device="cuda"), 2, 1e-5, 1.0, 1e-3))
    rejects(lambda: ops.basis_glow_inner_k(models, mx[:2], x, 2, 1e-5, 1.0, 1e-3))
    rejects(lambda: ops.basis_glow_inner_k(models, mx, x, 2, 1e-5, 1.0, 1e-3, noise=torch.zeros((2, 2) + SHP)))
    rejects(lambda: ops.basis_glow_inner_k(models, mx, x, 2, 1e-5, 1.0, 1e-3,
                                           per_step=torch.zeros((3, 3) + SHP, device="cuda")))
    rejects(lambda: ops.langevin_step_k(torch.zeros((9,) + SHP, device="cuda"), torch.zeros((9,) + SHP), mx, 0.0, 0.0, 1.0))
    rejects(lambda: ops.langevin_step_k(x[:1].contiguous(), torch.zeros((1,) + SHP), mx, 0.0, 0.0, 1.0))
    rejects(lambda: ops.mixing_db_k(torch.zeros((9, 4))))
    rejects(lambda: ops.basis_run_k(models, mx, x, 2, [1e-5], [1.0], [1e-3], snapshots=torch.zeros((2, 3) + SHP, device="cuda")))
    # the two-source calls: one injected noise tensor without the other, or states of different shapes
    a, b, s = x[0].clone(), x[1].clone(), torch.zeros(SHP, device="cuda")
    noise = torch.zeros((2,) + SHP, device="cuda")
    rejects(lambda: ops.langevin_step(a, b, s, s, mx, 0.0, 0.0, 1.0, n1=s), ValueError)
    rejects(lambda: ops.basis_glow_inner(models[0], models[1], mx, a, b, 2, 1e-5, 1.0, 1e-3, noise2=noise), ValueError)
    rejects(lambda: ops.langevin_step(a, b[:2].contiguous(), s, s, mx, 0.0, 0.0, 1.0), ValueError)
    rejects(lambda: ops.basis_run(models[0], models[1], mx, a[:2].contiguous(), b, 2, [1e-5], [1.0], [1e-3]), ValueError)


def test_run_basis_sep_glow_k3_cli_and_sdr(tmp_path):
    from audiosourcesep_b200 import ops
    from audiosourcesep_b200.run_basis_sep import build_parser, main
    out = tmp_path / "sep3"
    n_mixed, T, L, K = 2, 3, 3, 3
    argv = ["u1", "u2", "u3", "--output", str(out), "--model_type", "glow", "--synthetic", "--random_init", "7",
            "--n_mixed", str(n_mixed), "--T", str(T), "--K", "2", "--L", "3", "--n_filters", "512", "--learntop",
            "--sigma1", "0.05", "--sigmaL", "0.01", "--num_classes", str(L), "--progression", "logarithmic", "--seed", "5"]
    main(build_parser().parse_args(argv))
    z = np.load(out / "results.npz")
    assert sorted(z.files) == ["gt1", "gt2", "gt3", "mixed", "stft_mixture", "x1", "x2", "x3"]
    zc = np.load(out / "results_convergence.npz")
    assert sorted(zc.files) == ["x1", "x2", "x3"]
    assert all(zc[k].shape == (L + 1, n_mixed, 96, 64, 1) for k in zc.files)
    log = (out / "out.log").read_text()
    assert log.count("Sigma = ") == L and "Duration: " in log and "Data Loaded in" in log
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=2, n_filters=512, learntop=True, minval=0.0, maxval=1.0)
    oracles = [GlowOracle(cfg, init_glow_params(cfg, seed=7 + k, mode="perturbed")) for k in range(K)]
    sig = bo.get_sigmas(0.05, 0.01, L, "logarithmic")
    gts = [synthetic.mel_patches_db(n_mixed, k) for k in range(K)]
    mixed = synthetic.normalise(synthetic.mixture_db(*gts))
    rng = np.random.Generator(np.random.PCG64(5))
    xs = [rng.uniform(0.0, 1.0, mixed.shape).astype(np.float32) for _ in range(K)]

    def noise(i, t):
        return [ops.philox_normal(mixed.shape, seed=5, step=i * T + t, stream_id=k + 1).cpu().numpy() for k in range(K)]

    scores = [(lambda o: (lambda x, i: o.grad_log_prob(x)[0].numpy().astype(np.float32)))(o) for o in oracles]
    ys, _ = bko.basis_run_k(mixed, xs, scores, sig, T, noise)
    for k in range(K):
        assert np.array_equal(z[f"gt{k + 1}"], gts[k].squeeze(-1))
        gt = synthetic.normalise(gts[k].squeeze(-1))
        sdr_cuda = bo.sdr_db(gt, synthetic.normalise(z[f"x{k + 1}"]))
        sdr_orac = bo.sdr_db(gt, synthetic.normalise(bo.post_processing(ys[k].squeeze(-1))))
        print(f"source {k + 1}: mel-domain SDR cuda {sdr_cuda:.3f} dB, oracle {sdr_orac:.3f} dB")
        assert abs(sdr_cuda - sdr_orac) <= 0.1


def test_three_stem_wav_directory_to_separated_wav_files(tmp_path):
    from audiosourcesep_b200 import melspec_inversion_basis as inv
    from audiosourcesep_b200.run_basis_sep import build_parser, main, merge_config
    from oracle import mel_oracle as mo
    sr, L, n_win = 16000, 32640, 4
    rng = np.random.default_rng(0)
    t = np.arange(L * n_win) / sr
    stems = {"a": 0.25 * np.sin(2 * np.pi * 220 * t) + 0.002 * rng.standard_normal(t.size),
             "b": 0.2 * np.sin(2 * np.pi * 660 * t + 0.3 * np.sin(2 * np.pi * 5 * t)) + 0.002 * rng.standard_normal(t.size),
             "c": 0.2 * np.sin(2 * np.pi * 1500 * t) * (1 + 0.5 * np.sin(2 * np.pi * 3 * t)) + 0.002 * rng.standard_normal(t.size)}
    mix = stems["a"] + stems["b"] + stems["c"]
    song = tmp_path / "song"
    song.mkdir()
    for name, a in list(stems.items()) + [("mix", mix)]:
        with wave.open(str(song / f"{name}.wav"), "wb") as w:
            w.setnchannels(1); w.setsampwidth(2); w.setframerate(sr)
            w.writeframes((np.clip(a, -1, 1 - 1 / 32768) * 32768).astype("<i2").tobytes())
    out = tmp_path / "sep"
    cfg_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs", "melspec_ncsnv2.yml")
    args = merge_config(build_parser().parse_args(["u1", "u2", "u3", "--output", str(out), "--model_type", "ncsn",
                                                   "--song_dir", str(song), "--sources", "a,b,c", "--random_init", "3",
                                                   "--n_mixed", "2", "--config", cfg_path]))
    args.config = None
    args.T, args.num_classes, args.sigma1 = 1, 2, 0.05
    main(args)
    z = np.load(out / "results.npz")
    assert sorted(z.files) == ["gt1", "gt2", "gt3", "mixed", "stft_mixture", "x1", "x2", "x3"]
    pcm = (np.clip(mix, -1, 1 - 1 / 32768) * 32768).astype("<i2").astype(np.float32) / 32768.0
    want, _ = mo.melspectrogram_db(pcm[2 * L: 3 * L])
    assert np.max(np.abs(z["mixed"][0] - want)) <= 2e-3
    flat = inv.main(inv.build_parser().parse_args([str(out), "--wiener_filter"]))
    d = out / "inverse_reuse_phase_frame_wiener_filter"
    assert all(os.path.exists(d / f"sep{k}.wav") for k in (1, 2, 3))
    assert sorted(flat) == sorted([f"x{k}_audio" for k in (1, 2, 3)] + [f"gt{k}_audio" for k in (1, 2, 3)] + ["mix_audio"])
    n = 512 * 63
    ref = np.concatenate([stems["c"][2 * L: 2 * L + n], stems["c"][3 * L: 3 * L + n]])
    sdr = 10 * np.log10(np.sum(ref ** 2) / np.sum((flat["gt3_audio"] - ref) ** 2))
    print(f"inversion of the ground-truth third stem: SDR {sdr:.1f} dB")
    assert sdr > 8.0
