"""Oracle outputs of the FULL-DEPTH Glow-BASIS configuration, computed once on the CPU and committed.

The configuration is the one every reference config uses (configs/melspec_noisy_glow.yml: L=3, K=40, 512 filters,
96x64 patches) at the reference's n_mixed = 30 segments (run_basis_sep.py:478).  At this size one oracle
grad_log_prob takes ~10 s per pair of patches in float64, and a T=100 Langevin trajectory 200 evaluations, so the
GPU tests compare against these committed vectors instead of re-running the oracle on the GPU box.  Inputs are
NOT stored: the tests regenerate them from the same seeded generators (audiosourcesep_b200.synthetic,
weights.init_glow_params), so a drift of either generator fails the test loudly.

    python tests/golden/make_glow_k40_golden.py            (CPU, ~45 min on 8 cores)

Writes tests/golden/glow_k40.npz, a fixed sample of the oracle outputs that keeps the file under 1 MB:
  keep          uint8 packbits of a bool [30,96,64] mask: a seeded half of the score elements (every patch, row
                and column is represented)
  grad1, grad2  float32 [keep.sum()] oracle (float64) grad_log_prob of prior 1 at x1 / prior 2 at x2, at the
                                      elements of ``keep`` in C order
  logp1, logp2  float64 [30]         oracle (float64) log_prob
  traj_steps    int64 [2]            50, 100
  traj_x1, traj_x2  float32 [2,2,96,64]  oracle (float32, "as-TF") Langevin states of the first 2 segments at the
                                      LAST noise level (sigma index 9) after ``traj_steps`` steps with injected noise
                                      (run_basis_sep.py:152-181)
Seeds: weights 2 / 3 (mode "perturbed"), problem seeds 0 / 1, Langevin init 4, noise Generator(PCG64(3)),
score sample Generator(PCG64(0)).
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from audiosourcesep_b200 import GlowConfig, synthetic  # noqa: E402
from audiosourcesep_b200.weights import init_glow_params  # noqa: E402
from oracle import basis_oracle as bo  # noqa: E402
from oracle.glow_oracle import GlowOracle  # noqa: E402

N_MIXED, T, N_TRAJ = 30, 100, 2


def problem():
    cfg = GlowConfig(H=96, W=64, C=1, L=3, K=40, n_filters=512, minval=0.0, maxval=1.0)
    p1, p2 = init_glow_params(cfg, seed=2, mode="perturbed"), init_glow_params(cfg, seed=3, mode="perturbed")
    mixed, gt1, gt2 = synthetic.basis_problem(N_MIXED)
    x1, x2 = synthetic.langevin_init(N_MIXED, seed=4)
    return cfg, p1, p2, mixed, gt1, gt2, x1, x2


def traj_noise():
    rng = np.random.Generator(np.random.PCG64(3))
    return rng.standard_normal((T, 2, N_TRAJ, 96, 64, 1)).astype(np.float32)


def sample(full):
    """The stored subset of the full outputs: half of the score elements, the trajectory after 50 and 100 steps."""
    keep = np.random.Generator(np.random.PCG64(0)).random(full["grad1"].shape) < 0.5
    steps = np.array([50, 100])
    return {"keep": np.packbits(keep), "grad1": full["grad1"][keep], "grad2": full["grad2"][keep],
            "logp1": full["logp1"], "logp2": full["logp2"], "traj_steps": steps,
            "traj_x1": full["traj_x1"][steps // 10], "traj_x2": full["traj_x2"][steps // 10]}


def main():
    cfg, p1, p2, mixed, gt1, gt2, x1, x2 = problem()
    out = {}
    t0 = time.time()
    for k, (p, x) in enumerate(((p1, x1), (p2, x2)), start=1):
        o = GlowOracle(cfg, p, dtype=torch.float64)
        gs, lps = [], []
        for i in range(0, N_MIXED, 2):
            g, lp = o.grad_log_prob(x[i:i + 2])
            gs.append(g.numpy().astype(np.float32)[..., 0])
            lps.append(lp.numpy())
            print(f"prior {k}: patches {i}..{i + 1} done, {time.time() - t0:.0f} s", flush=True)
        out[f"grad{k}"] = np.concatenate(gs)
        out[f"logp{k}"] = np.concatenate(lps)
    # T = 100 steps at the last noise level, float32 oracle (the arithmetic TensorFlow would use)
    o1, o2 = GlowOracle(cfg, p1, dtype=torch.float32), GlowOracle(cfg, p2, dtype=torch.float32)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    eta, lam, ns = bo.step_constants(sig, 9)
    g, grad_g = bo.mixing_process("melspec", "dB")
    noise = traj_noise()
    a, b, m = x1[:N_TRAJ].copy(), x2[:N_TRAJ].copy(), mixed[:N_TRAJ]
    t1s, t2s = [a[..., 0].copy()], [b[..., 0].copy()]
    for t in range(T):
        s1 = o1.grad_log_prob(a)[0].numpy().astype(np.float32)
        s2 = o2.grad_log_prob(b)[0].numpy().astype(np.float32)
        a, b = bo.langevin_update(a, b, s1, s2, m, noise[t, 0], noise[t, 1], eta, lam, ns, g, grad_g)
        if (t + 1) % 10 == 0:
            t1s.append(a[..., 0].copy())
            t2s.append(b[..., 0].copy())
            print(f"trajectory step {t + 1}, {time.time() - t0:.0f} s", flush=True)
    out["traj_x1"], out["traj_x2"] = np.stack(t1s), np.stack(t2s)
    out = sample(out)
    np.savez_compressed(os.path.join(HERE, "glow_k40.npz"), **out)
    print("written", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
