"""Host-side mirror of the reference's ``ncsn/utils.py`` (noise schedule and score-model builders)."""
from __future__ import annotations

import numpy as np


def get_sigmas(sigma1, sigmaL, num_classes, progression="geometric"):
    """Geometric noise schedule sigma_1 ... sigma_L as float32 (reference: ncsn/utils.py:7-14)."""
    if progression == "geometric":
        sigmas = np.exp(np.linspace(np.log(sigma1), np.log(sigmaL), num=num_classes))
    elif progression == "logarithmic":
        sigmas = np.logspace(np.log(sigma1) / np.log(10), np.log(sigmaL) / np.log(10), num=num_classes)
    else:
        raise ValueError("progression should be geometric or logarithmic")
    return sigmas.astype(np.float32)


def langevin_step_constants(sigmas, sigma_idx, delta=2e-5):
    """eta, lambda and sqrt(2 eta) with the reference's float32/float64 casts
    (reference: run_basis_sep.py:158-164; delta is hard-wired to 2e-5 at :239)."""
    sigma = np.float32(sigmas[sigma_idx])
    ratio = np.float32(sigma / np.float32(sigmas[-1]))
    eta = np.float32(np.float64(delta) * np.float64(np.float32(ratio * ratio)))
    lam = np.float32(1.0 / np.float64(np.float32(sigma * sigma)))
    noise_scale = np.float32(np.sqrt(np.float32(np.float32(2.0) * eta)))
    return eta, lam, noise_scale


def _ncsn_cfg(args, version):
    from ..config import NCSNConfig
    H, W, C = (args.data_shape if getattr(args, "data_shape", None) else [args.height, args.width, 1])
    return NCSNConfig(version=version, H=int(H), W=int(W), C=int(C), ngf=int(args.n_filters),
                      num_classes=int(args.num_classes), sigma1=float(args.sigma1), sigmaL=float(args.sigmaL),
                      progression=getattr(args, "progression", "logarithmic"))


def _precision(args) -> int:
    """Default: the split-bf16 tensor-core parity mode (three products per convolution: per-step Langevin gate met at every
    noise level, DESIGN.md section 4).  ``args.fast`` (run_basis_sep --fast) selects one bf16 product per convolution
    (2.5x the throughput, score within 1-5 %)."""
    from .. import _lib
    return _lib.PREC_BF16 if getattr(args, "fast", False) else _lib.PREC_BF16X3


def get_uncompiled_model(args, name="ScoreNetwork", params=None, seed=None):
    """NCSN v1 ``CondRefineNetDilated`` behind the Keras-model call contract (reference: ncsn/utils.py:41-51).
    ``params`` (name -> array) loads weights; otherwise the seeded random init is used."""
    from ..weights import init_ncsn_params
    from .score_model import ScoreModel
    if getattr(args, "use_logit", False):
        raise NotImplementedError("logit_transform=True is not used by configs/melspec_ncsnv1.yml")
    cfg = _ncsn_cfg(args, "v1")
    if params is None:
        params = init_ncsn_params(cfg, seed=0 if seed is None else seed, mode="perturbed" if seed is not None else "faithful")
    return ScoreModel(cfg, params, name=name, precision=_precision(args))


def get_uncompiled_model_v2(args, sigmas, name="ScoreNetworkv2", params=None, seed=None):
    """NCSN v2 ``RefineNetDilated`` (reference: ncsn/utils.py:54-64); the output is divided by sigmas[idx]."""
    from ..weights import init_ncsn_params
    from .score_model import ScoreModel
    cfg = _ncsn_cfg(args, "v2")
    if params is None:
        params = init_ncsn_params(cfg, seed=0 if seed is None else seed, mode="perturbed" if seed is not None else "faithful")
    return ScoreModel(cfg, params, sigmas=np.asarray(sigmas, dtype=np.float32), name=name, precision=_precision(args))


def anneal_langevin_dynamics(x_mod, data_shape, model, n_samples, sigmas, n_steps_each=100, step_lr=2e-5,
                             return_arr=False, verbose=False, noise=None, seed=0):
    """Unconditional annealed Langevin sampler (reference: ncsn/utils.py:17-38):
    ``x <- x + step * score(x, i) + sqrt(2 step) * N(0,1)``, ``step = step_lr * (sigma_i / sigma_L)^2``.

    This is the single-source, lambda = 0 case of the fused BASIS update (SURVEY.md 8(a) row 19): the same
    kernel runs it with K = 2 and a dummy second source, held with x in one [2, ...] state so that no step stacks them.
    ``noise`` ([L, n_steps_each, n, H, W, C] standard normals) injects the draws for parity runs; otherwise Philox noise
    keyed by (seed, step, element) is generated in the kernel."""
    import torch
    from .. import ops
    x0 = torch.as_tensor(np.asarray(x_mod) if not torch.is_tensor(x_mod) else x_mod, dtype=torch.float32).cuda()
    state = torch.zeros((2,) + tuple(x0.shape), dtype=torch.float32, device=x0.device)
    state[0] = x0
    x, dummy = state[0], state[1]
    score = torch.zeros_like(state)                      # row 1: the dummy source's score, zero
    zeros = torch.zeros_like(x)
    injected = None if noise is None else torch.zeros_like(state)   # row 1: the dummy source's draws, zero
    arr = [x.cpu().numpy().copy()] if return_arr else None
    step_no = 0
    for i, sigma in enumerate(sigmas):
        if verbose:
            print("Sigma = {} ({} / {})".format(sigma, i + 1, len(sigmas)))
        labels = torch.full((int(n_samples),), i, dtype=torch.int32, device=x.device)
        ratio = np.float32(np.float32(sigma) / np.float32(sigmas[-1]))
        step_size = np.float32(np.float64(step_lr) * np.float64(np.float32(ratio * ratio)))
        noise_scale = np.float32(np.sqrt(np.float32(step_size * np.float32(2.0))))
        for s in range(int(n_steps_each)):
            score[0].copy_(model([x, labels], training=True))
            if injected is not None:
                injected[0].copy_(torch.as_tensor(noise[i][s], dtype=torch.float32))
            ops.langevin_step_k(state, score, zeros, float(step_size), 0.0, float(noise_scale), noise=injected, seed=seed,
                                step=step_no)
            dummy.zero_()
            step_no += 1
        if return_arr:
            arr.append(x.cpu().numpy().copy())
    return np.stack(arr, axis=0) if return_arr else x.cpu().numpy()
