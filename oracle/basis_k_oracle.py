"""CPU ORACLE (test infrastructure, NOT a product path) -- BASIS annealed Langevin loop with K sources.

Restates run_basis_sep.py:152-260 for K sources in numpy float32 with the reference's evaluation order, on top of the
K-general ``mixing_process`` of basis_oracle (run_basis_sep.py:106-149).  The operations of one update are those of
``basis_oracle.langevin_update`` in the same order, so K = 2 equals the two-source restatement bit for bit.
Noise is INJECTED (arrays of standard normals) so that CUDA and oracle see the same draws.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from .basis_oracle import mixing_process, step_constants


def langevin_update_k(xs: Sequence[np.ndarray], ss: Sequence[np.ndarray], mixed, ns: Sequence[np.ndarray], eta, lam,
                      noise_scale, g, grad_g) -> List[np.ndarray]:
    """One update of run_basis_sep.py:163-181 for K sources; ns are standard-normal draws."""
    mixing = g(*xs)
    gms = grad_g(*xs)
    out = []
    for x, s, n, gm in zip(xs, ss, ns, gms):
        eps = noise_scale * n
        out.append((x + eta * (s + lam * gm * (mixed - mixing)) + eps).astype(np.float32))
    return out


def basis_run_k(mixed, xs: Sequence[np.ndarray], scores: Sequence[Callable], sigmas, T: int,
                noise: Callable[[int, int], Sequence[np.ndarray]], delta: float = 2e-5, data_type="melspec", scale="dB",
                per_step: Optional[List] = None):
    """basis_outer_loop + basis_inner_loop for K sources.  ``scores[k](x, sigma_idx) -> grad log p`` (float32);
    ``noise(sigma_idx, t) -> K`` standard normal arrays.  Returns the K states and x_arr {"x1": [...], ..., "xK": [...]}."""
    g, grad_g = mixing_process(data_type, scale)
    xs = [x.copy() for x in xs]
    x_arr: Dict[str, List[np.ndarray]] = {f"x{k + 1}": [x.copy()] for k, x in enumerate(xs)}
    for i in range(len(sigmas)):
        eta, lam, ns = step_constants(sigmas, i, delta)
        for t in range(T):
            zs = noise(i, t)
            ss = [score(x, i) for score, x in zip(scores, xs)]
            xs = langevin_update_k(xs, ss, mixed, zs, eta, lam, ns, g, grad_g)
            if per_step is not None:
                per_step.append(tuple(x.copy() for x in xs))
        for k, x in enumerate(xs):
            x_arr[f"x{k + 1}"].append(x.copy())
    return xs, x_arr
