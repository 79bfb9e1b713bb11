"""Synthetic mel-spectrogram patches of the ``configs/melspec_*.yml`` shape.

There is no dataset in the build or benchmark environment, so the workload inputs are
generated: a white field smoothed by a separable AR(1) filter (lag-1 autocorrelation
0.78 along frequency, 0.96 along time), mapped to mean -46 dB / std 19 dB and clipped to
[-100, 20] dB -- the statistics of the 30 real patches shipped in the reference's
``basis_sep_results/beethoven_sonata_1_sep_1min/results.npz`` (SURVEY.md 8(c)(ii), 8(d)).
Mixtures are power sums of two sources; everything is normalised to [0, 1] exactly as
the separation script does (reference: run_basis_sep.py:355).
"""
from __future__ import annotations

import numpy as np

DB_MIN, DB_MAX = -100.0, 20.0


def _ar1(x: np.ndarray, rho: float, axis: int) -> np.ndarray:
    """Stationary AR(1) smoothing along ``axis`` (unit marginal variance)."""
    x = np.moveaxis(x, axis, 0).copy()
    g = np.sqrt(1.0 - rho * rho)
    for i in range(1, x.shape[0]):
        x[i] = rho * x[i - 1] + g * x[i]
    return np.moveaxis(x, 0, axis)


def mel_patches_db(n: int, seed: int, H: int = 96, W: int = 64) -> np.ndarray:
    """``[n, H, W, 1]`` float32 patches in dB, clipped to [-100, 20]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    f = rng.standard_normal((n, H, W))
    f = _ar1(f, 0.78, 1)
    f = _ar1(f, 0.96, 2)
    db = np.clip(-46.0 + 19.0 * f, DB_MIN, DB_MAX)
    return np.ascontiguousarray(db.astype(np.float32))[..., None]


def normalise(db: np.ndarray) -> np.ndarray:
    """(x - min) / (max - min)  (reference: run_basis_sep.py:355)."""
    return np.ascontiguousarray((db - DB_MIN) / (DB_MAX - DB_MIN), dtype=np.float32)


def mixture_db(*sources_db: np.ndarray) -> np.ndarray:
    """Power-sum mixture of two or more dB patches (summed in argument order), clipped like the data loader does."""
    if len(sources_db) < 2:
        raise ValueError("a mixture needs at least two sources")
    p = np.power(10.0, sources_db[0].astype(np.float64) / 10.0)
    for s in sources_db[1:]:
        p = p + np.power(10.0, s.astype(np.float64) / 10.0)
    return np.clip(10.0 * np.log10(p), DB_MIN, DB_MAX).astype(np.float32)


def basis_problem(n_mixed: int, seed1: int = 0, seed2: int = 1, H: int = 96, W: int = 64):
    """(mixed, gt1, gt2): mixture normalised to [0,1]; ground truths in dB."""
    gt1 = mel_patches_db(n_mixed, seed1, H, W)
    gt2 = mel_patches_db(n_mixed, seed2, H, W)
    mixed = normalise(mixture_db(gt1, gt2))
    return mixed, gt1, gt2


def langevin_init(n_mixed: int, seed: int, H: int = 96, W: int = 64):
    """x1, x2 ~ U(0,1)  (reference: run_basis_sep.py:360-361)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    x1 = rng.uniform(0.0, 1.0, (n_mixed, H, W, 1)).astype(np.float32)
    x2 = rng.uniform(0.0, 1.0, (n_mixed, H, W, 1)).astype(np.float32)
    return x1, x2
