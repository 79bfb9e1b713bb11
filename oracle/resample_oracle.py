"""CPU ORACLE (test infrastructure, NOT a product path) -- band-limited resampling as the reference loads audio.

The reference reads every wav with ``librosa.load(path, sr=16000)`` (datasets/preprocessing.py:9-26,
datasets/wav_to_spec.py), librosa 0.7 / 0.8 with its default ``res_type='kaiser_best'``, which calls
``resampy.resample(y, orig_sr, target_sr, filter='kaiser_best')`` and then ``librosa.util.fix_length`` to
``ceil(L * ratio)`` samples.  Neither library is installed here, so parity is unpinned; this float64 restatement of
resampy's published algorithm is the definition the device kernel is checked against:

  filter table   num_zeros = 64, precision = 9 (512 table entries per zero crossing), rolloff = 0.9475937167399596,
                 Kaiser beta = 14.769656459379492; win = rolloff * sinc(rolloff * linspace(0, 64, n + 1)) *
                 kaiser(2 n + 1, beta)[n:], n = 512 * 64; win *= ratio when downsampling; delta = diff(win), 0 appended
  resample_f     per output sample t the running time register T_t (0, inc, 2 inc, ... accumulated by repeated
                 addition, inc = 1 / ratio), k = int(T_t), and the left / right filter wings read with the TRUNCATED
                 table step int(min(1, ratio) * 512) -- both resampy quirks are kept (see tests/test_oracle_resample.py)

It owns its table and its loops and shares no code with audiosourcesep_b200/resample.py.
"""
from __future__ import annotations

import math

import numpy as np

NUM_ZEROS = 64
PRECISION = 9
ROLLOFF = 0.9475937167399596
BETA = 14.769656459379492


def kaiser_half(n_half: int, beta: float) -> np.ndarray:
    """The right half (centre included) of a symmetric Kaiser window of 2 n_half + 1 points, from its definition."""
    m = 2 * n_half                                              # M - 1
    k = np.arange(n_half, 2 * n_half + 1, dtype=np.float64)
    r = 2.0 * k / m - 1.0
    return np.i0(beta * np.sqrt(np.maximum(0.0, 1.0 - r * r))) / np.i0(beta)


def filter_table(ratio: float):
    """(win, delta) float64 [512 * 64 + 1] of kaiser_best for ``ratio`` = target_sr / orig_sr."""
    num_table = 2 ** PRECISION
    n = num_table * NUM_ZEROS
    t = np.linspace(0.0, NUM_ZEROS, n + 1)
    win = ROLLOFF * np.sinc(ROLLOFF * t) * kaiser_half(n, BETA)
    if ratio < 1:
        win = win * ratio
    delta = np.zeros_like(win)
    delta[:-1] = np.diff(win)
    return win, delta


def time_register_loop(n_out: int, ratio: float) -> np.ndarray:
    """resampy's time register, literally: T_0 = 0, T_{t+1} = T_t + 1 / ratio."""
    inc = 1.0 / ratio
    out = np.empty(n_out, dtype=np.float64)
    tr = 0.0
    for t in range(n_out):
        out[t] = tr
        tr += inc
    return out


def time_register(n_out: int, ratio: float) -> np.ndarray:
    """The same running sum by np.cumsum (a sequential float64 accumulation: bit-identical to the loop)."""
    steps = np.full(n_out, 1.0 / ratio)
    steps[0] = 0.0
    return np.cumsum(steps)


def resample_loop(x: np.ndarray, ratio: float) -> np.ndarray:
    """resampy's resample_f for one row, one output sample at a time, in float64 (length int(L * ratio))."""
    x = np.asarray(x, dtype=np.float64)
    win, delta = filter_table(ratio)
    num_table = 2 ** PRECISION
    scale = min(1.0, ratio)
    step = int(scale * num_table)
    nwin = win.shape[0]
    L = x.shape[0]
    n_out = int(L * ratio)
    y = np.zeros(n_out, dtype=np.float64)
    T = time_register_loop(n_out, ratio)
    for t in range(n_out):
        k = int(T[t])
        frac = scale * (T[t] - k)
        idx = frac * num_table
        off = int(idx)
        eta = idx - off
        acc = 0.0
        for i in range(min(k + 1, (nwin - off) // step)):
            acc += (win[off + i * step] + eta * delta[off + i * step]) * x[k - i]
        frac = scale - frac
        idx = frac * num_table
        off = int(idx)
        eta = idx - off
        for j in range(max(0, min(L - k - 1, (nwin - off) // step))):
            acc += (win[off + j * step] + eta * delta[off + j * step]) * x[k + 1 + j]
        y[t] = acc
    return y


def resample_rows(x: np.ndarray, ratio: float, t_index=None, chunk: int = 4096) -> np.ndarray:
    """Vectorised form of :func:`resample_loop` over rows ``x`` [N, L] (or [L]) in float64.  ``t_index``: evaluate
    only those output samples (the time register is still the running sum from t = 0)."""
    x = np.asarray(x, dtype=np.float64)
    one = x.ndim == 1
    x2 = x[None] if one else x
    N, L = x2.shape
    win, delta = filter_table(ratio)
    num_table = 2 ** PRECISION
    scale = min(1.0, ratio)
    step = int(scale * num_table)
    nwin = win.shape[0]
    n_out = int(L * ratio)
    T_all = time_register(n_out, ratio)
    ts = np.arange(n_out) if t_index is None else np.asarray(t_index, dtype=np.int64)
    y = np.zeros((N, ts.size), dtype=np.float64)
    nmax = (nwin + step - 1) // step
    taps = np.arange(nmax)
    xp = np.concatenate([np.zeros((N, nmax)), x2, np.zeros((N, nmax + 1))], axis=1)   # zero guards: masked taps
    for c0 in range(0, ts.size, chunk):
        tt = ts[c0: c0 + chunk]
        T = T_all[tt]
        k = T.astype(np.int64)
        frac = scale * (T - k)
        for side in (0, 1):
            if side:
                frac = scale - frac
            idx = frac * num_table
            off = idx.astype(np.int64)
            eta = idx - off
            limit = np.minimum(k + 1, (nwin - off) // step) if side == 0 else np.minimum(L - k - 1, (nwin - off) // step)
            ti = off[:, None] + taps[None, :] * step
            valid = taps[None, :] < limit[:, None]
            ti = np.where(valid, ti, 0)
            w = np.where(valid, win[ti] + eta[:, None] * delta[ti], 0.0)
            src = (k[:, None] - taps[None, :]) if side == 0 else (k[:, None] + 1 + taps[None, :])
            y[:, c0: c0 + tt.size] += np.einsum("tj,ntj->nt", w, xp[:, src + nmax])
    return y[0] if one else y


def resample(y: np.ndarray, orig_sr: int, target_sr: int) -> np.ndarray:
    """librosa.resample(y, orig_sr, target_sr, res_type='kaiser_best') in float64: resampy's int(L * ratio) samples,
    zero-padded or trimmed to ceil(L * ratio) (librosa.util.fix_length); equal rates return the input."""
    y = np.asarray(y, dtype=np.float64)
    if orig_sr == target_sr:
        return y
    ratio = float(target_sr) / orig_sr
    L = y.shape[-1]
    if int(L * ratio) < 1:
        raise ValueError(f"input of {L} samples is too short to resample from {orig_sr} to {target_sr}")
    out = resample_rows(y, ratio)
    n = int(math.ceil(L * ratio))
    if out.shape[-1] >= n:
        return out[..., :n]
    pad = [(0, 0)] * (out.ndim - 1) + [(0, n - out.shape[-1])]
    return np.pad(out, pad)
