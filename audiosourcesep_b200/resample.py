"""Band-limited resampling on the device: host side of csrc/resample_kernels.cu.

Replaces the resampler inside ``librosa.load(path, sr=16000)`` of the reference (datasets/preprocessing.py:9-26):
librosa 0.7 / 0.8 with ``res_type='kaiser_best'``, i.e. ``resampy.resample(y, orig_sr, target_sr, filter='kaiser_best')``
followed by ``librosa.util.fix_length`` to ``ceil(L * ratio)`` samples.  The interpolation table and resampy's running
time register are built here in float64 (the table once per ratio); the filter itself runs in libasep.so.  Two resampy
quirks are kept on purpose: the time register is a running sum (not ``t / ratio``) and the table stride is truncated
to an integer -- outputs where either matters differ from the textbook filter by ~1e-3 (oracle/resample_oracle.py).
"""
from __future__ import annotations

import functools
import math

import numpy as np
import torch

from . import _lib

NUM_ZEROS = 64
NUM_TABLE = 512                      # 2^precision, precision = 9
ROLLOFF = 0.9475937167399596
BETA = 14.769656459379492


def kaiser_best_table(ratio: float):
    """resampy's kaiser_best (win, delta) float64 [NUM_TABLE * NUM_ZEROS + 1], scaled by ``ratio`` when downsampling."""
    n = NUM_TABLE * NUM_ZEROS
    win = ROLLOFF * np.sinc(ROLLOFF * np.linspace(0, NUM_ZEROS, num=n + 1, endpoint=True))
    win *= np.kaiser(2 * n + 1, BETA)[n:]
    if ratio < 1:
        win *= ratio
    delta = np.zeros_like(win)
    delta[:-1] = np.diff(win)
    return win, delta


def running_time(n_out: int, ratio: float) -> np.ndarray:
    """resampy's time register 0, inc, inc + inc, ... (inc = 1 / ratio) as float64 [n_out]; np.cumsum accumulates in
    order, so every entry is bit-identical to resampy's ``time_register += time_increment``."""
    steps = np.full(int(n_out), 1.0 / ratio)
    if n_out:
        steps[0] = 0.0
    return np.cumsum(steps)


@functools.lru_cache(maxsize=8)
def _device_table(ratio: float, device: int):
    win, delta = kaiser_best_table(ratio)
    dev = torch.device("cuda", device)
    return (torch.as_tensor(win.astype(np.float32)).to(dev), torch.as_tensor(delta.astype(np.float32)).to(dev))


def resample(y, orig_sr: int, target_sr: int, device=None) -> torch.Tensor:
    """librosa.resample(y, orig_sr, target_sr, res_type='kaiser_best') of a 1-D signal or of every row of [N, L]:
    float32 device tensor of ``ceil(L * target_sr / orig_sr)`` samples per row (resampy's ``int(L * ratio)`` outputs,
    zero-padded by librosa's fix_length).  Equal rates return the input (as a float32 device tensor) untouched."""
    d = _lib.init(device)
    a = torch.as_tensor(y, dtype=torch.float32).to(torch.device("cuda", d)).contiguous()
    if a.ndim not in (1, 2):
        raise ValueError(f"resample: expected a 1-D signal or [N, L] rows, got shape {tuple(a.shape)}")
    if int(orig_sr) <= 0 or int(target_sr) <= 0:
        raise ValueError(f"resample: sampling rates must be positive ({orig_sr}, {target_sr})")
    if int(orig_sr) == int(target_sr):
        return a
    ratio = float(target_sr) / float(orig_sr)
    rows = a if a.ndim == 2 else a[None]
    N, L = rows.shape
    n_out = int(L * ratio)
    if n_out < 1:
        raise ValueError(f"resample: {L} samples are too few to resample from {orig_sr} Hz to {target_sr} Hz")
    n_fix = int(math.ceil(L * ratio))
    scale = min(1.0, ratio)
    win, delta = _device_table(ratio, d)
    time = torch.as_tensor(running_time(n_out, ratio)).to(a.device)
    out = torch.empty((N, n_out), dtype=torch.float32, device=a.device)
    dx, dt, dw, dd, do = (_lib.dl(v) for v in (rows, time, win, delta, out))
    _lib.check(_lib.load().asep_resample(dx.ptr, dt.ptr, dw.ptr, dd.ptr, float(scale), int(scale * NUM_TABLE), do.ptr,
                                         _lib.stream_ptr()))
    if n_fix > n_out:
        out = torch.nn.functional.pad(out, (0, n_fix - n_out))
    elif n_fix < n_out:
        out = out[:, :n_fix].contiguous()
    return out if a.ndim == 2 else out[0]
