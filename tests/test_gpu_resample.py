"""asep_resample (csrc/resample_kernels.cu) against the float64 restatement of resampy's kaiser_best
(oracle/resample_oracle.py), and the host wrapper audiosourcesep_b200.resample.resample."""
import math

import numpy as np
import pytest
import torch

from audiosourcesep_b200 import _lib
from audiosourcesep_b200.resample import resample
from oracle import resample_oracle as ro

pytestmark = pytest.mark.gpu

RATES = (44100, 48000, 22050, 8000)


def _rows(n, L, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, L)).astype(np.float32)
    x[1] = 0.6 * np.sin(2 * np.pi * 440 * np.arange(L) / 44100)
    return x


@pytest.mark.parametrize("orig_sr", RATES)
def test_kernel_matches_oracle_on_batched_rows(orig_sr):
    L = int(1.5 * orig_sr) + 17
    x = _rows(3, L, orig_sr)
    ratio = 16000 / orig_sr
    n_out = int(L * ratio)
    got = resample(x, orig_sr, 16000).cpu().numpy()
    want = ro.resample_rows(x.astype(np.float64), ratio)
    assert got.shape == (3, math.ceil(L * ratio)) and got.dtype == np.float32
    assert np.all(got[:, n_out:] == 0.0)
    err = np.max(np.abs(got[:, :n_out] - want), axis=1) / np.max(np.abs(x), axis=1)
    print(f"{orig_sr} -> 16000: max error / peak per row {err}")
    assert np.all(err <= 2e-6), err
    # outputs whose time register lies within 1e-9 of an integer (where the running sum and t / ratio part) are covered
    T = ro.time_register(n_out, ratio)
    assert (np.abs(T - np.round(T)) < 1e-9)[1:].any()


def test_kernel_on_ten_minutes_of_44k_audio():
    """One 10-minute 44.1 kHz row (26.5 M input samples): outputs at the start, the middle and the end against the
    oracle evaluated at those indices only (64-bit sample indices; the time register at ~2.6e7)."""
    sr = 44100
    L = 600 * sr
    rng = np.random.default_rng(11)
    x = (0.3 * rng.standard_normal(L)).astype(np.float32)
    got = resample(x, sr, 16000).cpu().numpy()
    ratio = 16000 / sr
    n_out = int(L * ratio)
    assert got.shape == (math.ceil(L * ratio),)
    idx = np.concatenate([np.arange(0, 3000), np.arange(n_out // 2 - 1500, n_out // 2 + 1500), np.arange(n_out - 3000, n_out)])
    want = ro.resample_rows(x.astype(np.float64), ratio, t_index=idx)
    err = np.max(np.abs(got[idx] - want)) / np.max(np.abs(x))
    print(f"10 min row: max error / peak {err:.2e}")
    assert err <= 2e-6


def test_equal_rates_and_one_dimensional_input():
    x = np.random.default_rng(0).standard_normal(5000).astype(np.float32)
    same = resample(x, 16000, 16000)
    assert same.is_cuda and np.array_equal(same.cpu().numpy(), x)
    y = resample(torch.as_tensor(x).cuda(), 8000, 16000)
    assert y.shape == (10000,)
    np.testing.assert_allclose(y.cpu().numpy(), ro.resample(x.astype(np.float64), 8000, 16000), rtol=0, atol=2e-6 * np.abs(x).max())
    with pytest.raises(ValueError):
        resample(x[:2], 44100, 16000)


def test_abi_validates_arguments():
    from audiosourcesep_b200.resample import _device_table, running_time
    _lib.init()
    lib = _lib.load()
    x = torch.zeros((2, 441), device="cuda")
    win, delta = _device_table(16000 / 44100, torch.cuda.current_device())
    t = torch.as_tensor(running_time(160, 16000 / 44100)).cuda()
    out = torch.empty((2, 160), device="cuda")

    def call(step=185, time=t, o=out, w=win):
        d = [_lib.dl(v) for v in (x, time, w, delta, o)]
        return lib.asep_resample(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, 16000 / 44100, step, d[4].ptr, _lib.stream_ptr())

    assert call() == 0
    assert call(step=0) != 0 and b"step" in lib.asep_last_error()
    assert call(time=t.float()) != 0                                  # time must be float64
    assert call(o=torch.empty((2, 159), device="cuda")) != 0          # out must be [N, len(time)]
    assert call(w=win[:-1].contiguous()) != 0                         # delta must match win
