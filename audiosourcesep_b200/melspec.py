"""Mel-spectrogram front end and inversion back end: host side of csrc/mel_kernels.cu.

Replaces the librosa calls of the reference (datasets/data_loader.py:144-162, melspec_inversion_basis.py:42-119).  The
filter bank (librosa.filters.mel, htk=False, norm='slaney'), its pseudo-inverse and the index ranges the kernels use are
built here in numpy once per parameter set; the transforms themselves run in libasep.so on the current CUDA device.
"""
from __future__ import annotations

import functools
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib


# ---- librosa.filters.mel restated (Slaney mel scale, Slaney area normalisation)
def hz_to_mel(f):
    f = np.asanyarray(f, dtype=np.float64)
    f_sp = 200.0 / 3
    min_log_hz, min_log_mel, logstep = 1000.0, 1000.0 / f_sp, np.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, 1e-30) / min_log_hz) / logstep, f / f_sp)


def mel_to_hz(m):
    m = np.asanyarray(m, dtype=np.float64)
    f_sp = 200.0 / 3
    min_log_hz, min_log_mel, logstep = 1000.0, 1000.0 / f_sp, np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_filters(sr=16000, n_fft=2048, n_mels=96, fmin=125.0, fmax=7600.0) -> np.ndarray:
    fftfreqs = np.linspace(0, float(sr) / 2, 1 + n_fft // 2)
    mel_f = mel_to_hz(np.linspace(hz_to_mel(fmin), hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    w = np.zeros((n_mels, 1 + n_fft // 2))
    for i in range(n_mels):
        w[i] = np.maximum(0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    w *= (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]
    return w.astype(np.float32)


class _Bank:
    """Device copies of one filter bank and of everything derived from it."""

    def __init__(self, sr, n_fft, n_mels, fmin, fmax, device):
        A = mel_filters(sr, n_fft, n_mels, fmin, fmax)
        nz = A > 0
        lo = np.array([np.argmax(r) if r.any() else 0 for r in nz], dtype=np.int32)
        hi = np.array([len(r) - np.argmax(r[::-1]) if r.any() else 0 for r in nz], dtype=np.int32)
        flo = np.array([np.argmax(c) if c.any() else 0 for c in nz.T], dtype=np.int32)
        fhi = np.array([len(c) - np.argmax(c[::-1]) if c.any() else 0 for c in nz.T], dtype=np.int32)
        A64 = A.astype(np.float64)
        self.step = float(1.0 / np.linalg.norm(A64, 2) ** 2)
        dev = torch.device("cuda", device)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)
        self.basis, self.pinv = t(A), t(np.linalg.pinv(A64).astype(np.float32))
        self.lo, self.hi, self.flo, self.fhi = t(lo), t(hi), t(flo), t(fhi)
        self.n_mels, self.n_bins = A.shape


@functools.lru_cache(maxsize=8)
def _bank(sr, n_fft, n_mels, fmin, fmax, device) -> _Bank:
    return _Bank(sr, n_fft, n_mels, fmin, fmax, device)


def _dev(device=None) -> int:
    return _lib.init(device)


def _f32(x, dev) -> torch.Tensor:
    return torch.as_tensor(x, dtype=torch.float32).to(torch.device("cuda", dev)).contiguous()


def stft(audio, n_fft: int = 2048, hop_length: int = 512, device=None) -> torch.Tensor:
    """librosa.stft(window='hann', center=True, pad_mode='reflect') of every row of ``audio`` [N, L]
    -> complex64 [N, 1 + n_fft/2, 1 + L // hop_length] (device)."""
    d = _dev(device)
    a = _f32(audio, d)
    if a.ndim == 1:
        a = a[None]
    N, L = a.shape
    out = torch.empty((N, n_fft // 2 + 1, 1 + L // hop_length, 2), dtype=torch.float32, device=a.device)
    da, do = _lib.dl(a), _lib.dl(out)
    _lib.check(_lib.load().asep_stft(da.ptr, int(n_fft), int(hop_length), do.ptr, _lib.stream_ptr()))
    return torch.view_as_complex(out)


def melspectrogram_db(stft_c: torch.Tensor, sr=16000, n_fft=2048, n_mels=96, fmin=125.0, fmax=7600.0, dbmin=-100.0, dbmax=20.0,
                      amin=1e-10, top_db=80.0) -> torch.Tensor:
    """np.clip(librosa.power_to_db(librosa.feature.melspectrogram(S=|stft|^2, power=2)), dbmin, dbmax) per segment
    (data_loader.py:151-162): complex64 [N, F, T] -> float32 [N, n_mels, T]."""
    d = stft_c.device.index
    bank = _bank(int(sr), int(n_fft), int(n_mels), float(fmin), float(fmax), d)
    s = torch.view_as_real(stft_c.contiguous()).contiguous()
    N, F, T, _ = s.shape
    out = torch.empty((N, n_mels, T), dtype=torch.float32, device=s.device)
    ds, db, dl, dh, do = (_lib.dl(v) for v in (s, bank.basis, bank.lo, bank.hi, out))
    _lib.check(_lib.load().asep_mel_db(ds.ptr, db.ptr, dl.ptr, dh.ptr, do.ptr, float(amin), float(top_db), float(dbmin), float(dbmax),
                                       _lib.stream_ptr()))
    return out


def mel_to_stft(mel_db: torch.Tensor, sr=16000, n_fft=2048, fmin=125.0, fmax=7600.0, iters: int = 300) -> torch.Tensor:
    """librosa.feature.inverse.mel_to_stft(librosa.db_to_power(mel_db), power=2): float32 [N, n_mels, T] dB -> STFT
    magnitudes [N, F, T].  NNLS by FISTA from the clipped least-squares start (see INTEGRATION.md)."""
    d = _dev(None)
    m = _f32(mel_db, d)
    N, M, T = m.shape
    bank = _bank(int(sr), int(n_fft), int(M), float(fmin), float(fmax), d)
    out = torch.empty((N, bank.n_bins, T), dtype=torch.float32, device=m.device)
    dm, db, dp, dl, dh, do = (_lib.dl(v) for v in (m, bank.basis, bank.pinv, bank.flo, bank.fhi, out))
    _lib.check(_lib.load().asep_mel_to_stft(dm.ptr, db.ptr, dp.ptr, dl.ptr, dh.ptr, do.ptr, float(bank.step), int(iters),
                                            _lib.stream_ptr()))
    return out


def stft_filter(mags: torch.Tensor, stft_mixture: torch.Tensor, wiener_filter: bool) -> torch.Tensor:
    """mags [S, N, F, T], stft_mixture complex64 [N, F, T] -> complex64 [S, N, F, T]: single_channel_wiener_filter on
    mags^2 (melspec_inversion_basis.py:93-119) or complex_array(mags, angle(stft_mixture)) (:17-18, :84)."""
    m = mags.contiguous()
    x = torch.view_as_real(stft_mixture.contiguous()).contiguous()
    out = torch.empty(tuple(m.shape) + (2,), dtype=torch.float32, device=m.device)
    dm, dx, do = _lib.dl(m), _lib.dl(x), _lib.dl(out)
    _lib.check(_lib.load().asep_stft_filter(dm.ptr, dx.ptr, do.ptr, int(bool(wiener_filter)), _lib.stream_ptr()))
    return torch.view_as_complex(out)


def istft(stft_c: torch.Tensor, hop_length: int = 512) -> torch.Tensor:
    """librosa.istft(hop_length, window='hann', center=True): complex64 [N, F, T] -> float32 [N, hop (T-1)]."""
    s = torch.view_as_real(stft_c.contiguous()).contiguous()
    N, F, T, _ = s.shape
    out = torch.empty((N, hop_length * (T - 1)), dtype=torch.float32, device=s.device)
    ds, do = _lib.dl(s), _lib.dl(out)
    _lib.check(_lib.load().asep_istft(ds.ptr, int(hop_length), do.ptr, _lib.stream_ptr()))
    return out


def istft_track(stft_c: torch.Tensor, overlap_frames: int, length: int, hop_length: int = 512) -> torch.Tensor:
    """iSTFT of the overlapping segments of one track, written as the whole track: complex64 [S, n_seg, F, T] -> float32
    [S, length].  Segment g starts at sample g P, P = hop (T-1) - hop overlap_frames; neighbours are cross-faded linearly
    over the hop * overlap_frames samples they share (asep_istft_track, restated in oracle/track_oracle.py)."""
    s = torch.view_as_real(stft_c.contiguous()).contiguous()
    if s.ndim != 5:
        raise ValueError(f"istft_track: expected complex [S, n_seg, F, T], got shape {tuple(stft_c.shape)}")
    _dev(s.device.index)
    out = torch.empty((s.shape[0], int(length)), dtype=torch.float32, device=s.device)
    ds, do = _lib.dl(s), _lib.dl(out)
    _lib.check(_lib.load().asep_istft_track(ds.ptr, int(hop_length), int(overlap_frames), do.ptr, _lib.stream_ptr()))
    return out


def griffinlim(mag: torch.Tensor, n_iter: int = 32, hop_length: int = 512, momentum: float = 0.99, seed: Optional[int] = None) -> torch.Tensor:
    """librosa.griffinlim(S, n_iter=32, hop_length, momentum=0.99, init='random'): STFT magnitudes [N, F, T] -> audio
    [N, hop (T-1)].  Random initial phases (librosa draws them from an unseeded RandomState, so outputs are not
    sample-comparable with it; ``seed`` makes this implementation reproducible); every iteration is istft -> stft ->
    phase update (asep_griffinlim_update), all on the device."""
    m = mag.contiguous().float()
    N, F, T = m.shape
    n_fft = 2 * (F - 1)
    g = torch.Generator(device=m.device)
    g.manual_seed(0 if seed is None else int(seed))
    phase = 2.0 * np.pi * torch.rand(m.shape, generator=g, device=m.device)
    cur = torch.view_as_real(torch.polar(m, phase)).contiguous()              # S * angles
    tprev = torch.zeros_like(cur)
    nxt = torch.empty_like(cur)
    lib = _lib.load()
    for _ in range(int(n_iter)):
        audio = istft(torch.view_as_complex(cur), hop_length)
        rebuilt = torch.view_as_real(stft(audio, n_fft=n_fft, hop_length=hop_length)).contiguous()
        dm, dr, dt, dn = (_lib.dl(v) for v in (m, rebuilt, tprev, nxt))
        _lib.check(lib.asep_griffinlim_update(dm.ptr, dr.ptr, dt.ptr, dn.ptr, float(momentum), _lib.stream_ptr()))
        cur, nxt = nxt, cur
    return istft(torch.view_as_complex(cur), hop_length)
