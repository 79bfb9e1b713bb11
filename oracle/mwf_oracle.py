"""CPU ORACLE (test infrastructure, NOT a product path) -- rendering a whole-track separation as multichannel Wiener masks
on the original recording (run_basis_sep --mix --render mask; audiosourcesep_b200/track.py:render_track and
csrc/mwf_kernels.cu), restated in float64 numpy.

Inputs: the K sources' NNLS magnitudes on the 16 kHz segment grid mag [K, n_seg, 1025, 64] (melspec.mel_to_stft of the
separated mel patches, as invert_track gets them), the segmentation (overlap_frames o, track_length) and the original
audio x [C, L] at orig_sr, C in {1, 2}.

a. Output STFT grid: n_fft' = 2^round(log2(2048 orig_sr / 16000)) clamped to [256, 4096], hop' = n_fft' / 4 (2048 / 512 at
   16 kHz, the mel grid itself; 4096 / 1024 at 44.1 and 48 kHz).  X = stft(x zero-padded to a multiple of hop', and to at
   least n_fft' samples) per channel: [C, F', T'].
b. Track PSD on that grid, psd [K, F', T']:
   * frame j of segment g is 16 kHz track frame g (63 - o) + j; T16 = (n_seg - 1)(63 - o) + 64 track frames;
   * segments sharing a frame blend their powers mag^2 with the cross-fade weight of the frame's centre sample
     (track_oracle.crossfade_weights, i.e. asep_istft_track): the frame at in-segment sample p = 512 j weighs 1, (p + 0.5)/O
     on the fade-in of a segment after the first, max(0, (V - p - 0.5)/O) on the fade-out of a segment before the last (0
     at o = 0), so the zero-weight edge frames drop out; the last frame of the last segment keeps weight 1;
   * output frame u sits at the fractional 16 kHz frame q = hop' u 16000 / (orig_sr 512), clamped to [0, T16 - 1]; output
     bin b' at the fractional 16 kHz bin p = b' orig_sr 2048 / (n_fft' 16000), clamped to [bin_lo, bin_hi], the first and
     last bins some mel filter covers (band_edges);
   * bilinear interpolation in power.  Outside the mel band every frame therefore takes the gains of the nearest covered
     bin: content the model never saw (below 133 Hz, above 7.6 kHz) is shared out like its nearest in-band neighbour.
c. Multichannel Wiener filter with EM (norbert.expectation_maximization), n >= 0 iterations, eps = 1e-10:
   y_k(0) = v_k / (sum_j v_j + eps) x per channel with v = psd; then for i = 1..n: v_k = mean_c |y_k|^2,
   R_k[f] = sum_t y_k y_k^H / (eps + sum_t v_k), C_xx = sum_k v_k R_k + eps I, y_k = v_k R_k C_xx^-1 x.  After every step
   the residual x - sum_k y_k is added to every source in equal shares of 1/K (mixture consistency).
   C_xx^-1 x is evaluated as (adj(M) x + eps x) / (max(det M, 0) + eps tr M + eps^2) with M = sum_k v_k R_k: the same
   quantity, but exact for rank-1 M (dual-mono input), where the naive (M + eps I)^-1 loses eps to rounding.
d. Each y_k through the iSTFT at hop', cut to L: [K, C, L] at orig_sr.
"""
from __future__ import annotations

import math

import numpy as np

from . import mel_oracle

SR = 16000
HOP = 512
N_FFT = 2048
EPS = 1e-10
MAX_ITERATIONS = 10


def out_grid(orig_sr: int):
    """(n_fft', hop') of the output STFT at orig_sr."""
    n = 2 ** int(round(math.log2(N_FFT * float(orig_sr) / SR)))
    n = min(4096, max(256, n))
    return n, n // 4


def padded_length(L: int, hop: int, n_fft: int) -> int:
    return max(-(-int(L) // hop) * hop, n_fft)


def band_edges(n_mels=96, fmin=125.0, fmax=7600.0):
    """(bin_lo, bin_hi): the first and last 16 kHz STFT bins that some mel filter covers."""
    cover = np.flatnonzero((mel_oracle.mel_filters(SR, N_FFT, n_mels, fmin, fmax) > 0).any(axis=0))
    return int(cover[0]), int(cover[-1])


def frame_weights(n_seg: int, T: int, overlap_frames: int, hop: int = HOP) -> np.ndarray:
    """float64 [n_seg, T]: the cross-fade weight of frame j of segment g (its centre sample)."""
    V, O = hop * (T - 1), hop * overlap_frames
    P = V - O
    p = hop * np.arange(T, dtype=np.float64)
    w = np.ones((n_seg, T))
    for g in range(n_seg):
        if g > 0 and O > 0:
            w[g] = np.where(p < O, (p + 0.5) / max(O, 1), w[g])
        if g < n_seg - 1:
            fade = np.maximum(0.0, (V - p - 0.5) / O) if O > 0 else np.zeros(T)
            w[g] = np.where(p >= P, fade, w[g])
    return w


def segment_power(mag: np.ndarray, overlap_frames: int, hop: int = HOP) -> np.ndarray:
    """mag [K, n_seg, F, T] -> float64 [K, F, T16]: the cross-faded power of every 16 kHz track frame."""
    K, n_seg, F, T = mag.shape
    Q = T - 1 - overlap_frames
    T16 = (n_seg - 1) * Q + T
    w = frame_weights(n_seg, T, overlap_frames, hop)
    num, den = np.zeros((K, F, T16)), np.zeros(T16)
    m2 = mag.astype(np.float64) ** 2
    for g in range(n_seg):
        num[:, :, g * Q: g * Q + T] += w[g] * m2[:, g]
        den[g * Q: g * Q + T] += w[g]
    return num / den


def track_psd(mag: np.ndarray, overlap_frames: int, bin_lo: int, bin_hi: int, out_sr: int, out_n_fft: int, out_hop: int,
              T_out: int, hop: int = HOP) -> np.ndarray:
    """float64 [K, out_n_fft/2 + 1, T_out]: the track PSD bilinearly mapped onto the output grid."""
    K, n_seg, F, T = mag.shape
    P16 = segment_power(mag, overlap_frames, hop)
    T16 = P16.shape[2]
    n16 = 2 * (F - 1)
    u = np.arange(T_out, dtype=np.int64)
    q = np.clip((u * out_hop * SR).astype(np.float64) / float(out_sr * hop), 0.0, T16 - 1)
    q0 = np.floor(q).astype(np.int64)
    q1, a = np.minimum(q0 + 1, T16 - 1), q - q0
    b = np.arange(out_n_fft // 2 + 1, dtype=np.int64)
    p = np.clip((b * out_sr * n16).astype(np.float64) / float(out_n_fft * SR), bin_lo, bin_hi)
    p0 = np.floor(p).astype(np.int64)
    p1, beta = np.minimum(p0 + 1, bin_hi), p - p0
    rows = P16[:, p0, :] * (1 - beta)[:, None] + P16[:, p1, :] * beta[:, None]
    return rows[:, :, q0] * (1 - a) + rows[:, :, q1] * a


def _consistent(y, x):
    return y + (x - y.sum(axis=0)) / y.shape[0]


def _solve(M, x):
    """(M + eps I)^-1 x per bin; M [F, T, C, C] Hermitian PSD, x [C, F, T]."""
    C = x.shape[0]
    if C == 1:
        return x / (M[..., 0, 0].real + EPS)[None]
    m00, m11, m01 = M[..., 0, 0].real, M[..., 1, 1].real, M[..., 0, 1]
    det = np.maximum(m00 * m11 - (m01.real * m01.real + m01.imag * m01.imag), 0.0) + EPS * (m00 + m11) + EPS * EPS
    z0 = m11 * x[0] - m01 * x[1] + EPS * x[0]
    z1 = -np.conj(m01) * x[0] + m00 * x[1] + EPS * x[1]
    return np.stack([z0, z1]) / det[None]


def mwf(psd: np.ndarray, X: np.ndarray, iterations: int = 1) -> np.ndarray:
    """psd [K, F, T] (power), X complex [C, F, T] -> complex128 [K, C, F, T]."""
    if not 0 <= iterations <= MAX_ITERATIONS:
        raise ValueError(iterations)
    v = np.asarray(psd, dtype=np.float64)
    x = np.asarray(X, dtype=np.complex128)
    y = _consistent(v[:, None] / (v.sum(axis=0) + EPS)[None, None] * x[None], x)
    for _ in range(iterations):
        v = np.mean(np.abs(y) ** 2, axis=1)                                              # [K, F, T]
        R = np.einsum("kcft,kdft->kfcd", y, np.conj(y)) / (EPS + v.sum(axis=-1))[:, :, None, None]
        M = np.einsum("kft,kfcd->ftcd", v, R)
        z = _solve(M, x)
        y = _consistent(v[:, None] * np.einsum("kfcd,dft->kcft", R, z), x)
    return y


def render(mag: np.ndarray, overlap_frames: int, audio: np.ndarray, orig_sr: int, iterations: int = 1,
           n_mels: int = 96) -> np.ndarray:
    """mag [K, n_seg, 1025, 64], audio [C, L] at orig_sr -> float64 [K, C, L]: a-d above."""
    audio = np.atleast_2d(np.asarray(audio, dtype=np.float64))
    C, L = audio.shape
    n_fft, hop = out_grid(orig_sr)
    pad = np.zeros((C, padded_length(L, hop, n_fft)))
    pad[:, :L] = audio
    X = np.stack([mel_oracle.stft(a, n_fft, hop) for a in pad])
    lo, hi = band_edges(n_mels)
    psd = track_psd(mag, overlap_frames, lo, hi, orig_sr, n_fft, hop, X.shape[2])
    y = mwf(psd, X, iterations)
    K = y.shape[0]
    return np.stack([[mel_oracle.istft(y[k, c], hop)[:L] for c in range(C)] for k in range(K)]).astype(np.float64)
