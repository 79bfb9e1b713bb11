"""CPU ORACLE (test infrastructure, NOT a product path) -- separating a whole track from its mixture alone.

numpy restatement of audiosourcesep_b200/track.py and of asep_istft_track (csrc/mel_kernels.cu: k_overlap_add_track):
  * the mixture x (16 kHz, L samples) is cut into windows of Wn = int(16000 * 2.04) = 32640 samples, the extract of the
    reference's front end, starting at s_i = i P; the window is zero-padded past the end of x;
  * one window's iSTFT (hop 512, T = 64 frames) reconstructs V = 512 * 63 = 32256 samples; neighbours overlap by
    O = 512 o samples (o = overlap_frames, 0 <= o <= 31, so at most two segments cover a sample), P = V - O;
  * n_seg = 1 if L <= V else 1 + ceil((L - V) / P): nothing is skipped and nothing is dropped;
  * sample n of the track is sum_i c_i(n) u_i(n - s_i) / sum_i c_i(n) over the segments covering n, with u_i segment i's
    iSTFT (mel_oracle.istft, in float64) and c_i a linear cross-fade over the O samples segment i shares with a neighbour
    (1 elsewhere, no ramp at either end of the track).
"""
from __future__ import annotations

import numpy as np

from . import mel_oracle

SR = 16000
HOP = 512
N_FFT = 2048
WINDOW = int(SR * 2.04)                   # 32640
FRAMES = 1 + WINDOW // HOP                # 64
SPAN = HOP * (FRAMES - 1)                 # 32256
MAX_OVERLAP_FRAMES = (FRAMES - 2) // 2    # 31


def segment_starts(L: int, overlap_frames: int = 8) -> np.ndarray:
    """int64 [n_seg] start sample of every segment of a track of L samples (16 kHz)."""
    if not 0 <= overlap_frames <= MAX_OVERLAP_FRAMES:
        raise ValueError(overlap_frames)
    P = SPAN - HOP * overlap_frames
    n_seg = 1 if L <= SPAN else 1 + -(-(L - SPAN) // P)
    return np.arange(n_seg, dtype=np.int64) * P


def windows(x: np.ndarray, overlap_frames: int = 8) -> np.ndarray:
    """[n_seg, WINDOW] analysis windows of the track x, zero-padded at the end."""
    starts = segment_starts(len(x), overlap_frames)
    pad = np.zeros(int(starts[-1]) + WINDOW, dtype=np.float64)
    pad[: len(x)] = x
    return np.stack([pad[s: s + WINDOW] for s in starts])


def crossfade_weights(L: int, overlap_frames: int = 8) -> np.ndarray:
    """float64 [n_seg, L]: c_i(n), zero where segment i does not cover sample n."""
    starts = segment_starts(L, overlap_frames)
    n_seg, O = len(starts), HOP * overlap_frames
    c = np.zeros((n_seg, L))
    for i, s in enumerate(starts):
        j = np.arange(SPAN, dtype=np.float64)
        w = np.ones(SPAN)
        if i > 0 and O > 0:
            w[:O] = (j[:O] + 0.5) / O
        if i < n_seg - 1 and O > 0:
            w[SPAN - O:] = (SPAN - j[SPAN - O:] - 0.5) / O
        hi = min(L, int(s) + SPAN)
        c[i, s:hi] = w[: hi - s]
    return c


def istft64(S: np.ndarray, hop: int = HOP) -> np.ndarray:
    """mel_oracle.istft without the final float32 cast."""
    n_fft = 2 * (S.shape[0] - 1)
    T = S.shape[1]
    w = mel_oracle.hann_periodic(n_fft)
    y = np.zeros(n_fft + hop * (T - 1))
    wss = np.zeros_like(y)
    frames = np.fft.irfft(S.astype(np.complex128), n=n_fft, axis=0)
    for t in range(T):
        y[t * hop: t * hop + n_fft] += w * frames[:, t]
        wss[t * hop: t * hop + n_fft] += w ** 2
    nz = wss > np.finfo(np.float32).tiny
    y[nz] /= wss[nz]
    return y[n_fft // 2: len(y) - n_fft // 2]


def istft_track(stfts: np.ndarray, overlap_frames: int, L: int, hop: int = HOP) -> np.ndarray:
    """stfts complex [n_seg, F, FRAMES] of one track's segments -> float64 [L]: the cross-faded overlap of their iSTFTs."""
    starts = segment_starts(L, overlap_frames)
    assert stfts.shape[0] == len(starts), (stfts.shape, len(starts))
    c = crossfade_weights(L, overlap_frames)
    num, den = np.zeros(L), np.zeros(L)
    for i, s in enumerate(starts):
        u = istft64(stfts[i], hop)
        hi = min(L, int(s) + len(u))
        num[s:hi] += c[i, s:hi] * u[: hi - s]
        den[s:hi] += c[i, s:hi]
    return num / den
