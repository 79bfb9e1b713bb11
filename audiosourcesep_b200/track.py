"""Separating a whole recording from its mixture alone (``run_basis_sep --mix``).

The reference separates fixed 2.04 s extracts of a song whose stems it already has, skips the first two, drops the tail,
and concatenates 32256-sample inversions of 32640-sample extracts, so its output drifts 384 samples per extract behind
the input.  This module cuts the whole mixture into overlapping windows instead, and writes one track per source with
the input's sample count and rate, aligned sample for sample:

* the mixture is read (``read_wav_mono``) and resampled to 16 kHz on the device when its rate differs: x, L samples;
* segment i starts at s_i = i P and analyses the window [s_i, s_i + WINDOW) of x, zero-padded past the end, WINDOW =
  int(16000 * 2.04) = 32640 samples, exactly the reference's extract, through the same front end (STFT, mel dB with the
  per-segment ``top_db`` floor, clip);
* one window's iSTFT reconstructs SPAN = 512 * 63 = 32256 samples; neighbours share O = 512 * overlap_frames of them
  (0 <= overlap_frames <= 31, so at most two segments cover a sample), P = SPAN - O, and n_seg = 1 if L <= SPAN else
  1 + ceil((L - SPAN) / P);
* the back end (``invert_track``) maps the K separated mel spectrograms to STFT magnitudes (NNLS), applies the mixture's
  phase or the K-source Wiener filter, and writes each track in one pass that cross-fades neighbouring segments over the
  O samples they share (asep_istft_track); the tracks are then resampled back to the input's rate and cut to its length.

The numpy restatement is oracle/track_oracle.py.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

SR = 16000
HOP = 512
N_FFT = 2048
N_MELS = 96
FMIN, FMAX = 125.0, 7600.0
DB_MIN, DB_MAX = -100.0, 20.0
WINDOW = int(SR * 2.04)                   # 32640: the reference's extract
FRAMES = 1 + WINDOW // HOP                # 64 STFT frames per window
SPAN = HOP * (FRAMES - 1)                 # 32256 samples reconstructed per window
MAX_OVERLAP_FRAMES = (FRAMES - 2) // 2    # 31: at most two segments cover any sample


def check_overlap_frames(overlap_frames) -> int:
    o = int(overlap_frames)
    if o != overlap_frames or not 0 <= o <= MAX_OVERLAP_FRAMES:
        raise ValueError(f"--overlap_frames must be an integer in 0..{MAX_OVERLAP_FRAMES}, got {overlap_frames}")
    return o


def segment_hop(overlap_frames: int) -> int:
    """P: samples between the starts of two segments."""
    return SPAN - HOP * check_overlap_frames(overlap_frames)


def segment_starts(L: int, overlap_frames: int = 8) -> np.ndarray:
    """int64 [n_seg]: the 16 kHz start sample of every segment of a track of L samples."""
    P = segment_hop(overlap_frames)
    if L < 1:
        raise ValueError("the track is empty")
    n_seg = 1 if L <= SPAN else 1 + -(-(int(L) - SPAN) // P)
    return np.arange(n_seg, dtype=np.int64) * P


def read_track(path: str, device=None):
    """(x [L] float32 at 16 kHz on the device, the file's rate, the file's sample count): mono down-mix, resampled with
    kaiser_best when the file is at another rate, as the reference's librosa.load(sr=16000)."""
    from .datasets.data_loader import read_wav_mono
    from .resample import resample
    a, rate = read_wav_mono(path)
    if len(a) == 0:
        raise ValueError(f"{path}: no samples")
    return resample(a, int(rate), SR, device=device), int(rate), int(len(a))


def segment_track(x, overlap_frames: int = 8):
    """Front end of a whole track.  x: [L] 16 kHz samples (array or device tensor).  Returns (mixed, stft_mixture, starts):
    mixed float32 [n_seg, 96, 64, 1] dB mel patches and stft_mixture complex64 [n_seg, 1025, 64] on the device, starts
    int64 [n_seg] -- each window through exactly the per-extract front end of data_loader.get_song_extract_k."""
    import torch
    from . import _lib, melspec
    d = _lib.init(None)
    x = torch.as_tensor(x, dtype=torch.float32).to(torch.device("cuda", d)).reshape(-1)
    L = int(x.numel())
    starts = segment_starts(L, overlap_frames)
    pad = torch.zeros(int(starts[-1]) + WINDOW, dtype=torch.float32, device=x.device)
    pad[:L] = x
    win = pad.unfold(0, WINDOW, segment_hop(overlap_frames)).contiguous()
    assert win.shape[0] == len(starts), (tuple(win.shape), len(starts))
    S = melspec.stft(win, n_fft=N_FFT, hop_length=HOP)
    mel = melspec.melspectrogram_db(S, sr=SR, n_fft=N_FFT, n_mels=N_MELS, fmin=FMIN, fmax=FMAX, dbmin=DB_MIN, dbmax=DB_MAX)
    return mel.unsqueeze(-1).contiguous(), S, starts


def fix_length(audio, length: int):
    """librosa.util.fix_length on the last axis: cut or zero-pad to ``length`` samples."""
    import torch
    n = audio.shape[-1]
    if n > length:
        return audio[..., :length].contiguous()
    if n < length:
        return torch.nn.functional.pad(audio, (0, length - n))
    return audio


def invert_track(mel_estimates, stft_mixture, track_length: int, overlap_frames: int, wiener_filter: bool = False,
                 orig_sr: int = SR, orig_length: Optional[int] = None, iters: int = 300):
    """Back end of a whole track: mel_estimates [K, n_seg, 96, 64] (dB), stft_mixture complex [n_seg, 1025, 64] ->
    float32 [K, orig_length] device tensor at ``orig_sr``.

    NNLS mel -> STFT magnitudes, the mixture's phase or (``wiener_filter``, K > 1) the K-source Wiener filter, the track
    iSTFT with cross-faded segments at 16 kHz (``track_length`` samples), then resampling to ``orig_sr`` and the length fix
    to ``orig_length`` (default: track_length * orig_sr / 16000, rounded up)."""
    import torch
    from . import _lib, melspec
    from .resample import resample
    d = _lib.init(None)
    dev = torch.device("cuda", d)
    m = torch.as_tensor(np.asarray(mel_estimates) if not torch.is_tensor(mel_estimates) else mel_estimates,
                        dtype=torch.float32).to(dev)
    if m.ndim == 5 and m.shape[-1] == 1:
        m = m.squeeze(-1)
    if m.ndim != 4:
        raise ValueError(f"invert_track: mel_estimates must be [K, n_seg, n_mels, T], got {tuple(m.shape)}")
    K, n_seg, M, T = m.shape
    mix = torch.as_tensor(stft_mixture).to(dev).to(torch.complex64)
    if tuple(mix.shape) != (n_seg, N_FFT // 2 + 1, T):
        raise ValueError(f"invert_track: stft_mixture {tuple(mix.shape)} does not match {n_seg} segments of {T} frames")
    if len(segment_starts(int(track_length), overlap_frames)) != n_seg:
        raise ValueError(f"invert_track: {n_seg} segments do not tile a track of {track_length} samples at "
                         f"overlap_frames = {overlap_frames}")
    mags = melspec.mel_to_stft(m.reshape(K * n_seg, M, T), sr=SR, n_fft=N_FFT, fmin=FMIN, fmax=FMAX, iters=iters)
    cs = melspec.stft_filter(mags.reshape(K, n_seg, -1, T), mix, bool(wiener_filter) and K > 1)
    audio = melspec.istft_track(cs, overlap_frames, int(track_length), hop_length=HOP)
    orig_sr = int(orig_sr)
    if orig_length is None:
        orig_length = int(math.ceil(int(track_length) * orig_sr / SR))
    if orig_sr != SR:
        audio = resample(audio, SR, orig_sr, device=d)
    return fix_length(audio, int(orig_length))


def track_results(mel_estimates: Sequence[np.ndarray], mixed: np.ndarray, stft_mixture: np.ndarray, starts: np.ndarray,
                  track_length: int, orig_sr: int, orig_length: int, overlap_frames: int) -> Dict[str, np.ndarray]:
    """The arrays ``results.npz`` holds for a whole track: x1..xK, mixed, stft_mixture and the segmentation."""
    out = {f"x{k + 1}": np.asarray(x) for k, x in enumerate(mel_estimates)}
    out.update({"mixed": np.asarray(mixed), "stft_mixture": np.asarray(stft_mixture),
                "segment_start": np.asarray(starts, dtype=np.int64), "track_length": np.int64(track_length),
                "orig_sr": np.int64(orig_sr), "orig_length": np.int64(orig_length), "overlap_frames": np.int64(overlap_frames)})
    return out


def invert_results(res, wiener_filter: bool = False) -> np.ndarray:
    """invert_track on the contents of a whole-track ``results.npz``: float32 [K, orig_length] on the host."""
    K = sum(1 for k in res if k[0] == "x" and k[1:].isdigit())
    xs = np.stack([np.asarray(res[f"x{k + 1}"]) for k in range(K)])
    starts = np.asarray(res["segment_start"])
    o = int(res["overlap_frames"])
    if not np.array_equal(starts, segment_starts(int(res["track_length"]), o)):
        raise ValueError("segment_start does not match track_length and overlap_frames")
    audio = invert_track(xs, res["stft_mixture"], int(res["track_length"]), o, wiener_filter, int(res["orig_sr"]),
                         int(res["orig_length"]))
    return audio.cpu().numpy()


def write_tracks(out_dir: str, names: Sequence[str], tracks: np.ndarray, sr: int) -> None:
    """<out_dir>/<name>.wav (16-bit PCM at ``sr``) per source, and separated.npz with the float32 tracks x1..xK."""
    from .melspec_inversion_basis import write_wav
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(names, tracks):
        write_wav(os.path.join(out_dir, name + ".wav"), t, sr)
    np.savez(os.path.join(out_dir, "separated"), sr=np.int64(sr),
             **{f"x{k + 1}": np.asarray(t, dtype=np.float32) for k, t in enumerate(tracks)})


def separate_file(mix_path: str, restores: Sequence[str], output: str = "basis_sep", overlap_frames: int = 8,
                  wiener_filter: bool = False, **options) -> Tuple[Dict[str, np.ndarray], int]:
    """Separate the wav file ``mix_path`` with one prior per restore directory (K = len(restores), 2..8) without the CLI:
    run_basis_sep --mix.  ``options`` are any other run_basis_sep flags by their argument name (``model_type="glow"``,
    ``config=...``, ``random_init=3``, ``sources="bass,drums"``, ``T=...``).  Writes ``output`` as the CLI does and returns
    ({source name: float32 track}, rate)."""
    from . import run_basis_sep
    if len(restores) < 2:
        raise ValueError("BASIS needs at least two priors")
    parser = run_basis_sep.build_parser()
    args = parser.parse_args(list(restores))
    for key, value in options.items():
        if not hasattr(args, key):
            raise TypeError(f"separate_file: unknown option {key!r}")
        setattr(args, key, value)
    args.mix, args.output = mix_path, output
    args.overlap_frames, args.wiener_filter = overlap_frames, bool(wiener_filter)
    res = run_basis_sep.main(args)
    if res is None:                                # not rank 0
        return {}, 0
    return res["separated"], int(res["orig_sr"])
