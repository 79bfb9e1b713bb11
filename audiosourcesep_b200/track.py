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
  These are the ``mel`` rendering's stems: mono, limited to the mel band (133 Hz .. 7.6 kHz), and they need not sum to
  the input;
* the ``mask`` rendering (``render_track``, ``--render mask``) instead turns the same NNLS magnitudes into per-source
  powers on an STFT grid of the original recording (asep_track_psd) and applies a multichannel Wiener filter with EM and
  mixture consistency to that recording's own STFT (asep_mwf): the stems keep the input's channels (1 or 2), rate and
  full band, and sum to the input.  Outside the mel band every frame takes the gains of the nearest covered bin.

The numpy restatements are oracle/track_oracle.py and oracle/mwf_oracle.py.
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
MAX_CHANNELS = 2                          # the mask rendering's spatial model is C x C, C = 1 or 2
MAX_MWF_ITERATIONS = 10                   # asep_mwf keeps every EM iteration's spatial covariances in shared memory


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


def read_track_channels(path: str) -> Tuple[np.ndarray, int]:
    """(audio float32 [C, L] at the file's rate, the rate): every channel of the file, C = 1 or 2, for the mask rendering."""
    from .datasets.data_loader import read_wav
    a, rate = read_wav(path)
    if a.shape[0] > MAX_CHANNELS:
        raise ValueError(f"{path}: {a.shape[0]} channels; the mask rendering handles mono and stereo recordings")
    if a.shape[1] == 0:
        raise ValueError(f"{path}: no samples")
    return np.ascontiguousarray(a), int(rate)


def out_grid(orig_sr: int) -> Tuple[int, int]:
    """(n_fft, hop) of the mask rendering's STFT at ``orig_sr``: the 2048 / 512 mel grid scaled to the rate, n_fft rounded
    to a power of two in 256..4096, hop = n_fft / 4 (2048 / 512 at 16 kHz, 4096 / 1024 at 44.1 and 48 kHz)."""
    n = 2 ** int(round(math.log2(N_FFT * float(orig_sr) / SR)))
    n = min(4096, max(256, n))
    return n, n // 4


def check_mwf_iterations(iterations) -> int:
    n = int(iterations)
    if n != iterations or not 0 <= n <= MAX_MWF_ITERATIONS:
        raise ValueError(f"--mwf_iterations must be an integer in 0..{MAX_MWF_ITERATIONS}, got {iterations}")
    return n


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


def _mel_estimates(mel_estimates, dev):
    import torch
    m = torch.as_tensor(np.asarray(mel_estimates) if not torch.is_tensor(mel_estimates) else mel_estimates,
                        dtype=torch.float32).to(dev)
    if m.ndim == 5 and m.shape[-1] == 1:
        m = m.squeeze(-1)
    if m.ndim != 4:
        raise ValueError(f"mel_estimates must be [K, n_seg, n_mels, T], got {tuple(m.shape)}")
    return m


def _check_tiling(n_seg: int, track_length: int, overlap_frames: int) -> None:
    if len(segment_starts(int(track_length), overlap_frames)) != n_seg:
        raise ValueError(f"{n_seg} segments do not tile a track of {track_length} samples at overlap_frames = {overlap_frames}")


def render_track(mel_estimates, track_length: int, overlap_frames: int, audio, orig_sr: int, iterations: int = 1,
                 iters: int = 300):
    """Mask rendering of a whole track: mel_estimates [K, n_seg, 96, 64] (dB) of a track of ``track_length`` 16 kHz
    samples and the original recording audio [C, L] (C = 1 or 2) at ``orig_sr`` -> float32 [K, C, L] device tensor.

    NNLS mel -> STFT magnitudes as invert_track, then the sources' powers on the STFT grid of the recording (out_grid;
    asep_track_psd), the multichannel Wiener filter with ``iterations`` EM steps on the recording's STFT (asep_mwf) and
    the iSTFT of every source and channel.  The stems sum to ``audio``."""
    import torch
    from . import _lib, melspec
    d = _lib.init(None)
    dev = torch.device("cuda", d)
    m = _mel_estimates(mel_estimates, dev)
    K, n_seg, M, T = m.shape
    _check_tiling(n_seg, track_length, overlap_frames)
    n_iter = check_mwf_iterations(iterations)
    a = torch.as_tensor(np.asarray(audio) if not torch.is_tensor(audio) else audio, dtype=torch.float32).to(dev)
    if a.ndim == 1:
        a = a[None]
    if a.ndim != 2 or not 1 <= a.shape[0] <= MAX_CHANNELS or a.shape[1] < 1:
        raise ValueError(f"render_track: audio must be [C, L] with C = 1 or 2, got {tuple(a.shape)}")
    C, L = a.shape
    mags = melspec.mel_to_stft(m.reshape(K * n_seg, M, T), sr=SR, n_fft=N_FFT, fmin=FMIN, fmax=FMAX, iters=iters)
    n_fft, hop = out_grid(int(orig_sr))
    pad = torch.zeros((C, max(-(-L // hop) * hop, n_fft)), dtype=torch.float32, device=dev)   # reflect padding needs > n_fft/2
    pad[:, :L] = a
    X = melspec.stft(pad, n_fft=n_fft, hop_length=hop)
    lo, hi = melspec.band_edges(SR, N_FFT, M, FMIN, FMAX)
    psd = melspec.track_psd(mags.reshape(K, n_seg, -1, T), overlap_frames, lo, hi, int(orig_sr), n_fft, hop, X.shape[2],
                            hop_length=HOP)
    Y = melspec.mwf(psd, X, n_iter)
    out = melspec.istft(Y.reshape((K * C,) + tuple(Y.shape[2:])), hop)
    return out[:, :L].reshape(K, C, L)


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
    m = _mel_estimates(mel_estimates, dev)
    K, n_seg, M, T = m.shape
    mix = torch.as_tensor(stft_mixture).to(dev).to(torch.complex64)
    if tuple(mix.shape) != (n_seg, N_FFT // 2 + 1, T):
        raise ValueError(f"invert_track: stft_mixture {tuple(mix.shape)} does not match {n_seg} segments of {T} frames")
    _check_tiling(n_seg, track_length, overlap_frames)
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


def _results_estimates(res):
    K = sum(1 for k in res if k[0] == "x" and k[1:].isdigit())
    xs = np.stack([np.asarray(res[f"x{k + 1}"]) for k in range(K)])
    o = int(res["overlap_frames"])
    if not np.array_equal(np.asarray(res["segment_start"]), segment_starts(int(res["track_length"]), o)):
        raise ValueError("segment_start does not match track_length and overlap_frames")
    return xs, o


def invert_results(res, wiener_filter: bool = False) -> np.ndarray:
    """invert_track on the contents of a whole-track ``results.npz``: float32 [K, orig_length] on the host."""
    xs, o = _results_estimates(res)
    audio = invert_track(xs, res["stft_mixture"], int(res["track_length"]), o, wiener_filter, int(res["orig_sr"]),
                         int(res["orig_length"]))
    return audio.cpu().numpy()


def render_results(res, mix_path: str, iterations: int = 1, audio: Optional[Tuple[np.ndarray, int]] = None) -> np.ndarray:
    """render_track on the contents of a whole-track ``results.npz`` and the recording it was separated from: float32
    [K, C, orig_length] on the host.  ``audio``: the recording as read_track_channels(mix_path) returns it, if already read.
    The file must have the rate and length the results were made from (``orig_sr``, ``orig_length``)."""
    xs, o = _results_estimates(res)
    a, rate = read_track_channels(mix_path) if audio is None else audio
    if rate != int(res["orig_sr"]) or a.shape[1] != int(res["orig_length"]):
        raise ValueError(f"{mix_path}: {a.shape[1]} samples at {rate} Hz, but the results were separated from "
                         f"{int(res['orig_length'])} samples at {int(res['orig_sr'])} Hz")
    return render_track(xs, int(res["track_length"]), o, a, rate, iterations).cpu().numpy()


def write_tracks(out_dir: str, names: Sequence[str], tracks: np.ndarray, sr: int) -> None:
    """<out_dir>/<name>.wav (16-bit PCM at ``sr``) per source, and separated.npz with the float32 tracks x1..xK.  A track
    is [L] (mono) or [C, L] (C channels)."""
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
    ``config=...``, ``random_init=3``, ``sources="bass,drums"``, ``T=...``, ``render="mask"``, ``mwf_iterations=2``).
    Writes ``output`` as the CLI does and returns ({source name: float32 track}, rate); a track is [L] with the default
    ``render="mel"`` and [C, L] with ``render="mask"``."""
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
