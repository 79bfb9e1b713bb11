"""Inversion of the separated mel spectrograms to audio -- mirror of the reference's ``melspec_inversion_basis.py``
(``stft_inversion_fn`` :42-90, ``single_channel_wiener_filter`` :93-119, ``main`` :122-236): reads ``results.npz`` of a
BASIS run, inverts x1 / x2 / gt1 / gt2 / mixed with the mixture's phase (optionally through the single-channel Wiener
filter) and writes ``inverse_spectrograms.npz`` + 16-bit wav files.  The transforms run on the GPU (melspec.py).
``--algorithm griffin`` runs Griffin-Lim (:21-39; 32 iterations, momentum 0.99) on the same STFT / iSTFT kernels.
Results of ``run_basis_sep --mix`` (a ``segment_start`` key) are inverted as whole tracks instead (track.invert_track)."""
from __future__ import annotations

import argparse
import os
import re
import time
import wave

import numpy as np
import torch

from . import melspec


def single_channel_wiener_filter(psd_sources, stft_mixture):
    """reference: :93-119 -- psd_sources [S, N, F, T] (power), stft_mixture complex [N, F, T]."""
    psd = torch.as_tensor(psd_sources)
    assert psd.ndim >= 3 and psd.shape[0] > 1, tuple(psd.shape)
    return melspec.stft_filter(torch.sqrt(psd.float().cuda()), torch.as_tensor(stft_mixture).cuda(), True)


def stft_inversion_fn(sr=16000, fmin=125, fmax=7600, n_fft=2048, hop_length=512, scale="dB", wiener_filter=False, iters=300):
    if scale != "dB":
        raise NotImplementedError("only the dB scale of the configs is rebuilt")

    def stft_inversion(inputs):
        """inputs = (melspecs, stft_mixture): melspecs a list of S arrays [N, n_mels, T] (dB), stft_mixture complex
        [N, F, T].  Returns a list of S float32 arrays [N, hop (T-1)] (one waveform per extract)."""
        melspecs, stft_mixture = inputs
        n_src = len(melspecs)
        use_wiener = wiener_filter and n_src > 1                                   # :59
        mix = torch.as_tensor(np.asarray(stft_mixture)).to(torch.complex64).cuda()
        mags = torch.stack([melspec.mel_to_stft(torch.as_tensor(np.asarray(m, dtype=np.float32)), sr=sr, n_fft=n_fft, fmin=fmin,
                                                fmax=fmax, iters=iters) for m in melspecs])
        cs = melspec.stft_filter(mags, mix, use_wiener)
        return [melspec.istft(c, hop_length).cpu().numpy() for c in cs]

    return stft_inversion


def griffin_inversion_fn(sr=16000, fmin=125, fmax=7600, n_fft=2048, hop_length=512, scale="dB", n_iter=32, seed=0):
    """reference: :21-39 -- librosa.feature.inverse.mel_to_audio = mel_to_stft (NNLS) followed by Griffin-Lim (32
    iterations, momentum 0.99, random initial phase)."""
    if scale != "dB":
        raise NotImplementedError("only the dB scale of the configs is rebuilt")

    def griffin_inversion(melspecs):
        """melspecs: list of arrays [N, n_mels, T] (dB) -> list of float32 arrays [N, hop (T-1)]."""
        out = []
        for m in melspecs:
            mag = melspec.mel_to_stft(torch.as_tensor(np.asarray(m, dtype=np.float32)), sr=sr, n_fft=n_fft, fmin=fmin, fmax=fmax)
            out.append(melspec.griffinlim(mag, n_iter=n_iter, hop_length=hop_length, seed=seed).cpu().numpy())
        return out

    return griffin_inversion


def write_wav(path: str, data: np.ndarray, samplerate: int) -> None:
    pcm = np.clip(np.asarray(data, dtype=np.float64), -1.0, 1.0 - 1.0 / 32768.0)
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(int(samplerate))
        w.writeframes((pcm * 32768.0).astype("<i2").tobytes())


def main(args):
    sr, fmin, fmax, n_fft, hop_length = 16000, 125, 7600, 2048, 512
    res = np.load(os.path.join(args.basis_results, "results.npz"))
    out_dir = args.output or os.path.join(args.basis_results, "inverse_" + args.algorithm + "_" + args.method + ("_wiener_filter" if args.wiener_filter else ""))
    os.makedirs(out_dir, exist_ok=True)
    if args.algorithm not in ("reuse_phase", "griffin"):
        raise ValueError("method should be griffin or reuse_phase")                 # :197-198
    K = sum(1 for k in res.files if re.fullmatch(r"x[0-9]+", k))                   # one x{k} / gt{k} pair per source
    if "segment_start" in res.files:                                               # a whole track (run_basis_sep --mix)
        return _main_track(args, res, out_dir, K)
    xs = [res[f"x{k + 1}"] for k in range(K)]
    gts = [res[f"gt{k + 1}"] for k in range(K)]
    mix, stft_mixture = res["mixed"], res["stft_mixture"]
    assert all(x.ndim == 3 for x in xs) and stft_mixture.ndim == 3, ([x.shape for x in xs], stft_mixture.shape)
    if args.method == "whole":                                                     # :164-170: one long spectrogram
        cat = lambda a: np.concatenate(list(a), axis=-1)[None]
        xs, gts, mix, stft_mixture = [cat(a) for a in xs], [cat(a) for a in gts], cat(mix), cat(stft_mixture)
    t0 = time.time()
    if args.algorithm == "griffin":                                                # :173-183
        gfn = griffin_inversion_fn(sr, fmin, fmax, n_fft, hop_length, args.scale)
        x_inv = gfn(xs)
        gt_inv = gfn(gts)
        mix_inv = gfn([mix])[0]
    else:
        fn = stft_inversion_fn(sr, fmin, fmax, n_fft, hop_length, args.scale, args.wiener_filter)
        x_inv = fn((xs, stft_mixture))
        gt_inv = fn((gts, stft_mixture))
        mix_inv = fn(([mix], stft_mixture))[0]
    torch.cuda.synchronize()
    print("Inversion duration: {} seconds".format(round(time.time() - t0, 4)))
    items = [(f"x{k + 1}_audio", x_inv[k]) for k in range(K)] + [(f"gt{k + 1}_audio", gt_inv[k]) for k in range(K)]
    flat = {k: np.concatenate(list(v), axis=-1) for k, v in items + [("mix_audio", mix_inv)]}
    names = [(f"sep{k + 1}", f"x{k + 1}_audio") for k in range(K)] + [(f"gt{k + 1}", f"gt{k + 1}_audio") for k in range(K)]
    for name, key in names + [("mix", "mix_audio")]:
        write_wav(os.path.join(out_dir, name + ".wav"), flat[key], sr)
    np.savez(os.path.join(out_dir, "inverse_spectrograms"), **flat)
    return flat


def _main_track(args, res, out_dir, K):
    """Results of ``run_basis_sep --mix``: every x{k} is inverted as one full-length track (track.invert_track: segments
    cross-faded, resampled back to the input's rate and length) and written as sep{k}.wav, with the float32 tracks in
    separated.npz.  gt{k} keys are not needed; --method does not apply (the track is always inverted whole)."""
    from . import track
    if args.algorithm != "reuse_phase":
        raise ValueError("a whole track is inverted with the mixture's phase (reuse_phase); Griffin-Lim draws random phases per "
                         "segment, which do not cross-fade coherently")
    t0 = time.time()
    tracks = track.invert_results({k: res[k] for k in res.files}, args.wiener_filter)
    torch.cuda.synchronize()
    print("Inversion duration: {} seconds".format(round(time.time() - t0, 4)))
    track.write_tracks(out_dir, [f"sep{k + 1}" for k in range(K)], tracks, int(res["orig_sr"]))
    return {f"x{k + 1}_audio": tracks[k] for k in range(K)}


def build_parser():
    p = argparse.ArgumentParser(description="Spectrograms Inversion")
    p.add_argument("basis_results", type=str)
    p.add_argument("--output", type=str, default=None)
    p.add_argument("--algorithm", type=str, default="reuse_phase", help="griffin or reuse_phase")
    p.add_argument("--method", type=str, default="frame", help="frame or whole")
    p.add_argument("--scale", type=str, default="dB")
    p.add_argument("--wiener_filter", action="store_true")
    p.add_argument("--debug", action="store_true")
    return p


if __name__ == "__main__":
    main(build_parser().parse_args())
