"""The mask rendering of a whole track (run_basis_sep --mix --render mask) on one GPU.

    python tools/mask_render_bench.py --out <dir>

A seeded 3-minute 44.1 kHz stereo recording (tones, a chirp, a bass line, a 12 kHz tone and noise) goes through the front
end; K separated mel estimates are made from its mel patches (the mixture's, offset and perturbed per source, as
tools/track_sep_bench.py does).  For K in {2, 4, 8} and EM iterations n in {0, 1, 3}:
1. k_track_psd (asep_track_psd) and k_mwf (asep_mwf) alone: CUDA events around `reps` launches after a warm-up launch;
   each kernel's algorithmic bytes (track_psd: the segment magnitudes read once + the PSD written; mwf: (n + 1)(C 8 + K 4) B
   read and K C 8 B written per bin) over its time, and the least time the 7.7 TB/s HBM data-sheet bandwidth allows for
   those bytes over the measured time.  The PSD and the STFT of 8 sources exceed the 126 MB L2; at K = 2 part of them fits;
2. the whole mask back end (track.render_track: NNLS, the recording's STFT, both kernels, iSTFT): host clock around a
   call that ends in a device synchronise, median of `reps` after a warm-up;
3. the existing mel back end (track.invert_track, mixture phase: the CLI's default rendering) on the same estimates, timed
   the same way, for comparison (it depends on K only).
The card's name and power limit are recorded beside the numbers.  Writes <out>/mask_render_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audiosourcesep_b200 import _lib, melspec, track  # noqa: E402
from audiosourcesep_b200.resample import resample  # noqa: E402

SR_IN, SECONDS, OVERLAP = 44100, 180, 8
HBM_BPS = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def recording():
    rng = np.random.default_rng(0)
    n = SR_IN * SECONDS
    t = np.arange(n) / SR_IN
    x = (0.2 * np.sin(2 * np.pi * 220 * t) * (1 + 0.5 * np.sin(2 * np.pi * 0.5 * t))
         + 0.15 * np.sin(2 * np.pi * 660 * t + 0.3 * np.sin(2 * np.pi * 5 * t))
         + 0.05 * np.sin(2 * np.pi * (100 + 20 * t) * t) + 0.1 * np.sin(2 * np.pi * 55 * t)
         + 0.02 * np.sin(2 * np.pi * 12000 * t) + 0.01 * rng.standard_normal(n))
    return np.stack([x, 0.8 * x + 0.01 * rng.standard_normal(n)]).astype(np.float32)


def clock(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def events(fn, reps):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def roofline(nbytes, ms):
    return {"ms": ms, "algorithmic_bytes": nbytes, "GBps": nbytes / (ms * 1e-3) / 1e9,
            "hbm_bound_share": nbytes / HBM_BPS / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    d = _lib.init()
    dev = torch.device("cuda", d)
    audio = recording()
    C, L = audio.shape
    x16 = resample(audio.mean(axis=0), SR_IN, track.SR)
    mel, S16, starts = track.segment_track(x16, OVERLAP)
    mel = mel.squeeze(-1)
    L16, n_seg = int(x16.numel()), len(starts)
    n_fft, hop = track.out_grid(SR_IN)
    a = torch.as_tensor(audio).to(dev)
    pad = torch.zeros((C, max(-(-L // hop) * hop, n_fft)), device=dev)
    pad[:, :L] = a
    X = melspec.stft(pad, n_fft=n_fft, hop_length=hop)
    F, T = X.shape[1], X.shape[2]
    lo, hi = melspec.band_edges()
    out = {"card": card(), "input": f"{SECONDS} s, {SR_IN} Hz, {C} channels", "overlap_frames": OVERLAP, "segments": n_seg,
           "grid": {"n_fft": n_fft, "hop": hop, "bins": F, "frames": T, "bins_x_frames": F * T}, "hbm_TBps": HBM_BPS / 1e12,
           "rows": {}}
    for K in (2, 4, 8):
        g = torch.Generator(device="cuda").manual_seed(K)
        ests = torch.stack([(mel - 6.0 * k + torch.randn(mel.shape, device=dev, generator=g)).clamp(-100, 20)
                            for k in range(K)])
        mags = melspec.mel_to_stft(ests.reshape(K * n_seg, track.N_MELS, -1)).reshape(K, n_seg, -1, track.FRAMES)
        psd = melspec.track_psd(mags, OVERLAP, lo, hi, SR_IN, n_fft, hop, T)
        ms_psd = events(lambda: melspec.track_psd(mags, OVERLAP, lo, hi, SR_IN, n_fft, hop, T), args.reps)
        psd_bytes = mags.numel() * 4 + K * F * T * 4
        mel_ms = float(np.median([clock(lambda: track.invert_track(ests, S16, L16, OVERLAP, orig_sr=SR_IN, orig_length=L))[1]
                                  for _ in range(args.reps + 1)][1:]))
        for n in (0, 1, 3):
            ms_mwf = events(lambda: melspec.mwf(psd, X, n), args.reps)
            mwf_bytes = F * T * ((n + 1) * (C * 8 + K * 4) + K * C * 8)
            run = lambda: track.render_track(ests, L16, OVERLAP, a, SR_IN, n)
            times = [clock(run)[1] for _ in range(args.reps + 1)][1:]
            y = run()
            row = {"K": K, "iterations": n, "k_track_psd": roofline(psd_bytes, ms_psd), "k_mwf": roofline(mwf_bytes, ms_mwf),
                   "mask_back_end_ms": float(np.median(times)), "mel_back_end_ms": mel_ms,
                   "stems_sum_to_input_max_abs_err": float((y.sum(0) - a).abs().max()),
                   "finite": bool(torch.isfinite(y).all())}
            out["rows"][f"K{K}_n{n}"] = row
            print(json.dumps(row), flush=True)
        del ests, mags, psd
        torch.cuda.empty_cache()
    out["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "mask_render_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"card": out["card"]}))


if __name__ == "__main__":
    main()
