"""Whole-track separation (run_basis_sep --mix) on one GPU: where the time goes for a 3-minute recording.

    python tools/track_sep_bench.py --out <dir>

A seeded 3-minute 44.1 kHz stereo 24-bit mixture (tones, a chirp and noise) is written to a temporary wav file, then:
1. front end: reading and decoding the file, resampling to 16 kHz, STFT and mel dB of the n_seg overlapping segments
   (overlap_frames = 8) -- host clock around each part, each ending in a device synchronise; median of 5 after a warm-up;
2. BASIS at that segment count, K = 2 and K = 4 sources, with NCSN v2 (128 filters) and Glow (K_flow = 40, 512 filters)
   priors in bf16 (random init; a 10-level sigma schedule: the cost of a step does not depend on the level): ms per
   Langevin step, CUDA events around `calls` library calls of T = 8 steps after one warm-up call;
3. back end for K = 2 and 4 (Wiener filter): invert_track end to end (host clock, median of 5), and its kernels split by
   torch.profiler in a separate run: NNLS (k_nnls), filter (k_stft_filter), iSTFT frames (k_istft_frames), track kernel
   (k_overlap_add_track) and resampling back to 44.1 kHz (k_resample); the track kernel's algorithmic bytes (frames read +
   samples written) over its time;
4. seconds of compute per minute of audio for the full schedules of the shipped configs (NCSN v2: 200 levels x T = 8,
   Glow: 10 levels x T = 100): (front end + steps x ms/step + back end) / 3.
The card's name and power limit are recorded beside the numbers.  Writes <out>/track_sep_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import wave

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audiosourcesep_b200 import GlowConfig, NCSNConfig, _lib, melspec, ops, track  # noqa: E402
from audiosourcesep_b200.datasets.data_loader import read_wav_mono  # noqa: E402
from audiosourcesep_b200.glow import Glow  # noqa: E402
from audiosourcesep_b200.ncsn.score_model import ScoreModel  # noqa: E402
from audiosourcesep_b200.resample import resample  # noqa: E402
from audiosourcesep_b200.weights import init_glow_params, init_ncsn_params  # noqa: E402
from oracle import basis_oracle as bo  # noqa: E402

SR_IN, SECONDS = 44100, 180
FULL_STEPS = {"ncsn_v2_bf16": 200 * 8, "glow_bf16": 10 * 100}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def write_mixture(path):
    rng = np.random.default_rng(0)
    n = SR_IN * SECONDS
    t = np.arange(n) / SR_IN
    x = (0.2 * np.sin(2 * np.pi * 220 * t) * (1 + 0.5 * np.sin(2 * np.pi * 0.5 * t))
         + 0.15 * np.sin(2 * np.pi * 660 * t + 0.3 * np.sin(2 * np.pi * 5 * t))
         + 0.05 * np.sin(2 * np.pi * (100 + 20 * t) * t) + 0.01 * rng.standard_normal(n))
    st = np.stack([x, 0.8 * x + 0.01 * rng.standard_normal(n)], axis=1).reshape(-1)
    pcm = np.round(np.clip(st, -1, 1 - 2 ** -23) * 2 ** 23).astype("<i4")
    with wave.open(path, "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(3)
        w.setframerate(SR_IN)
        w.writeframes(pcm.view(np.uint8).reshape(-1, 4)[:, :3].tobytes())
    return n


def clock(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def front_end(path, reps=5):
    rows = []
    for _ in range(reps + 1):
        (a, rate), t_read = clock(lambda: read_wav_mono(path))
        x, t_res = clock(lambda: resample(a, rate, track.SR))
        starts = track.segment_starts(int(x.numel()), 8)
        pad = torch.zeros(int(starts[-1]) + track.WINDOW, device=x.device)
        pad[: x.numel()] = x
        win = pad.unfold(0, track.WINDOW, track.segment_hop(8)).contiguous()
        S, t_stft = clock(lambda: melspec.stft(win, n_fft=track.N_FFT, hop_length=track.HOP))
        mel, t_mel = clock(lambda: melspec.melspectrogram_db(S, fmin=track.FMIN, fmax=track.FMAX))
        rows.append((t_read, t_res, t_stft, t_mel))
    med = np.median(np.array(rows[1:]), axis=0)
    out = {"read_decode_ms": med[0], "resample_ms": med[1], "stft_ms": med[2], "mel_db_ms": med[3], "total_ms": float(med.sum())}
    return {k: float(v) for k, v in out.items()}, x, mel, S, starts


def basis_rows(kind, mixed, Ks, T, calls):
    n = mixed.shape[0]
    rows = {}
    for K in Ks:
        if kind == "glow_bf16":
            cfg = GlowConfig(K=40, minval=0.0, maxval=1.0)
            models = [Glow(cfg, init_glow_params(cfg, seed=2 + k), precision=_lib.PREC_BF16) for k in range(K)]
            sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
        else:
            ncfg = NCSNConfig(version="v2", ngf=128, num_classes=10, sigma1=1.0)
            sig = bo.get_sigmas(ncfg.sigma1, ncfg.sigmaL, ncfg.num_classes, "logarithmic")
            models = [ScoreModel(ncfg, init_ncsn_params(ncfg, seed=11 + k), sigmas=sig, precision=_lib.PREC_BF16)
                      for k in range(K)]
        eta, lam, ns = bo.step_constants(sig, 5)
        x = torch.rand((K,) + tuple(mixed.shape), device="cuda", generator=torch.Generator(device="cuda").manual_seed(K))
        step = [0]

        def call():
            if kind == "glow_bf16":
                ops.basis_glow_inner_k(models, mixed, x, T, float(eta), float(lam), float(ns), seed=1, step0=step[0])
            else:
                ops.basis_ncsn_inner_k(models, mixed, x, 5, T, float(eta), float(lam), float(ns), seed=1, step0=step[0])
            step[0] += T

        call()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            call()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b) / (calls * T)
        rows[str(K)] = {"ms_per_langevin_step": ms, "segments": n, "segment_steps_per_s": n / (ms * 1e-3),
                        "timed_steps": calls * T, "finite": bool(torch.isfinite(x).all())}
        print(kind, K, f"{n} segments: {ms:.2f} ms/step", flush=True)
        del models, x
        torch.cuda.empty_cache()
    return rows


KERNELS = {"nnls": "k_nnls", "filter": "k_stft_filter", "istft_frames": "k_istft_frames", "track_kernel": "k_overlap_add_track",
           "resample": "k_resample"}


def back_end(mel, S, L16, orig_length, K, reps=5):
    g = torch.Generator(device="cuda").manual_seed(K)
    ests = torch.stack([(mel - 6.0 * k + torch.randn(mel.shape, device="cuda", generator=g)).clamp(-100, 20)
                        for k in range(K)])
    run = lambda: track.invert_track(ests, S, L16, 8, wiener_filter=True, orig_sr=SR_IN, orig_length=orig_length)
    times = [clock(run)[1] for _ in range(reps + 1)][1:]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run()
        torch.cuda.synchronize()
    split = {k: 0.0 for k in KERNELS}
    for ev in prof.key_averages():
        for k, name in KERNELS.items():
            if name in ev.key:
                split[k] += getattr(ev, "device_time_total", 0.0) / 1e3
    n_seg = S.shape[0]
    track_bytes = K * n_seg * 64 * track.N_FFT * 4 + K * L16 * 4        # frames read once + samples written
    row = {"total_ms": float(np.median(times)), "kernel_ms_profiled": split,
           "track_kernel_algorithmic_bytes": track_bytes,
           "track_kernel_GBps": track_bytes / (split["track_kernel"] * 1e-3) / 1e9 if split["track_kernel"] > 0 else None,
           "output_shape": list(out.shape), "finite": bool(torch.isfinite(out).all())}
    print("back end", K, json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--T", type=int, default=8)
    ap.add_argument("--calls", type=int, default=3)
    args = ap.parse_args()
    _lib.init()
    out = {"card": card(), "input": f"{SECONDS} s, {SR_IN} Hz, stereo, 24-bit PCM", "overlap_frames": 8}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "mix.wav")
        n = write_mixture(path)
        out["front_end"], x, mel, S, starts = front_end(path)
    L16 = int(x.numel())
    out["track_length_16k"], out["segments"] = L16, len(starts)
    print("front end", json.dumps(out["front_end"]), len(starts), "segments", flush=True)
    mixed = ((mel - track.DB_MIN) / (track.DB_MAX - track.DB_MIN)).unsqueeze(-1).contiguous()
    out["basis"] = {kind: basis_rows(kind, mixed, (2, 4), args.T, args.calls) for kind in ("ncsn_v2_bf16", "glow_bf16")}
    out["back_end"] = {str(K): back_end(mel, S, L16, n, K) for K in (2, 4)}
    per_min = {}
    for kind, steps in FULL_STEPS.items():
        for K in ("2", "4"):
            total_ms = out["front_end"]["total_ms"] + steps * out["basis"][kind][K]["ms_per_langevin_step"] + \
                out["back_end"][K]["total_ms"]
            per_min[f"{kind}_K{K}"] = {"steps": steps, "total_s": total_ms / 1e3,
                                       "compute_s_per_audio_minute": total_ms / 1e3 / (SECONDS / 60)}
    out["compute_per_audio_minute"] = per_min
    out["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "track_sep_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
