"""Audio front-end timings on one GPU: asep_resample alone, the whole wav -> mel dataset build, and the CPU oracle.

    python tools/audio_frontend_bench.py --out <dir>

1. asep_resample on 10 min of 44.1 kHz audio -> 16 kHz: CUDA events around each call, after warm-up calls, >= 20 timed
   calls (the 106 MB input and 38 MB output fit in the 126 MB L2 only in part; the 256 KB table is L2-resident).
2. datasets.wav_to_spec.build_dataset over a generated directory of 3 files x 10 min, 44.1 kHz, 24-bit stereo
   (host clock around the call, ending in a device synchronise; one untimed warm-up on a short file first).
3. The float64 CPU restatement (oracle/resample_oracle.py) per second of 44.1 kHz audio, for context.
The card's name and power limit are recorded beside the numbers.  Writes <out>/audio_frontend_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import struct
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audiosourcesep_b200 import _lib  # noqa: E402
from audiosourcesep_b200 import resample as rs  # noqa: E402
from audiosourcesep_b200.datasets import wav_to_spec  # noqa: E402
from oracle import resample_oracle as ro  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def write_pcm24_stereo(path, n, sr, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    a = np.stack([0.3 * np.sin(2 * np.pi * 440 * t), 0.3 * np.sin(2 * np.pi * 660 * t)], axis=1) + 0.05 * rng.standard_normal((n, 2))
    ints = np.clip(np.round(a * 2 ** 23), -2 ** 23, 2 ** 23 - 1).astype(np.int64)
    data = (ints.reshape(-1) & 0xFFFFFF).astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    fmt = struct.pack("<HHIIHH", 1, 2, sr, sr * 6, 6, 24)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def bench_resample(reps: int):
    sr, minutes = 44100, 10
    L = minutes * 60 * sr
    ratio = 16000 / sr
    d = _lib.init()
    x = torch.randn((1, L), device="cuda") * 0.3
    win, delta = rs._device_table(ratio, d)
    n_out = int(L * ratio)
    tt = torch.as_tensor(rs.running_time(n_out, ratio)).cuda()
    out = torch.empty((1, n_out), device="cuda")
    scale = min(1.0, ratio)
    lib = _lib.load()
    dl = [_lib.dl(v) for v in (x, tt, win, delta, out)]

    def call():
        _lib.check(lib.asep_resample(dl[0].ptr, dl[1].ptr, dl[2].ptr, dl[3].ptr, scale, int(scale * rs.NUM_TABLE), dl[4].ptr,
                                     _lib.stream_ptr()))

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    step = int(scale * rs.NUM_TABLE)
    nwin = int(win.numel())
    taps = 2 * (nwin // step)                                    # ~ taps per output sample (both wings)
    med = float(np.median(ms))
    return {"input": f"{minutes} min at {sr} Hz -> 16000 Hz, 1 row", "input_samples": L, "output_samples": n_out,
            "taps_per_output_approx": taps, "reps": reps, "ms_median": med, "ms_min": float(np.min(ms)),
            "ms_max": float(np.max(ms)), "output_samples_per_s": n_out / (med * 1e-3),
            "audio_seconds_per_s": minutes * 60 / (med * 1e-3), "taps_per_s": n_out * taps / (med * 1e-3)}


def bench_wav_to_spec(tmp, reps: int):
    sr, minutes, n_files = 44100, 10, 3
    src = os.path.join(tmp, "wavs")
    os.makedirs(src)
    for i in range(n_files):
        write_pcm24_stereo(os.path.join(src, f"song{i}.wav"), minutes * 60 * sr, sr, i)
    warm = os.path.join(tmp, "warm.wav")
    write_pcm24_stereo(warm, 10 * sr, sr, 99)
    quiet = lambda *a, **k: None                                 # noqa: E731
    wav_to_spec.build_dataset([warm], os.path.join(tmp, "warm.npz"), log=quiet)
    torch.cuda.synchronize()
    secs = []
    for r in range(reps):
        t0 = time.perf_counter()
        res = wav_to_spec.build_dataset([src], os.path.join(tmp, f"ds{r}.npz"), log=quiet)
        torch.cuda.synchronize()
        secs.append(time.perf_counter() - t0)
    n = int(res["train"].shape[0] + res["test"].shape[0])
    return {"input": f"{n_files} files x {minutes} min, {sr} Hz, 24-bit stereo", "patches": n, "reps": reps,
            "s_each": secs, "s_min": float(min(secs)), "audio_seconds_per_s": n_files * minutes * 60 / min(secs)}


def bench_oracle():
    sr = 44100
    x = np.random.default_rng(0).standard_normal(2 * sr)
    t0 = time.perf_counter()
    ro.resample_rows(x, 16000 / sr)
    s = time.perf_counter() - t0
    return {"input": "2 s at 44100 Hz -> 16000 Hz, float64 numpy (vectorised form)", "s_per_audio_second": s / 2.0}


def main():
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--out", type=str, required=True, help="output directory for audio_frontend_bench.json")
    p.add_argument("--reps", type=int, default=20)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("audio_frontend_bench needs a CUDA device")
    res = {"card": card()}
    res["asep_resample"] = bench_resample(max(20, args.reps))
    with tempfile.TemporaryDirectory() as tmp:
        res["wav_to_spec"] = bench_wav_to_spec(tmp, 2)
    res["cpu_oracle"] = bench_oracle()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "audio_frontend_bench.json"), "w") as f:
        json.dump(res, f, indent=2)
    print(json.dumps(res, indent=2))


if __name__ == "__main__":
    main()
