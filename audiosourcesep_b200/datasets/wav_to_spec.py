"""Mel-spectrogram dataset builder: wav files -> one ``.npz`` of train / test patches for ``train_glow --dataset`` and
``train_ncsn --dataset``.

The module name follows the reference's ``datasets/wav_to_spec.py``, which writes TFRecord shards that its
``load_melspec_ds`` reads; the container here is deliberately an ``.npz`` (the reference's TFRecord feature schema is
not restated in this repository).  Per file: read and down-mix (data_loader.read_wav_mono), resample to ``sr`` on the
GPU (kaiser_best, as librosa.load does), cut into non-overlapping windows of int(sr * length_sec) samples (the remainder
is dropped, like load_wav), then STFT -> mel -> dB -> clip on the GPU in bounded chunks of windows (top_db per window),
the spec parameters of run_basis_sep.py:207.  The windows are split into train / test per window with a seeded
permutation.

    python -m audiosourcesep_b200.datasets.wav_to_spec piano_dir/ extra.wav --output piano.npz

Output keys: ``train`` / ``test`` float32 [n, n_mels, 1 + LENGTH // hop, 1] in dB; ``train_file`` / ``test_file`` int32
indices into ``files``; ``files``; and the spec parameters as scalars.
"""
from __future__ import annotations

import argparse
import glob
import os
from typing import Dict, List, Sequence

import numpy as np
import torch

from .. import _lib, melspec
from ..resample import resample
from .data_loader import read_wav_mono

SPEC_DEFAULTS = dict(sr=16000, length_sec=2.04, n_fft=2048, hop_length=512, n_mels=96, fmin=125.0, fmax=7600.0,
                     dbmin=-100.0, dbmax=20.0)


def list_wavs(inputs: Sequence[str]) -> List[str]:
    """Files as given; directories expand to their ``*.wav`` files, sorted."""
    files = []
    for p in inputs:
        if os.path.isdir(p):
            found = sorted(glob.glob(os.path.join(p, "*.wav")))
            if not found:
                raise ValueError(f"{p}: no .wav file in the directory")
            files += found
        elif os.path.isfile(p):
            files.append(p)
        else:
            raise FileNotFoundError(p)
    if not files:
        raise ValueError("no input wav file")
    return files


def file_patches(path: str, sr=16000, length_sec=2.04, n_fft=2048, hop_length=512, n_mels=96, fmin=125.0, fmax=7600.0,
                 dbmin=-100.0, dbmax=20.0, chunk: int = 256, device=None) -> np.ndarray:
    """float32 [n_windows, n_mels, T, 1] dB patches of one wav file (see the module docstring)."""
    d = _lib.init(device)
    song, rate = read_wav_mono(path)
    if rate != sr:
        y = resample(song, rate, sr, device=d)
    else:
        y = torch.as_tensor(song).to(torch.device("cuda", d))
    length = int(sr * length_sec)
    n = int(y.shape[0]) // length
    frames = y[: n * length].reshape(n, length)
    out = []
    for c0 in range(0, n, int(chunk)):
        S = melspec.stft(frames[c0: c0 + int(chunk)], n_fft=n_fft, hop_length=hop_length, device=d)
        mel = melspec.melspectrogram_db(S, sr=sr, n_fft=n_fft, n_mels=n_mels, fmin=fmin, fmax=fmax, dbmin=dbmin, dbmax=dbmax)
        out.append(mel.unsqueeze(-1).cpu().numpy())
    T = 1 + length // hop_length
    return np.concatenate(out) if out else np.zeros((0, n_mels, T, 1), np.float32)


def split(n: int, test_fraction: float, seed: int) -> np.ndarray:
    """Boolean [n]: True for the round(test_fraction * n) windows a seeded permutation puts in the test set."""
    if not 0.0 <= test_fraction < 1.0:
        raise ValueError(f"test_fraction must be in [0, 1), got {test_fraction}")
    is_test = np.zeros(n, dtype=bool)
    is_test[np.random.default_rng(seed).permutation(n)[: int(round(test_fraction * n))]] = True
    return is_test


def build_dataset(inputs: Sequence[str], output: str, test_fraction: float = 0.2, seed: int = 0, chunk: int = 256,
                  log=print, **spec) -> Dict[str, np.ndarray]:
    """Writes ``output`` (.npz) and returns its arrays."""
    params = dict(SPEC_DEFAULTS, **spec)
    files = list_wavs(inputs)
    patches, owner = [], []
    for i, f in enumerate(files):
        p = file_patches(f, chunk=chunk, **params)
        log(f"{f}: {p.shape[0]} windows")
        patches.append(p)
        owner.append(np.full(p.shape[0], i, dtype=np.int32))
    X, owner = np.concatenate(patches), np.concatenate(owner)
    if X.shape[0] == 0:
        raise ValueError(f"no window of {params['length_sec']} s in the input files")
    is_test = split(X.shape[0], float(test_fraction), int(seed))
    arrays = dict(train=X[~is_test], test=X[is_test], train_file=owner[~is_test], test_file=owner[is_test],
                  files=np.array(files), test_fraction=np.float64(test_fraction), seed=np.int64(seed),
                  **{k: np.asarray(v) for k, v in params.items()})
    d = os.path.dirname(os.path.abspath(output))
    os.makedirs(d, exist_ok=True)
    np.savez(output, **arrays)
    log(f"{output}: {arrays['train'].shape[0]} train / {arrays['test'].shape[0]} test patches of shape {X.shape[1:]}")
    return arrays


def load_patches(path: str, height: int, width: int):
    """(train, test) float32 [n, height, width, 1] dB patches of a dataset written by :func:`build_dataset`."""
    with np.load(path) as z:
        train, test = z["train"], z["test"]
    for name, a in (("train", train), ("test", test)):
        if a.ndim != 4 or tuple(a.shape[1:]) != (int(height), int(width), 1):
            raise ValueError(f"{path}: {name} patches have shape {a.shape[1:]}, the model expects ({height}, {width}, 1)")
    return np.ascontiguousarray(train, dtype=np.float32), np.ascontiguousarray(test, dtype=np.float32)


def build_parser():
    p = argparse.ArgumentParser(description="wav files -> .npz of train / test mel-spectrogram patches (dB)")
    p.add_argument("inputs", nargs="+", help="wav files or directories (their *.wav files, sorted)")
    p.add_argument("--output", type=str, required=True, help="output .npz")
    p.add_argument("--sr", type=int, default=SPEC_DEFAULTS["sr"])
    p.add_argument("--length_sec", type=float, default=SPEC_DEFAULTS["length_sec"])
    p.add_argument("--n_fft", type=int, default=SPEC_DEFAULTS["n_fft"])
    p.add_argument("--hop_length", type=int, default=SPEC_DEFAULTS["hop_length"])
    p.add_argument("--n_mels", type=int, default=SPEC_DEFAULTS["n_mels"])
    p.add_argument("--fmin", type=float, default=SPEC_DEFAULTS["fmin"])
    p.add_argument("--fmax", type=float, default=SPEC_DEFAULTS["fmax"])
    p.add_argument("--dbmin", type=float, default=SPEC_DEFAULTS["dbmin"])
    p.add_argument("--dbmax", type=float, default=SPEC_DEFAULTS["dbmax"])
    p.add_argument("--test_fraction", type=float, default=0.2)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--chunk", type=int, default=256, help="windows per STFT / mel launch (bounds device memory)")
    return p


def main(args):
    spec = {k: getattr(args, k) for k in SPEC_DEFAULTS}
    return build_dataset(args.inputs, args.output, test_fraction=args.test_fraction, seed=args.seed, chunk=args.chunk, **spec)


if __name__ == "__main__":
    main(build_parser().parse_args())
