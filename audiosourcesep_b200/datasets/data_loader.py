"""``get_song_extract`` -- mirror of the reference's ``datasets/data_loader.py:113-180`` (+ ``load_wav``,
datasets/preprocessing.py:9-26): cut a mixture and its two sources into 2.04 s extracts, STFT them, map to 96 mel bands in
dB.  The wav files are read here (8 / 16 / 24 / 32-bit PCM and 32-bit IEEE float, plain or WAVE_FORMAT_EXTENSIBLE,
down-mixed to mono like librosa.load(mono=True)); a file at another rate than ``sr`` is resampled on the GPU with
librosa.load's default kaiser_best filter (audiosourcesep_b200.resample -> csrc/resample_kernels.cu); the STFT, the mel
projection and the dB conversion run on the GPU (audiosourcesep_b200.melspec -> csrc/mel_kernels.cu)."""
from __future__ import annotations

import struct

import numpy as np
import torch

from .. import melspec

_WAVE_FORMAT_PCM, _WAVE_FORMAT_IEEE_FLOAT, _WAVE_FORMAT_EXTENSIBLE = 0x0001, 0x0003, 0xFFFE
# KSDATAFORMAT_SUBTYPE_* GUIDs are the format tag followed by this fixed suffix
_GUID_SUFFIX = b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"


def _riff_chunks(path: str):
    """(fmt chunk body, data chunk body) of a RIFF/WAVE file."""
    with open(path, "rb") as f:
        blob = f.read()
    if len(blob) < 12 or blob[:4] != b"RIFF" or blob[8:12] != b"WAVE":
        raise ValueError(f"{path}: not a RIFF/WAVE file")
    fmt = data = None
    pos = 12
    while pos + 8 <= len(blob):
        cid, size = blob[pos:pos + 4], struct.unpack("<I", blob[pos + 4:pos + 8])[0]
        body = blob[pos + 8: pos + 8 + size]                  # a streamed file may declare more than it holds
        if cid == b"fmt ":
            fmt = body
        elif cid == b"data":
            data = body
        pos += 8 + size + (size & 1)                          # chunks are word-aligned
    if fmt is None or len(fmt) < 16:
        raise ValueError(f"{path}: no valid 'fmt ' chunk")
    if data is None:
        raise ValueError(f"{path}: no 'data' chunk")
    return fmt, data


def read_wav_mono(path: str):
    """wav -> (float32 mono, rate), scaled as soundfile reads it: PCM of 8 bits ((u - 128) / 128), 16 bits (/ 2^15),
    24 bits (/ 2^23) or 32 bits (/ 2^31); 32-bit IEEE float as stored.  Channels are averaged."""
    fmt, raw = _riff_chunks(path)
    tag, nch, rate, _, block_align, bits = struct.unpack("<HHIIHH", fmt[:16])
    if tag == _WAVE_FORMAT_EXTENSIBLE:
        if len(fmt) < 40 or fmt[26:40] != _GUID_SUFFIX:
            raise ValueError(f"{path}: WAVE_FORMAT_EXTENSIBLE with an unknown sub-format")
        tag = struct.unpack("<H", fmt[24:26])[0]
    if nch < 1 or block_align != nch * (bits // 8) or bits % 8:
        raise ValueError(f"{path}: inconsistent format ({nch} channels, {bits} bits, block align {block_align})")
    raw = raw[: len(raw) - len(raw) % block_align]
    width = bits // 8
    if tag == _WAVE_FORMAT_PCM and width == 2:
        a = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif tag == _WAVE_FORMAT_PCM and width == 4:
        a = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
    elif tag == _WAVE_FORMAT_PCM and width == 1:
        a = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    elif tag == _WAVE_FORMAT_PCM and width == 3:
        b = np.zeros((len(raw) // 3, 4), dtype=np.uint8)
        b[:, 1:] = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3)    # sample in the top 24 bits, sign-extended by >> 8
        a = (b.view("<i4").reshape(-1) >> 8).astype(np.float32) / 8388608.0
    elif tag == _WAVE_FORMAT_IEEE_FLOAT and width == 4:
        a = np.frombuffer(raw, dtype="<f4").astype(np.float32)
    else:
        kind = {_WAVE_FORMAT_PCM: "PCM", _WAVE_FORMAT_IEEE_FLOAT: "IEEE float"}.get(tag, f"format tag 0x{tag:04x}")
        raise ValueError(f"{path}: unsupported wav format: {kind}, {bits} bits per sample")
    if nch > 1:
        a = a.reshape(-1, nch).mean(axis=1)
    return a, rate


def load_wav(path, length_sec, sr=None):
    """reference: datasets/preprocessing.py:9-26 -- librosa.load(path, sr=sr) (mono; resampled with kaiser_best on the
    GPU when the file's rate differs from ``sr``), cut into windows of int(sr * length_sec) samples
    (drop_remainder=True).  Returns (float32 [n_windows, LENGTH], rate)."""
    song, rate = read_wav_mono(path)
    if sr is not None and rate != sr:
        from ..resample import resample
        song, rate = resample(song, rate, sr).cpu().numpy(), sr
    LENGTH = int(rate * length_sec)
    n = len(song) // LENGTH
    return song[: n * LENGTH].reshape(n, LENGTH), rate


def get_song_extract(mix_path, piano_path, violin_path, duration, **kwargs):
    """reference: datasets/data_loader.py:113-180.  Returns (mel_spec, raw_audio, stft_mixture):
    mel_spec = [mix, piano, violin], each float32 [n_extract, n_mels, T, 1]; raw_audio = the three concatenated
    waveforms; stft_mixture complex64 [n_extract, 1 + n_fft/2, T]."""
    return get_song_extract_k(mix_path, [piano_path, violin_path], duration, **kwargs)


def get_song_extract_k(mix_path, source_paths, duration, **kwargs):
    """get_song_extract for any number of stems: mel_spec = [mix, s_1, ..., s_K] and raw_audio the K + 1 concatenated
    waveforms, in the order of ``source_paths``."""
    length_sec = kwargs["length_sec"]
    fmin, fmax, sr = kwargs["fmin"], kwargs["fmax"], kwargs["sr"]
    dbmin, dbmax = kwargs["dbmin"], kwargs["dbmax"]
    n_fft, hop_length, n_mels = kwargs["n_fft"], kwargs["hop_length"], kwargs["n_mels"]
    use_dB = kwargs["use_dB"]
    if not use_dB:
        raise NotImplementedError("power-scale mel spectrograms (use_dB=False) are not on the separation path of the configs")
    n_extract = int(round(duration / length_sec, 0))
    tracks = []
    for p in [mix_path] + list(source_paths):
        frames, _ = load_wav(p, length_sec, sr=sr)
        if frames.shape[0] < 2 + n_extract:
            raise ValueError(f"{p}: {frames.shape[0]} windows of {length_sec} s, {2 + n_extract} needed (the first two are skipped)")
        tracks.append(frames[2: 2 + n_extract])                       # "skip 2 first frames" (:131-134)
    raw_audio = [np.concatenate(list(t)) for t in tracks]
    mel_spec, stft_mixture = [], None
    for i, t in enumerate(tracks):
        S = melspec.stft(t, n_fft=n_fft, hop_length=hop_length)
        if i == 0:
            stft_mixture = S.cpu().numpy()
        mel = melspec.melspectrogram_db(S, sr=sr, n_fft=n_fft, n_mels=n_mels, fmin=fmin, fmax=fmax, dbmin=dbmin, dbmax=dbmax)
        mel_spec.append(mel.unsqueeze(-1).contiguous())
    return mel_spec, raw_audio, stft_mixture
