"""CPU checks of the resampling restatement (oracle/resample_oracle.py), of the host half of
audiosourcesep_b200/resample.py, and of the wav reader's formats -- no GPU needed."""
import math
import struct
import wave

import numpy as np
import pytest
from scipy import signal

from audiosourcesep_b200 import resample as rs
from audiosourcesep_b200.datasets.data_loader import read_wav_mono
from oracle import resample_oracle as ro

RATES = (44100, 48000, 22050, 8000)


@pytest.mark.parametrize("orig_sr", RATES)
def test_literal_loop_and_vectorised_form_agree(orig_sr):
    x = np.random.default_rng(orig_sr).standard_normal(1200)
    ratio = 16000 / orig_sr
    a = ro.resample_loop(x, ratio)
    b = ro.resample_rows(x, ratio)
    assert a.shape == b.shape == (int(1200 * ratio),)
    assert np.max(np.abs(a - b)) <= 1e-12
    # a subset of output samples and batched rows give the same numbers
    rows = np.stack([x, -0.5 * x])
    sub = np.array([0, 3, a.size // 2, a.size - 1])
    np.testing.assert_allclose(ro.resample_rows(rows, ratio, t_index=sub), np.stack([a[sub], -0.5 * a[sub]]), rtol=0, atol=1e-12)


@pytest.mark.parametrize("orig_sr", RATES)
def test_time_register_cumsum_is_the_running_sum(orig_sr):
    ratio = 16000 / orig_sr
    n = int(2 * orig_sr * ratio) + 7
    loop = ro.time_register_loop(n, ratio)
    assert np.array_equal(ro.time_register(n, ratio), loop)
    assert np.array_equal(rs.running_time(n, ratio), loop)          # the product's host time register too
    if orig_sr in (44100, 22050):       # inexact increments: the running sum is not t / ratio in the last bits
        assert not np.array_equal(loop, np.arange(n) / ratio)


def test_filter_table():
    win, delta = ro.filter_table(2.0)
    assert win.shape == delta.shape == (32769,)
    assert win[0] == ro.ROLLOFF and delta[-1] == 0.0
    w2, d2 = ro.filter_table(16000 / 44100)
    np.testing.assert_allclose(w2, win * (16000 / 44100), rtol=1e-15, atol=0)
    for ratio in (2.0, 16000 / 44100):
        pw, pd = rs.kaiser_best_table(ratio)
        ow, od = ro.filter_table(ratio)
        np.testing.assert_allclose(pw, ow, rtol=0, atol=1e-14)
        np.testing.assert_allclose(pd, od, rtol=0, atol=1e-14)


@pytest.mark.parametrize("L", [1000, 1001, 4410, 4413])
def test_length_fix_and_identity(L):
    x = np.random.default_rng(L).standard_normal(L)
    y = ro.resample(x, 44100, 16000)
    n_fix, n_out = math.ceil(L * 16000 / 44100), int(L * 16000 / 44100)
    assert y.shape == (n_fix,)
    assert np.all(y[n_out:] == 0.0)
    np.testing.assert_array_equal(y[:n_out], ro.resample_rows(x, 16000 / 44100))
    assert np.array_equal(ro.resample(x, 16000, 16000), x)
    with pytest.raises(ValueError):
        ro.resample(x[:2], 44100, 16000)


def _tone_amplitude(y, f, sr, edge):
    seg = y[edge:-edge]
    t = np.arange(y.size)[edge:-edge] / sr
    A = np.stack([np.sin(2 * np.pi * f * t), np.cos(2 * np.pi * f * t)], axis=1)
    c, *_ = np.linalg.lstsq(A, seg, rcond=None)
    return float(np.hypot(*c)), float(np.sqrt(2.0 * np.mean(seg ** 2)))


def test_known_answers_on_tones():
    """Recorded from the restatement (44.1 -> 16 kHz): 1 kHz gain 1 + 2.7e-3 (the truncated table stride compresses the
    filter by ~0.4 %, so this is NOT the textbook kaiser_best figure), 9 kHz rejected by ~63.8 dB."""
    sr = 44100
    t = np.arange(2 * sr) / sr
    gain, _ = _tone_amplitude(ro.resample(np.sin(2 * np.pi * 1000 * t), sr, 16000), 1000, 16000, 4000)
    assert abs(gain - 1.0) <= 5e-3
    _, rms_amp = _tone_amplitude(ro.resample(np.sin(2 * np.pi * 9000 * t), sr, 16000), 9000, 16000, 4000)
    assert 20 * np.log10(rms_amp) <= -55.0


def test_independent_cross_check_with_resample_poly():
    """scipy's polyphase resampler (a different filter design) agrees on noise band-limited below 6 kHz."""
    sr = 44100
    rng = np.random.default_rng(3)
    X = np.fft.rfft(rng.standard_normal(4 * sr))
    X[np.fft.rfftfreq(4 * sr, 1 / sr) > 6000] = 0
    x = np.fft.irfft(X, 4 * sr)
    x /= x.std()
    a = ro.resample(x, sr, 16000)
    b = signal.resample_poly(x, 160, 441)
    n = min(a.size, b.size)
    a, b = a[2000:n - 2000], b[2000:n - 2000]
    rel = np.linalg.norm(a - b) / np.linalg.norm(b)
    assert rel <= 1e-2, rel


# ---------------------------------------------------------------- wav reader
def _write_riff(path, fmt_chunk: bytes, data: bytes):
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt_chunk)) + fmt_chunk + b"data" + struct.pack("<I", len(data)) + data
    if len(data) & 1:
        body += b"\x00"
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def _fmt(tag, nch, rate, bits):
    return struct.pack("<HHIIHH", tag, nch, rate, rate * nch * bits // 8, nch * bits // 8, bits)


def _fmt_extensible(sub_tag, nch, rate, bits):
    guid = struct.pack("<H", sub_tag) + b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
    return _fmt(0xFFFE, nch, rate, bits) + struct.pack("<HHI", 22, bits, 0x3) + guid


def test_wav_reader_decodes_24_bit_float_and_extensible(tmp_path):
    rng = np.random.default_rng(0)
    # 24-bit PCM stereo: integers written, integers / 2^23 read back (mean over channels)
    ints = rng.integers(-2 ** 23, 2 ** 23, size=(1001, 2))
    b = (ints & 0xFFFFFF).astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    _write_riff(tmp_path / "a24.wav", _fmt(1, 2, 44100, 24), b)
    a, rate = read_wav_mono(str(tmp_path / "a24.wav"))
    assert rate == 44100 and a.dtype == np.float32 and a.shape == (1001,)
    np.testing.assert_array_equal(a, (ints.astype(np.float32) / 8388608.0).mean(axis=1))
    # 32-bit IEEE float, mono: the samples themselves
    f = rng.uniform(-1, 1, 777).astype(np.float32)
    _write_riff(tmp_path / "f32.wav", _fmt(3, 1, 48000, 32), f.astype("<f4").tobytes())
    a, rate = read_wav_mono(str(tmp_path / "f32.wav"))
    assert rate == 48000 and np.array_equal(a, f)
    # WAVE_FORMAT_EXTENSIBLE with the float and the PCM sub-formats
    _write_riff(tmp_path / "xf.wav", _fmt_extensible(3, 1, 22050, 32), f.astype("<f4").tobytes())
    assert np.array_equal(read_wav_mono(str(tmp_path / "xf.wav"))[0], f)
    _write_riff(tmp_path / "x24.wav", _fmt_extensible(1, 2, 44100, 24), b)
    np.testing.assert_array_equal(read_wav_mono(str(tmp_path / "x24.wav"))[0], (ints.astype(np.float32) / 8388608.0).mean(axis=1))
    # 16-bit through the standard library's writer keeps its scaling
    s16 = rng.integers(-32768, 32768, 500).astype("<i2")
    with wave.open(str(tmp_path / "s16.wav"), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000)
        w.writeframes(s16.tobytes())
    np.testing.assert_array_equal(read_wav_mono(str(tmp_path / "s16.wav"))[0], s16.astype(np.float32) / 32768.0)
    # anything else is refused by name
    _write_riff(tmp_path / "f64.wav", _fmt(3, 1, 16000, 64), np.zeros(4, "<f8").tobytes())
    with pytest.raises(ValueError, match="IEEE float, 64 bits"):
        read_wav_mono(str(tmp_path / "f64.wav"))
    _write_riff(tmp_path / "alaw.wav", _fmt(6, 1, 8000, 8), b"\x00" * 8)
    with pytest.raises(ValueError, match="format tag 0x0006"):
        read_wav_mono(str(tmp_path / "alaw.wav"))
