"""CPU checks of the mask rendering's restatement (oracle/mwf_oracle.py): the output STFT grid, the track PSD map, the
multichannel Wiener filter with EM and mixture consistency, the flag rules of --render mask, and the multichannel wav
reading / writing it relies on."""
import struct
import wave

import numpy as np
import pytest

from audiosourcesep_b200 import melspec, melspec_inversion_basis as inv, run_basis_sep, track
from audiosourcesep_b200.datasets import data_loader
from oracle import mel_oracle as mo
from oracle import mwf_oracle as mw
from oracle import track_oracle as to


@pytest.mark.parametrize("sr, grid", [(8000, (1024, 256)), (16000, (2048, 512)), (22050, (2048, 512)),
                                      (32000, (4096, 1024)), (44100, (4096, 1024)), (48000, (4096, 1024))])
def test_output_grid(sr, grid):
    assert mw.out_grid(sr) == grid
    assert track.out_grid(sr) == grid


def test_band_edges_come_from_the_filter_bank():
    lo, hi = mw.band_edges()
    assert (lo, hi) == melspec.band_edges()
    A = mo.mel_filters()
    assert A[:, lo].max() > 0 and A[:, hi].max() > 0
    assert not A[:, :lo].any() and not A[:, hi + 1:].any()


def _mags(K, n_seg, seed=0, F=1025, T=64):
    return np.random.default_rng(seed).uniform(0.0, 2.0, (K, n_seg, F, T)).astype(np.float32)


@pytest.mark.parametrize("o", [0, 1, 8, 31])
def test_frame_weights_are_the_crossfade_at_frame_centres(o):
    L = 3 * to.SPAN + 1000
    n_seg = len(to.segment_starts(L, o))
    w = mw.frame_weights(n_seg, 64, o)
    c = to.crossfade_weights(L, o)
    starts = to.segment_starts(L, o)
    for g in range(n_seg):
        for j in range(64):
            n = int(starts[g]) + 512 * j
            if n < L and (j < 63 or g < n_seg - 1):
                assert w[g, j] == c[g, n], (g, j)
    if o > 0:
        assert w[0, 63] == 0.0 and w[1, 0] > 0.0                   # the zero-weight edge frame drops out
    assert w[-1, 63] == 1.0


@pytest.mark.parametrize("o", [0, 8, 31])
def test_psd_at_16k_is_the_crossfaded_segment_psd(o):
    K, n_seg = 2, 3
    mag = _mags(K, n_seg, o)
    lo, hi = mw.band_edges()
    Q = 63 - o
    T16 = (n_seg - 1) * Q + 64
    psd = mw.track_psd(mag, o, lo, hi, 16000, 2048, 512, T16 + 5)
    L = (n_seg - 1) * (to.SPAN - 512 * o) + to.SPAN
    c = to.crossfade_weights(L, o)
    starts = to.segment_starts(L, o)
    for tau in range(T16):
        n = 512 * tau
        if n >= L:
            continue
        num, den = 0.0, 0.0
        for g in range(n_seg):
            j = tau - g * Q
            if 0 <= j < 64 and c[g, n] > 0:
                num = num + c[g, n] * mag[:, g, :, j].astype(np.float64) ** 2
                den += c[g, n]
        np.testing.assert_allclose(psd[:, lo:hi + 1, tau], (num / den)[:, lo:hi + 1], rtol=1e-12, atol=0)
    np.testing.assert_array_equal(psd[:, :, T16:], np.repeat(psd[:, :, T16 - 1:T16], 5, axis=2))   # clamped in time
    assert starts[-1] + to.SPAN >= L


def test_out_of_band_bins_take_the_edge_and_time_ramps_interpolate_exactly():
    K, n_seg, o = 2, 3, 8
    Q = 63 - o
    tau = np.arange(64)[None, :] + Q * np.arange(n_seg)[:, None]       # track frame of every segment frame
    power = 0.5 + 0.01 * tau                                            # linear in time, the same in every bin
    mag = np.broadcast_to(np.sqrt(power)[None, :, None, :], (K, n_seg, 1025, 64)).astype(np.float64)
    lo, hi = mw.band_edges()
    sr = 44100
    n_fft, hop = mw.out_grid(sr)
    T_out = 300
    psd = mw.track_psd(mag, o, lo, hi, sr, n_fft, hop, T_out)
    T16 = (n_seg - 1) * Q + 64
    q = np.clip(np.arange(T_out) * hop * 16000 / (sr * 512), 0, T16 - 1)
    np.testing.assert_allclose(psd[0, 500], 0.5 + 0.01 * q, rtol=1e-12)
    # out of band: the rows of the edge bins
    mag2 = _mags(K, n_seg, 5).astype(np.float64)
    psd2 = mw.track_psd(mag2, o, lo, hi, sr, n_fft, hop, T_out)
    P16 = mw.segment_power(mag2, o)
    b = np.arange(n_fft // 2 + 1)
    p = b * sr * 2048 / (n_fft * 16000)
    below, above = b[p <= lo], b[p >= hi]
    assert len(below) > 10 and len(above) > 500
    q0 = np.floor(q).astype(int)
    q1, a = np.minimum(q0 + 1, T16 - 1), q - q0
    for edge, rows in ((lo, below), (hi, above)):
        want = P16[:, edge, q0] * (1 - a) + P16[:, edge, q1] * a
        for r in rows:
            np.testing.assert_allclose(psd2[:, r], want, rtol=1e-12)


def _rand_stft(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


@pytest.mark.parametrize("C", [1, 2])
@pytest.mark.parametrize("n", [0, 1, 2, 3])
def test_stems_sum_to_the_mixture(C, n):
    rng = np.random.default_rng(10 * C + n)
    K, F, T = 3, 17, 40
    psd = rng.uniform(0, 2, (K, F, T)) ** 3
    psd[:, 3] = 0.0                                                     # all-zero PSD bins
    psd[:, :, 7] = 0.0
    X = _rand_stft(rng, C, F, T) * 10
    X[:, 5] = 0.0                                                       # a silent row
    y = mw.mwf(psd, X, n)
    assert y.shape == (K, C, F, T) and np.all(np.isfinite(y))
    np.testing.assert_allclose(y.sum(axis=0), X, rtol=0, atol=1e-12)
    np.testing.assert_allclose(y[:, :, 3], np.broadcast_to(X[None, :, 3] / K, (K, C, T)), rtol=0, atol=1e-12)


def test_mono_without_iterations_is_the_single_channel_wiener_filter():
    rng = np.random.default_rng(1)
    K, F, T = 4, 9, 30
    psd = rng.uniform(0, 1, (K, F, T))
    X = _rand_stft(rng, 1, F, T)
    y = mw.mwf(psd, X, 0)
    w = mo.single_channel_wiener_filter(psd, X[0])
    np.testing.assert_allclose(y[:, 0], w + (X[0] - w.sum(axis=0)) / K, rtol=0, atol=1e-13)


def test_dual_mono_matches_mono():
    rng = np.random.default_rng(2)
    K, F, T = 3, 9, 30
    psd = rng.uniform(0, 1, (K, F, T)) * 1e6
    X = _rand_stft(rng, 1, F, T) * 1e3
    for n in (0, 1, 3):
        mono = mw.mwf(psd, X, n)
        dual = mw.mwf(psd, np.concatenate([X, X]), n)
        np.testing.assert_array_equal(dual[:, 0], dual[:, 1])
        np.testing.assert_allclose(dual[:, 0], mono[:, 0], rtol=0, atol=1e-9 * np.abs(X).max())


def _sdr(ref, est):
    return 10 * np.log10(np.sum(np.abs(ref) ** 2) / np.sum(np.abs(est - ref) ** 2))


def test_em_iteration_learns_hard_panning():
    rng = np.random.default_rng(3)
    F, T = 33, 200
    env = [rng.uniform(0.2, 1.0, (F, 1)) * rng.uniform(0.2, 1.0, (1, T)) for _ in range(2)]
    s1 = np.stack([_rand_stft(rng, F, T) * env[0], np.zeros((F, T))])          # left only
    s2 = np.stack([np.zeros((F, T)), _rand_stft(rng, F, T) * env[1]])          # right only
    X = s1 + s2
    psd = np.stack([np.mean(np.abs(s) ** 2, axis=0) for s in (s1, s2)])
    sdr = {n: min(_sdr(s, y) for s, y in zip((s1, s2), mw.mwf(psd, X, n))) for n in (0, 1)}
    assert sdr[1] > sdr[0] + 1, sdr


def _args(argv):
    return run_basis_sep.build_parser().parse_args(argv)


def test_render_flag_rules():
    ok = [["a", "b", "--mix", "m.wav"], ["a", "b", "--mix", "m.wav", "--render", "mask"],
          ["a", "b", "--mix", "m.wav", "--render", "mask", "--mwf_iterations", "0"],
          ["a", "b", "--mix", "m.wav", "--render", "mask", "--mwf_iterations", "10"],
          ["a", "b", "--mix", "m.wav", "--render", "mel", "--wiener_filter"]]
    for argv in ok:
        run_basis_sep.check_mix_args(_args(argv))
    bad = [(["a", "b", "--render", "mask"], "--mix"), (["a", "b", "--song_dir", "s", "--render", "mask"], "--mix"),
           (["a", "b", "--mix", "m.wav", "--render", "mask", "--wiener_filter"], "--wiener_filter"),
           (["a", "b", "--mix", "m.wav", "--mwf_iterations", "2"], "--render mask"),
           (["a", "b", "--mix", "m.wav", "--render", "mel", "--mwf_iterations", "1"], "--render mask"),
           (["a", "b", "--mix", "m.wav", "--render", "mask", "--mwf_iterations", "11"], "mwf_iterations"),
           (["a", "b", "--mix", "m.wav", "--render", "mask", "--mwf_iterations", "-1"], "mwf_iterations")]
    for argv, match in bad:
        with pytest.raises(ValueError, match=match):
            run_basis_sep.check_mix_args(_args(argv))
    with pytest.raises(SystemExit):
        _args(["a", "b", "--mix", "m.wav", "--render", "griffin"])


def test_merge_config_keeps_the_render_fields(tmp_path):
    yml = tmp_path / "c.yml"
    yml.write_text("T: 7\nrender: mel\nmwf_iterations: 4\n")
    merged = run_basis_sep.merge_config(_args(["a", "b", "--config", str(yml), "--mix", "m.wav", "--render", "mask",
                                               "--mwf_iterations", "2"]))
    assert merged.render == "mask" and merged.mwf_iterations == 2 and merged.T == 7


def test_inversion_cli_render_rules(tmp_path):
    track_dir, seg_dir = tmp_path / "track", tmp_path / "seg"
    track_dir.mkdir()
    seg_dir.mkdir()
    z = np.zeros((1, 96, 64), np.float32)
    np.savez(track_dir / "results", x1=z, x2=z, mixed=z, stft_mixture=np.zeros((1, 1025, 64), np.complex64),
             segment_start=np.zeros(1, np.int64), track_length=np.int64(1000), orig_sr=np.int64(16000),
             orig_length=np.int64(1000), overlap_frames=np.int64(8))
    np.savez(seg_dir / "results", x1=z, x2=z, gt1=z, gt2=z, mixed=z, stft_mixture=np.zeros((1, 1025, 64), np.complex64))
    p = inv.build_parser()
    for argv, match in (([str(track_dir), "--render", "mask"], "--mix"),
                        ([str(seg_dir), "--render", "mask", "--mix", "m.wav"], "whole track"),
                        ([str(track_dir), "--render", "mask", "--mix", "m.wav", "--wiener_filter"], "--wiener_filter"),
                        ([str(track_dir), "--render", "mask", "--mix", "m.wav", "--mwf_iterations", "11"], "mwf_iterations"),
                        ([str(track_dir), "--mwf_iterations", "2"], "--render mask")):
        with pytest.raises(ValueError, match=match):
            inv.main(p.parse_args(argv))


def _write(path, frames: bytes, nch, rate, bits, tag=1):
    fmt = struct.pack("<HHIIHH", tag, nch, rate, rate * nch * bits // 8, nch * bits // 8, bits)
    data = b"RIFF" + struct.pack("<I", 4 + 8 + len(fmt) + 8 + len(frames)) + b"WAVE"
    data += b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(frames)) + frames
    path.write_bytes(data)


@pytest.mark.parametrize("kind", ["pcm16_mono", "pcm16_stereo", "pcm24_stereo", "float_stereo", "float_mono"])
def test_read_wav_and_the_unchanged_mono_mix(tmp_path, kind):
    rng = np.random.default_rng(4)
    nch = 2 if kind.endswith("stereo") else 1
    n = 1001
    if kind.startswith("pcm16"):
        ints = rng.integers(-32768, 32768, n * nch).astype("<i2")
        frames, bits, tag, flat = ints.tobytes(), 16, 1, ints.astype(np.float32) / 32768.0
    elif kind.startswith("pcm24"):
        ints = rng.integers(-2 ** 23, 2 ** 23, n * nch).astype("<i4")
        frames, bits, tag = ints.view(np.uint8).reshape(-1, 4)[:, :3].tobytes(), 24, 1
        flat = ints.astype(np.float32) / 8388608.0
    else:
        vals = rng.standard_normal(n * nch).astype("<f4")
        vals[:7] = -0.0
        frames, bits, tag, flat = vals.tobytes(), 32, 3, vals
    path = tmp_path / "a.wav"
    _write(path, frames, nch, 22050, bits, tag)
    x, rate = data_loader.read_wav(str(path))
    assert rate == 22050 and x.shape == (nch, n) and x.dtype == np.float32
    np.testing.assert_array_equal(x, flat.reshape(-1, nch).T)
    mono, rate = data_loader.read_wav_mono(str(path))
    want = flat.reshape(-1, nch).mean(axis=1) if nch > 1 else flat          # the down-mix as it was before read_wav
    assert mono.shape == (n,) and mono.tobytes() == want.tobytes()


def test_write_wav_keeps_mono_bytes_and_writes_channels(tmp_path):
    rng = np.random.default_rng(5)
    a = rng.uniform(-1.2, 1.2, 999)
    inv.write_wav(str(tmp_path / "m.wav"), a, 44100)
    with wave.open(str(tmp_path / "m.wav"), "rb") as w:
        assert w.getnchannels() == 1 and w.getsampwidth() == 2
        got = w.readframes(w.getnframes())
    pcm = np.clip(a, -1.0, 1.0 - 1.0 / 32768.0)
    assert got == (pcm * 32768.0).astype("<i2").tobytes()
    st = rng.uniform(-1, 1, (2, 999))
    inv.write_wav(str(tmp_path / "s.wav"), st, 44100)
    with wave.open(str(tmp_path / "s.wav"), "rb") as w:
        assert w.getnchannels() == 2 and w.getnframes() == 999 and w.getframerate() == 44100
        back = np.frombuffer(w.readframes(999), "<i2").reshape(-1, 2).T
    np.testing.assert_array_equal(back, (st * 32768.0).astype("<i2"))
