"""Mask rendering of a whole track on the GPU (run_basis_sep --mix --render mask): asep_track_psd and asep_mwf against
oracle/mwf_oracle.py, their reproducibility and argument checks, dual-mono input, the end-to-end CLI / inversion CLI /
separate_file on a 44.1 kHz 24-bit stereo file, and the full-band quality of stems rendered from ground-truth mel patches."""
import wave

import numpy as np
import pytest
import torch

from audiosourcesep_b200 import _lib, melspec, track
from audiosourcesep_b200.resample import resample
from oracle import mwf_oracle as mw

pytestmark = pytest.mark.gpu

BAD_ARG, BAD_SHAPE = -1, -2


def _mags(K, n_seg, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(K, n_seg, 1025, 64, generator=g) * 2).contiguous()


@pytest.mark.parametrize("sr", [16000, 22050, 44100, 48000])
@pytest.mark.parametrize("o", [0, 1, 8, 31])
def test_track_psd_matches_the_oracle(o, sr):
    K = (2, 3, 8)[(o + sr // 1000) % 3]
    n_seg = 3
    mag = _mags(K, n_seg, 7 * o + sr)
    lo, hi = melspec.band_edges()
    n_fft, hop = track.out_grid(sr)
    L = int(((n_seg - 1) * (track.SPAN - 512 * o) + track.SPAN) * sr / 16000)
    T_out = 1 + max(-(-L // hop) * hop, n_fft) // hop
    got = melspec.track_psd(mag.cuda(), o, lo, hi, sr, n_fft, hop, T_out).cpu().numpy()
    want = mw.track_psd(mag.numpy(), o, lo, hi, sr, n_fft, hop, T_out)
    assert got.shape == want.shape == (K, n_fft // 2 + 1, T_out)
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=0)


def _mix_case(K, C, seed, F=41, T=300):
    rng = np.random.default_rng(seed)
    psd = (rng.uniform(0, 2, (K, F, T)) ** 4 * rng.uniform(0, 1e4, (1, F, 1))).astype(np.float32)
    psd[:, 4] = 0.0                                                     # all-zero PSD rows and frames
    psd[:, :, 11] = 0.0
    X = ((rng.standard_normal((C, F, T)) + 1j * rng.standard_normal((C, F, T))) * 100).astype(np.complex64)
    X[:, 6] = 0.0                                                       # a silent row
    X[:, :, 13] = 0.0                                                   # a silent frame
    if C == 2:
        X[1, 20:30] = X[0, 20:30]                                       # dual-mono rows
        X[1, 30:35] = 0.5 * X[0, 30:35]                                 # proportional rows
    return psd, X


@pytest.mark.parametrize("n", [0, 1, 3])
@pytest.mark.parametrize("K", [2, 3, 8])
@pytest.mark.parametrize("C", [1, 2])
def test_mwf_matches_the_oracle(C, K, n):
    psd, X = _mix_case(K, C, 100 * C + 10 * K + n)
    got = melspec.mwf(torch.as_tensor(psd).cuda(), torch.as_tensor(X).cuda(), n).cpu().numpy()
    want = mw.mwf(psd, X, n)
    assert got.shape == want.shape == (K, C) + psd.shape[1:] and got.dtype == np.complex64
    scale = np.abs(X).max()
    ok = np.ones(psd.shape[1], bool)
    if C == 2:
        ok[30:35] = False                                               # rank-1 rows off the dual-mono symmetry: ill-posed
    np.testing.assert_allclose(got[:, :, ok], want[:, :, ok], rtol=0, atol=2e-6 * scale)
    np.testing.assert_allclose(got.sum(axis=0), X, rtol=0, atol=2e-6 * scale)   # the stems sum to the mixture everywhere
    np.testing.assert_allclose(got[:, :, 4], np.broadcast_to(X[None, :, 4] / K, got[:, :, 4].shape), rtol=0,
                               atol=2e-6 * scale)
    assert not got[:, :, 6].any()
    if C == 2:
        np.testing.assert_array_equal(got[:, 0, 20:30], got[:, 1, 20:30])


def test_two_identical_calls_are_bitwise_equal():
    psd, X = _mix_case(8, 2, 5, F=257, T=2000)
    p, x = torch.as_tensor(psd).cuda(), torch.as_tensor(X).cuda()
    a, b = melspec.mwf(p, x, 3), melspec.mwf(p, x, 3)
    assert torch.equal(torch.view_as_real(a), torch.view_as_real(b))
    mag = _mags(3, 4, 1).cuda()
    lo, hi = melspec.band_edges()
    a, b = (melspec.track_psd(mag, 8, lo, hi, 44100, 4096, 1024, 170) for _ in range(2))
    assert torch.equal(a, b)


def _raw_track_psd(mag, hop, o, lo, hi, sr, n_fft, out_hop, psd):
    dm, dp = _lib.dl(mag), _lib.dl(psd)
    return _lib.load().asep_track_psd(dm.ptr, hop, o, lo, hi, sr, n_fft, out_hop, dp.ptr, _lib.stream_ptr())


def _raw_mwf(psd, X, n, out):
    dp, dx, do = _lib.dl(psd), _lib.dl(X), _lib.dl(out)
    return _lib.load().asep_mwf(dp.ptr, dx.ptr, n, do.ptr, _lib.stream_ptr())


def test_bad_arguments_raise_before_any_launch():
    _lib.init()
    dev = "cuda"
    mag = torch.zeros(2, 3, 1025, 64, device=dev)
    psd = torch.zeros(2, 2049, 50, device=dev)
    good = (512, 8, 17, 972, 44100, 4096, 1024)
    assert _raw_track_psd(mag, *good, psd) == 0
    cases = [(torch.zeros(1, 3, 1025, 64, device=dev), good, torch.zeros(1, 2049, 50, device=dev), BAD_ARG),
             (torch.zeros(9, 3, 1025, 64, device=dev), good, torch.zeros(9, 2049, 50, device=dev), BAD_ARG),
             (mag, (512, 32, 17, 972, 44100, 4096, 1024), psd, BAD_ARG),
             (mag, (512, -1, 17, 972, 44100, 4096, 1024), psd, BAD_ARG),
             (mag, (512, 8, 973, 972, 44100, 4096, 1024), psd, BAD_ARG),
             (mag, (512, 8, -1, 972, 44100, 4096, 1024), psd, BAD_ARG),
             (mag, (512, 8, 17, 1025, 44100, 4096, 1024), psd, BAD_ARG),
             (mag, good, torch.zeros(2, 2048, 50, device=dev), BAD_SHAPE),
             (mag, good, torch.zeros(3, 2049, 50, device=dev), BAD_SHAPE),
             (mag[0], good, psd, BAD_SHAPE)]
    for m, args, p, code in cases:
        n0 = _lib.launch_count()
        assert _raw_track_psd(m.contiguous(), *args, p) == code, args
        assert _lib.launch_count() == n0
    P = torch.zeros(3, 65, 40, device=dev)
    X = torch.zeros(2, 65, 40, 2, device=dev)
    out = torch.zeros(3, 2, 65, 40, 2, device=dev)
    assert _raw_mwf(P, X, 1, out) == 0
    cases = [(torch.zeros(1, 65, 40, device=dev), X, 1, torch.zeros(1, 2, 65, 40, 2, device=dev), BAD_ARG),
             (torch.zeros(9, 65, 40, device=dev), X, 1, torch.zeros(9, 2, 65, 40, 2, device=dev), BAD_ARG),
             (P, torch.zeros(3, 65, 40, 2, device=dev), 1, torch.zeros(3, 3, 65, 40, 2, device=dev), BAD_ARG),
             (P, X, -1, out, BAD_ARG), (P, X, 11, out, BAD_ARG),
             (P, torch.zeros(2, 64, 40, 2, device=dev), 1, out, BAD_SHAPE),
             (P, torch.zeros(2, 65, 41, 2, device=dev), 1, out, BAD_SHAPE),
             (P, X, 1, torch.zeros(3, 1, 65, 40, 2, device=dev), BAD_SHAPE),
             (P, X, 1, torch.zeros(2, 2, 65, 40, 2, device=dev), BAD_SHAPE)]
    for p, x, n, o, code in cases:
        n0 = _lib.launch_count()
        assert _raw_mwf(p, x, n, o) == code, (tuple(p.shape), tuple(x.shape), n, tuple(o.shape))
        assert _lib.launch_count() == n0
    with pytest.raises(ValueError, match="mwf_iterations"):
        track.render_track(np.zeros((2, 1, 96, 64), np.float32), 1000, 8, np.zeros((1, 3000), np.float32), 48000, 11)
    with pytest.raises(ValueError, match="C = 1 or 2"):
        track.render_track(np.zeros((2, 1, 96, 64), np.float32), 1000, 8, np.zeros((3, 3000), np.float32), 48000)


def _tone_mels(stems, sr, o):
    """Ground-truth mel patches of stereo stems [K, 2, L] at sr: the 16 kHz mono down-mix through the front end."""
    mels = []
    for s in stems:
        x16 = resample(s.mean(axis=0).astype(np.float32), sr, 16000)
        mels.append(track.segment_track(x16, o)[0].squeeze(-1))
    return torch.stack(mels), int(x16.numel())


def test_dual_mono_file_gives_identical_channels_equal_to_mono():
    sr, L, o = 44100, 100_000, 8
    rng = np.random.default_rng(0)
    t = np.arange(L) / sr
    stems = np.stack([np.stack([0.3 * np.sin(2 * np.pi * 220 * t)] * 2),
                      np.stack([0.1 * rng.standard_normal(L)] * 2)])
    mels, L16 = _tone_mels(stems, sr, o)
    est = torch.stack([mels[1] - 3.0, mels[0] + 2.0]).clamp(-100, 20)      # estimates that are not the truth
    mix = stems.sum(0).astype(np.float32)
    dual = track.render_track(est, L16, o, mix, sr, 1).cpu().numpy()
    mono = track.render_track(est, L16, o, mix[:1], sr, 1).cpu().numpy()
    assert dual.shape == (2, 2, L) and mono.shape == (2, 1, L)
    np.testing.assert_array_equal(dual[:, 0], dual[:, 1])
    np.testing.assert_allclose(dual[:, 0], mono[:, 0], rtol=0, atol=1e-5 * np.abs(mix).max())


def _sdr(ref, est):
    return 10 * np.log10(np.sum(ref ** 2) / np.sum((est - ref) ** 2))


def _tone_level(x, f, sr):
    t = np.arange(x.shape[-1]) / sr
    return np.sqrt(np.sum(np.abs(x @ np.exp(-2j * np.pi * f * t)) ** 2))


def test_full_band_stems_from_ground_truth_mel_patches():
    """Stems rendered from the true sources' mel patches (BASIS bypassed) keep the bass below 133 Hz and the content
    above 8 kHz that the mel rendering drops, and follow each source's panning.  Above the mel band a bin takes the gains
    of the top covered bin (7.6 kHz), so the source with the 12 kHz tone is the one with content at the band's top edge."""
    sr, L, o = 44100, 6 * 44100 + 123, 8
    t = np.arange(L) / sr
    env = 1 + 0.5 * np.sin(2 * np.pi * 0.7 * t)
    low = env * (0.3 * np.sin(2 * np.pi * 55 * t) + 0.15 * np.sin(2 * np.pi * 110 * t) + 0.1 * np.sin(2 * np.pi * 165 * t)
                 + 0.03 * np.sin(2 * np.pi * 7500 * t) + 0.05 * np.sin(2 * np.pi * 12000 * t))
    mid = (1.2 - 0.5 * env) * (0.2 * np.sin(2 * np.pi * 660 * t + 0.3 * np.sin(2 * np.pi * 5 * t))
                               + 0.1 * np.sin(2 * np.pi * 1500 * t) + 0.05 * np.sin(2 * np.pi * 3000 * t))
    stems = np.stack([np.stack([0.9 * low, 0.3 * low]), np.stack([0.2 * mid, 1.0 * mid])])
    mix = stems.sum(0).astype(np.float32)
    mels, L16 = _tone_mels(stems, sr, o)
    mask = track.render_track(mels, L16, o, mix, sr, 1).cpu().numpy()
    np.testing.assert_allclose(mask.sum(0), mix, rtol=0, atol=1e-5)
    _, S16, _ = track.segment_track(resample(mix.mean(0), sr, 16000), o)       # the mel rendering's mixture
    mel = track.invert_track(mels, S16, L16, o, orig_sr=sr, orig_length=L).cpu().numpy()
    for k in range(2):
        sdr_mask = _sdr(stems[k], mask[k])
        sdr_mel = _sdr(stems[k], np.broadcast_to(mel[k], stems[k].shape))
        print(f"source {k + 1}: full-band SDR mask {sdr_mask:.2f} dB, mel {sdr_mel:.2f} dB")
        assert sdr_mask >= 10.0 and sdr_mask > sdr_mel
    kept = 20 * np.log10(_tone_level(mask[0], 12000, sr) / _tone_level(stems[0], 12000, sr))
    print(f"12 kHz tone in its stem: {kept:+.3f} dB")
    assert abs(kept) <= 1.0


def _write_wav24(path, data, sr):
    """data [C, n] -> 24-bit PCM."""
    pcm = np.round(np.clip(data.T.reshape(-1), -1, 1 - 2 ** -23) * 2 ** 23).astype("<i4")
    with wave.open(str(path), "wb") as w:
        w.setnchannels(data.shape[0])
        w.setsampwidth(3)
        w.setframerate(sr)
        w.writeframes(pcm.view(np.uint8).reshape(-1, 4)[:, :3].tobytes())


FLAGS = ["--model_type", "ncsn", "--version", "v2", "--n_filters", "128", "--num_classes", "2", "--sigma1", "0.05", "--T",
         "1", "--random_init", "3", "--fast"]


def test_mask_render_end_to_end(tmp_path):
    from audiosourcesep_b200 import melspec_inversion_basis as inv
    from audiosourcesep_b200.datasets.data_loader import read_wav
    from audiosourcesep_b200.run_basis_sep import cli
    sr, n = 44100, 321_987
    t = np.arange(n) / sr
    a = 0.3 * np.sin(2 * np.pi * 330 * t) + 0.1 * np.sin(2 * np.pi * 60 * t)
    b = 0.2 * np.sin(2 * np.pi * 880 * t) + 0.02 * np.sin(2 * np.pi * 11000 * t)
    _write_wav24(tmp_path / "song.wav", np.stack([a + 0.3 * b, 0.4 * a + b]), sr)
    song = str(tmp_path / "song.wav")
    x, _ = read_wav(song)
    res = cli(["r1", "r2", "r3", "--mix", song, "--render", "mask", "--output", str(tmp_path / "mask")] + FLAGS)
    mel = cli(["r1", "r2", "r3", "--mix", song, "--output", str(tmp_path / "mel")] + FLAGS)
    zm, zl = np.load(tmp_path / "mask" / "results.npz"), np.load(tmp_path / "mel" / "results.npz")
    for k in range(3):
        assert np.array_equal(zm[f"x{k + 1}"], zl[f"x{k + 1}"])
    sep = np.load(tmp_path / "mask" / "separated.npz")
    names = ("source1", "source2", "source3")
    for k, name in enumerate(names):
        with wave.open(str(tmp_path / "mask" / f"{name}.wav"), "rb") as w:
            assert (w.getframerate(), w.getnchannels(), w.getnframes(), w.getsampwidth()) == (sr, 2, n, 2)
        assert sep[f"x{k + 1}"].shape == (2, n) and sep[f"x{k + 1}"].dtype == np.float32
        assert np.array_equal(res["separated"][name], sep[f"x{k + 1}"])
    np.testing.assert_allclose(sum(sep[f"x{k + 1}"] for k in range(3)), x, rtol=0, atol=1e-4)
    assert mel["separated"]["source1"].shape == (n,)
    # the inversion CLI re-renders the same tracks from the results directory and the file
    flat = inv.main(inv.build_parser().parse_args([str(tmp_path / "mask"), "--render", "mask", "--mix", song]))
    again = np.load(tmp_path / "mask" / "inverse_mask" / "separated.npz")
    for k in range(3):
        np.testing.assert_allclose(again[f"x{k + 1}"], sep[f"x{k + 1}"], rtol=0, atol=1e-6)
        assert np.array_equal(flat[f"x{k + 1}_audio"], again[f"x{k + 1}"])
    # ... and from a different file it refuses
    _write_wav24(tmp_path / "other.wav", np.stack([a, a])[:, :-5], sr)
    with pytest.raises(ValueError, match="samples at"):
        inv.main(inv.build_parser().parse_args([str(tmp_path / "mask"), "--render", "mask", "--mix",
                                                str(tmp_path / "other.wav")]))
    # the Python entry point
    tracks, rate = track.separate_file(song, ["r1", "r2", "r3"], output=str(tmp_path / "py"), model_type="ncsn",
                                       version="v2", n_filters=128, num_classes=2, sigma1=0.05, T=1, random_init=3,
                                       fast=True, render="mask")
    assert rate == sr
    for k, name in enumerate(names):
        assert tracks[name].shape == (2, n)
        np.testing.assert_allclose(tracks[name], sep[f"x{k + 1}"], rtol=0, atol=1e-4)
    # more than two channels fail before anything runs on the device
    _write_wav24(tmp_path / "three.wav", np.stack([a, a, a])[:, :20000], sr)
    n0 = _lib.launch_count()
    with pytest.raises(ValueError, match="3 channels"):
        cli(["r1", "r2", "--mix", str(tmp_path / "three.wav"), "--render", "mask", "--output", str(tmp_path / "x")] + FLAGS)
    assert _lib.launch_count() == n0
