"""Whole-track separation on the GPU (run_basis_sep --mix): the track iSTFT kernel against oracle/track_oracle.py, exact
reconstruction of a mixture from its own segments, the Wiener sum, alignment over the whole track, and the end-to-end CLI
on a mixture-only 44.1 kHz 24-bit stereo file."""
import wave

import numpy as np
import pytest
import torch

from audiosourcesep_b200 import _lib, melspec, track
from oracle import track_oracle as to

pytestmark = pytest.mark.gpu

V = 512 * 63


def _tones(L, sr=16000, seed=0):
    rng = np.random.default_rng(seed)
    t = np.arange(L) / sr
    piano = 0.3 * np.sin(2 * np.pi * 330 * t) * (1 + 0.5 * np.sin(2 * np.pi * 2 * t)) + 0.002 * rng.standard_normal(L)
    violin = 0.2 * np.sin(2 * np.pi * 880 * t + 0.3 * np.sin(2 * np.pi * 5 * t)) + 0.002 * rng.standard_normal(L)
    return piano, violin


@pytest.mark.parametrize("S", list(range(1, 9)))
def test_track_kernel_matches_the_oracle(S):
    o = [0, 1, 8, 31][S % 4]
    P, O = V - 512 * o, 512 * o
    n_seg = 1 + S % 3 + 1                                   # 2..4 segments
    L = (n_seg - 1) * P + V - 1234 - 17 * S                 # the last segment is partial, L is not a multiple of P
    assert len(to.segment_starts(L, o)) == n_seg
    g = torch.Generator().manual_seed(S)
    spec = torch.complex(torch.randn(S, n_seg, 1025, 64, generator=g), torch.randn(S, n_seg, 1025, 64, generator=g)) * 20
    got = melspec.istft_track(spec.cuda(), o, L).cpu().numpy()
    assert got.shape == (S, L) and got.dtype == np.float32
    spec_np = spec.numpy().astype(np.complex64)
    for s in range(S):
        want = to.istft_track(spec_np[s], o, L)
        assert np.max(np.abs(want)) > 0.1
        np.testing.assert_allclose(got[s], want, rtol=0, atol=1e-6)
        # the overlap boundary of segments 0 and 1 and the end of the last, partial segment
        edges = [P - 1, P, P + O // 2, V - 1, V, L - 1] if O else [P - 1, P, L - 1]
        np.testing.assert_allclose(got[s, edges], want[edges], rtol=0, atol=1e-6)


def test_track_kernel_rejects_bad_arguments():
    spec = torch.zeros(2, 3, 1025, 64, dtype=torch.complex64, device="cuda")
    P = V - 512 * 8
    melspec.istft_track(spec, 8, 2 * P + V)                 # the longest track three segments cover
    for o, L in ((32, 1000), (-1, 1000), (8, 2 * P + V + 1)):
        with pytest.raises(_lib.AsepError) as e:
            melspec.istft_track(spec, o, L)
        assert e.value.code == -1                           # ASEP_ERR_BAD_ARG
    with pytest.raises(ValueError):
        melspec.istft_track(spec[0], 8, 1000)


@pytest.mark.parametrize("o", [0, 8, 31])
def test_exact_reconstruction_from_the_mixture_segments(o):
    L = 123457
    piano, violin = _tones(L)
    x = (piano + violin).astype(np.float32)
    _, S, starts = track.segment_track(x, o)
    assert S.shape == (len(starts), 1025, 64)
    y = melspec.istft_track(S[None], o, L)[0].cpu().numpy()
    np.testing.assert_allclose(y, x, rtol=0, atol=1e-5)


def test_wiener_outputs_sum_to_the_mixture():
    L, o, K = 100003, 8, 3
    rng = np.random.default_rng(3)
    stems = [rng.standard_normal(L).astype(np.float32) * a for a in (0.3, 0.1, 0.05)]
    mix = np.sum(stems, axis=0).astype(np.float32)
    _, S_mix, _ = track.segment_track(mix, o)
    mags = torch.stack([track.segment_track(s, o)[1].abs() for s in stems])
    cs = melspec.stft_filter(mags, S_mix, True)
    out = melspec.istft_track(cs, o, L).cpu().numpy()
    assert out.shape == (K, L)
    np.testing.assert_allclose(out.sum(0), mix, rtol=0, atol=1e-5)


@pytest.mark.parametrize("wiener", [True, False])
@pytest.mark.parametrize("o", [0, 8])
def test_alignment_over_the_whole_track(o, wiener):
    """The stems' own mel spectrograms through invert_track come back aligned with the stems over every sample of the track.
    With the Wiener filter they score > 8 dB SDR against the stems (a track lagging 384 samples per segment scores below
    5 dB).  With the mixture's phase every sample equals the existing per-extract inversion (stft_inversion_fn) of the
    segment covering it, placed at that segment's start and cross-faded with its neighbour."""
    from audiosourcesep_b200 import melspec_inversion_basis as inv
    L = 84800 + 313
    piano, violin = _tones(L)
    mix = piano + violin
    mels = torch.stack([track.segment_track(s.astype(np.float32), o)[0].squeeze(-1) for s in (piano, violin)])
    _, S_mix, starts = track.segment_track(mix.astype(np.float32), o)
    out = track.invert_track(mels, S_mix, L, o, wiener_filter=wiener).cpu().numpy()
    assert out.shape == (2, L)
    for y, ref in zip(out, (piano, violin)):
        sdr = 10 * np.log10(np.sum(ref ** 2) / np.sum((y - ref) ** 2))
        print(f"overlap {o}, wiener {wiener}: SDR {sdr:.1f} dB over {L} samples")
        if wiener:
            assert sdr > 8.0
    if not wiener:
        per_extract = inv.stft_inversion_fn()(([m.cpu().numpy() for m in mels], S_mix.cpu().numpy()))
        c = to.crossfade_weights(L, o)
        for k in range(2):
            assert per_extract[k].shape == (len(starts), V)
            want = np.zeros(L)
            for i, s in enumerate(starts):
                hi = min(L, int(s) + V)
                want[s:hi] += c[i, s:hi] * per_extract[k][i, : hi - s]
            want /= c.sum(0)
            np.testing.assert_allclose(out[k], want, rtol=0, atol=1e-6)


def _write_wav24_stereo(path, data, sr):
    pcm = np.round(np.clip(data, -1, 1 - 2 ** -23) * 2 ** 23).astype("<i4")
    b = pcm.view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    with wave.open(str(path), "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(3)
        w.setframerate(sr)
        w.writeframes(b)


def test_mix_only_directory_end_to_end(tmp_path):
    from audiosourcesep_b200 import melspec_inversion_basis as inv
    from audiosourcesep_b200.run_basis_sep import cli
    sr, n = 44100, 321_987                                  # about 7.3 s
    piano, violin = _tones(n, sr)
    third = 0.1 * np.sin(2 * np.pi * 150 * np.arange(n) / sr)
    mix = piano + violin + third
    stereo = np.stack([mix, 0.9 * mix], axis=1).reshape(-1)
    song = tmp_path / "song"
    song.mkdir()
    _write_wav24_stereo(song / "mix.wav", stereo, sr)
    out = tmp_path / "sep"
    flags = ["--model_type", "ncsn", "--version", "v2", "--n_filters", "128", "--num_classes", "2", "--sigma1", "0.05",
             "--T", "1", "--random_init", "3", "--fast"]
    res = cli(["r1", "r2", "r3", "--mix", str(song / "mix.wav"), "--output", str(out)] + flags)
    L16 = int(np.ceil(n * 16000 / sr))
    n_seg = len(track.segment_starts(L16, 8))
    z = np.load(out / "results.npz")
    assert sorted(z.files) == sorted(["x1", "x2", "x3", "mixed", "stft_mixture", "segment_start", "track_length", "orig_sr",
                                      "orig_length", "overlap_frames"])
    assert z["x1"].shape == (n_seg, 96, 64) and z["stft_mixture"].shape == (n_seg, 1025, 64)
    assert z["segment_start"].dtype == np.int64 and np.array_equal(z["segment_start"], track.segment_starts(L16, 8))
    assert int(z["track_length"]) == L16 and int(z["orig_sr"]) == sr and int(z["orig_length"]) == n
    assert int(z["overlap_frames"]) == 8
    sep = np.load(out / "separated.npz")
    for k, name in enumerate(("source1", "source2", "source3")):
        with wave.open(str(out / f"{name}.wav"), "rb") as w:
            assert w.getframerate() == sr and w.getnframes() == n and w.getnchannels() == 1 and w.getsampwidth() == 2
        t = sep[f"x{k + 1}"]
        assert t.shape == (n,) and t.dtype == np.float32 and np.all(np.isfinite(t))
        assert np.array_equal(res["separated"][name], t)
    # the inversion CLI on the same results directory writes the same tracks
    flat = inv.main(inv.build_parser().parse_args([str(out)]))
    inv_dir = out / "inverse_reuse_phase_frame"
    again = np.load(inv_dir / "separated.npz")
    for k in range(3):
        np.testing.assert_allclose(again[f"x{k + 1}"], sep[f"x{k + 1}"], rtol=0, atol=1e-6)
        assert np.array_equal(flat[f"x{k + 1}_audio"], again[f"x{k + 1}"])
        with wave.open(str(inv_dir / f"sep{k + 1}.wav"), "rb") as w:
            assert w.getframerate() == sr and w.getnframes() == n
    with pytest.raises(ValueError, match="Griffin-Lim"):
        inv.main(inv.build_parser().parse_args([str(out), "--algorithm", "griffin"]))
    # the Python entry point runs the same separation
    tracks, rate = track.separate_file(str(song / "mix.wav"), ["r1", "r2", "r3"], output=str(tmp_path / "sep_py"),
                                       model_type="ncsn", version="v2", n_filters=128, num_classes=2, sigma1=0.05, T=1,
                                       random_init=3, fast=True)
    assert rate == sr and sorted(tracks) == ["source1", "source2", "source3"]
    for k, name in enumerate(("source1", "source2", "source3")):     # same seeds; summation order may differ in the last bits
        np.testing.assert_allclose(tracks[name], sep[f"x{k + 1}"], rtol=0, atol=1e-4)
    # flag rules hold before anything runs on the device
    with pytest.raises(ValueError, match="--song_dir"):
        cli(["r1", "r2", "--mix", str(song / "mix.wav"), "--song_dir", str(song), "--output", str(tmp_path / "x")])
