"""Real-audio input path on the GPU: wav files at other rates than 16 kHz through get_song_extract and run_basis_sep
--song_dir, the wav -> mel dataset builder (datasets/wav_to_spec.py), and train_glow / train_ncsn --dataset."""
import os
import re
import struct

import numpy as np
import pytest

from oracle import mel_oracle as mo
from oracle import resample_oracle as ro

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENGTH = 32640                                    # int(16000 * 2.04)


def _write(path, samples, rate, kind):
    """samples [n] or [n, channels] in [-1, 1) -> wav; kind 'pcm24' or 'float32'.  Returns what a reader must decode
    (float32 [n, channels])."""
    a = np.asarray(samples, dtype=np.float64)
    a = a[:, None] if a.ndim == 1 else a
    nch = a.shape[1]
    if kind == "pcm24":
        ints = np.clip(np.round(a * 2 ** 23), -2 ** 23, 2 ** 23 - 1).astype(np.int64)
        data = (ints.reshape(-1) & 0xFFFFFF).astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
        tag, bits, decoded = 1, 24, ints.astype(np.float32) / 8388608.0
    else:
        f = a.astype(np.float32)
        data, tag, bits, decoded = f.astype("<f4").tobytes(), 3, 32, f
    fmt = struct.pack("<HHIIHH", tag, nch, rate, rate * nch * bits // 8, nch * bits // 8, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    body += b"\x00" * (len(data) & 1)
    with open(path, "wb") as fh:
        fh.write(b"RIFF" + struct.pack("<I", len(body)) + body)
    return decoded


def _music(n, sr, f0, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    return 0.3 * np.sin(2 * np.pi * f0 * t) * (1 + 0.5 * np.sin(2 * np.pi * 2 * t)) + 0.01 * rng.standard_normal(n)


def _oracle_patches(decoded, rate):
    """Oracle patches of one file: mean over channels (float32, as read), float64 resampling, float32 PCM, windows."""
    mono = decoded.mean(axis=1) if decoded.shape[1] > 1 else decoded[:, 0]
    y = mono if rate == 16000 else ro.resample(mono, rate, 16000).astype(np.float32)
    n = y.size // LENGTH
    return [mo.melspectrogram_db(y[i * LENGTH:(i + 1) * LENGTH])[0] for i in range(n)], y.size


def test_get_song_extract_at_44k(tmp_path):
    from audiosourcesep_b200.datasets.data_loader import get_song_extract
    sr = 44100
    n = int(5.3 * LENGTH / 16000 * sr)
    dec = {}
    for name, f0 in (("mix", 330.0), ("piano", 262.0), ("violin", 880.0)):
        stereo = np.stack([_music(n, sr, f0, 1), _music(n, sr, f0 * 1.01, 2)], axis=1)
        dec[name] = _write(tmp_path / f"{name}.wav", stereo, sr, "pcm24")
    kw = dict(length_sec=2.04, fmin=125, fmax=7600, sr=16000, dbmin=-100, dbmax=20, n_fft=2048, hop_length=512, n_mels=96,
              use_dB=True)
    mel_spec, raw_audio, stft_mixture = get_song_extract(str(tmp_path / "mix.wav"), str(tmp_path / "piano.wav"),
                                                         str(tmp_path / "violin.wav"), 2 * 2.04, **kw)
    assert stft_mixture.shape == (2, 1025, 64)
    for name, mel in zip(("mix", "piano", "violin"), mel_spec):
        want, _ = _oracle_patches(dec[name], sr)
        got = mel.cpu().numpy()[..., 0]
        assert got.shape == (2, 96, 64)
        err = max(np.max(np.abs(got[i] - want[2 + i])) for i in range(2))          # windows 2, 3 (the first two skipped)
        print(f"{name}: max |dB error| {err:.2e}")
        assert err <= 2e-3


def test_run_basis_sep_song_dir_at_44k_24bit_stereo(tmp_path):
    from audiosourcesep_b200.run_basis_sep import build_parser, main, merge_config
    sr = 44100
    n = int(4.5 * LENGTH / 16000 * sr)
    song = tmp_path / "song"
    song.mkdir()
    p = np.stack([_music(n, sr, 330.0, 1), _music(n, sr, 331.0, 2)], axis=1)
    v = np.stack([_music(n, sr, 880.0, 3), _music(n, sr, 881.0, 4)], axis=1)
    for name, a in (("piano", p), ("violin", v), ("mix", 0.5 * (p + v))):
        _write(song / f"{name}.wav", a, sr, "pcm24")
    out = tmp_path / "sep"
    cfg_path = os.path.join(ROOT, "configs", "melspec_ncsnv2.yml")
    args = merge_config(build_parser().parse_args(["unused1", "unused2", "--output", str(out), "--model_type", "ncsn", "--song_dir",
                                                   str(song), "--random_init", "3", "--n_mixed", "2", "--config", cfg_path]))
    args.config = None
    args.T, args.num_classes, args.sigma1 = 1, 2, 0.05
    main(args)
    z = np.load(out / "results.npz")
    assert z["stft_mixture"].shape == (2, 1025, 64) and np.abs(z["stft_mixture"]).max() > 1.0
    assert z["mixed"].shape == (2, 96, 64) and np.all(np.isfinite(z["x1"])) and np.all(np.isfinite(z["x2"]))


@pytest.fixture(scope="module")
def dataset_files(tmp_path_factory):
    """Two mixed-format files: 44.1 kHz 24-bit stereo (3 windows + a remainder) and 48 kHz float32 mono (2 + remainder)."""
    d = tmp_path_factory.mktemp("wavs")
    na = int(3.4 * 44100 * 2.04)
    a = _write(d / "a.wav", np.stack([_music(na, 44100, 330.0, 5), _music(na, 44100, 440.0, 6)], axis=1), 44100, "pcm24")
    b = _write(d / "b.wav", 0.5 * _music(int(2.7 * 48000 * 2.04), 48000, 523.0, 7), 48000, "float32")
    return d, {"a.wav": (a, 44100), "b.wav": (b, 48000)}


def test_wav_to_spec_counts_values_and_split(dataset_files, tmp_path):
    from audiosourcesep_b200.datasets.wav_to_spec import build_parser, main
    d, decoded = dataset_files
    out = tmp_path / "ds.npz"
    res = main(build_parser().parse_args([str(d), "--output", str(out), "--test_fraction", "0.4", "--seed", "3", "--chunk", "2"]))
    z = np.load(out)
    assert [os.path.basename(f) for f in z["files"]] == ["a.wav", "b.wav"]
    assert z["train"].dtype == np.float32 and z["train"].shape[1:] == (96, 64, 1)
    assert z["train_file"].dtype == np.int32 and int(z["sr"]) == 16000 and int(z["n_mels"]) == 96
    # patch count: sum over files of floor(resampled length / 32640)
    want, count = [], 0
    for i, name in enumerate(("a.wav", "b.wav")):
        pats, n_res = _oracle_patches(*decoded[name])
        assert n_res == int(np.ceil(decoded[name][0].shape[0] * 16000 / decoded[name][1]))
        count += n_res // LENGTH
        want += [(i, p) for p in pats]
    n_train, n_test = z["train"].shape[0], z["test"].shape[0]
    assert n_train + n_test == count == 5 and n_test == 2
    # every patch matches the oracle of its window (the split keeps window order within each set)
    from audiosourcesep_b200.datasets.wav_to_spec import split
    is_test = split(count, 0.4, 3)
    for k, (i, p) in enumerate(want):
        j = int(np.sum(is_test[:k] == is_test[k]))
        arr, owner = (z["test"], z["test_file"]) if is_test[k] else (z["train"], z["train_file"])
        assert owner[j] == i
        assert np.max(np.abs(arr[j, ..., 0] - p)) <= 2e-3
    # the split is reproducible from the seed
    res2 = main(build_parser().parse_args([str(d), "--output", str(tmp_path / "ds2.npz"), "--test_fraction", "0.4", "--seed", "3"]))
    assert np.array_equal(res2["test"], res["test"]) and np.array_equal(res2["train_file"], res["train_file"])


@pytest.fixture(scope="module")
def training_set(dataset_files, tmp_path_factory):
    from audiosourcesep_b200.datasets.wav_to_spec import build_dataset
    out = tmp_path_factory.mktemp("ds") / "train.npz"
    build_dataset([str(dataset_files[0])], str(out), test_fraction=0.4, seed=1)
    return out


def _test_losses(text):
    vals = [float(v) for v in re.findall(r"Epoch \d{3}: Test Loss: (\S+)", text)]
    assert all(np.isfinite(vals))
    return vals


def test_train_glow_with_dataset_logs_the_test_loss(training_set, tmp_path, capsys):
    import torch
    from audiosourcesep_b200 import GlowConfig
    from audiosourcesep_b200.flow_models.flow_builder import build_glow
    from audiosourcesep_b200.datasets.wav_to_spec import load_patches
    from audiosourcesep_b200.train_glow import build_parser, main
    out = tmp_path / "glow"
    main(build_parser().parse_args(["--dataset", str(training_set), "--output", str(out), "--K", "1", "--n_filters", "64",
                                    "--n_epochs", "2", "--batch_size", "2", "--learning_rate", "1e-4"]))
    losses = _test_losses(capsys.readouterr().out)
    assert len(losses) == 2
    # the last logged test loss is -log_prob of the test patches under the saved weights
    _, test = load_patches(str(training_set), 96, 64)
    with np.load(out / "weights.npz") as w:
        params = {k: w[k] for k in w.files}
    flow = build_glow(None, [96, 64, 1], L=3, K=1, n_filters=64, learntop=True, data_type="melspec", minval=-100.0, maxval=20.0,
                      use_logit=False, params=params)
    again = float(-flow.log_prob(torch.as_tensor(test)).double().mean())
    print(f"logged {losses[-1]:.6f}, recomputed {again:.6f}")
    assert abs(losses[-1] - again) <= 1e-5 * abs(again)


def test_train_noisy_glow_with_dataset_logs_the_test_loss(training_set, tmp_path, capsys):
    from audiosourcesep_b200.train_glow import build_parser, main
    main(build_parser().parse_args(["--dataset", str(training_set), "--output", str(tmp_path / "noisy"), "--noisy", "--K", "1",
                                    "--n_filters", "64", "--n_epochs", "1", "--batch_size", "2", "--num_classes", "2",
                                    "--sigma1", "1.0", "--sigmaL", "0.1", "--learning_rate", "1e-4"]))
    text = capsys.readouterr().out
    assert text.count("Training at noise level") == 2 and len(_test_losses(text)) == 2
    assert os.path.exists(tmp_path / "noisy" / "sigma_0.1" / "weights.npz")


def test_train_ncsn_with_dataset_logs_the_test_loss(training_set, tmp_path, capsys):
    from audiosourcesep_b200.train_ncsn import build_parser, main
    hist = main(build_parser().parse_args(["--dataset", str(training_set), "--output", str(tmp_path / "ncsn"), "--version", "v2",
                                           "--n_filters", "128", "--sigma1", "1.0", "--num_classes", "5", "--progression",
                                           "logarithmic", "--n_epochs", "2", "--batch_size", "2", "--learning_rate", "1e-5"]))
    text = capsys.readouterr().out
    assert len(hist) == 2 and text.count("Train Loss:") == 2 and len(_test_losses(text)) == 2


def test_dataset_shape_mismatch_is_refused(training_set, tmp_path):
    from audiosourcesep_b200.train_glow import build_parser, main
    with pytest.raises(ValueError, match="expects"):
        main(build_parser().parse_args(["--dataset", str(training_set), "--output", str(tmp_path / "x"), "--height", "32",
                                        "--width", "32", "--K", "1", "--n_filters", "64"]))
