"""CPU checks of the whole-track segmentation (audiosourcesep_b200/track.py, restated in oracle/track_oracle.py), of the
restated cross-fade, and of the flag rules of run_basis_sep --mix."""
import math

import numpy as np
import pytest

from audiosourcesep_b200 import run_basis_sep, track
from oracle import mel_oracle as mo
from oracle import track_oracle as to

V, P8 = 512 * 63, 512 * 63 - 512 * 8


def test_constants_are_the_reference_extract():
    assert track.WINDOW == to.WINDOW == 32640
    assert track.SPAN == to.SPAN == V == 32256
    assert track.FRAMES == 64 and track.MAX_OVERLAP_FRAMES == 31


@pytest.mark.parametrize("L, n_seg", [(1, 1), (1000, 1), (V - 1, 1), (V, 1), (V + 1, 2), (V + P8, 2), (V + 3 * P8, 4),
                                      (V + 3 * P8 + 1, 5)])
def test_segment_count_and_starts(L, n_seg):
    starts = track.segment_starts(L, 8)
    assert starts.dtype == np.int64 and len(starts) == n_seg
    assert np.array_equal(starts, np.arange(n_seg) * P8)
    assert np.array_equal(starts, to.segment_starts(L, 8))
    # the last segment reaches the end of the track, the one before it does not
    assert starts[-1] + V >= L
    if n_seg > 1:
        assert starts[-2] + V < L


def test_segment_count_of_a_44k1_length_that_is_not_round():
    orig = 321_987                                      # 7.3 s at 44.1 kHz
    L = math.ceil(orig * 16000 / 44100)                 # what the resampler's length fix gives
    for o in (0, 1, 8, 31):
        P = V - 512 * o
        starts = track.segment_starts(L, o)
        assert len(starts) == 1 + math.ceil((L - V) / P)
        assert np.array_equal(starts, to.segment_starts(L, o))
        assert starts[-1] + V >= L > starts[-1]


@pytest.mark.parametrize("o", [0, 1, 8, 31])
def test_crossfade_weights_sum_to_one_everywhere(o):
    L = 3 * V + 12345
    c = to.crossfade_weights(L, o)
    np.testing.assert_allclose(c.sum(0), 1.0, rtol=0, atol=1e-12)
    assert np.all((c > 0).sum(0) <= 2)                  # at most two segments cover any sample
    if o == 0:
        assert np.all((c > 0).sum(0) == 1) and set(np.unique(c)) <= {0.0, 1.0}
    else:
        O, s1 = 512 * o, V - 512 * o
        ramp = c[1, s1: s1 + O]
        assert np.all(np.diff(ramp) > 0) and ramp[0] > 0 and ramp[-1] < 1
        assert c[0, 0] == 1.0 and c[-1, L - 1] == 1.0   # no ramp at either end of the track


@pytest.mark.parametrize("o", [0, 8, 31])
def test_oracle_reconstructs_the_track_from_its_own_segments(o):
    rng = np.random.default_rng(o)
    L = 2 * V + 7777
    x = rng.standard_normal(L) * 0.3
    S = np.stack([mo.stft(w) for w in to.windows(x, o)])
    y = to.istft_track(S, o, L)
    np.testing.assert_allclose(y, x, rtol=0, atol=1e-5)


def _args(argv):
    return run_basis_sep.build_parser().parse_args(argv)


def test_mix_flag_rules():
    run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav"]))
    run_basis_sep.check_mix_args(_args(["a", "b", "--song_dir", "s"]))        # no --mix: nothing to check
    with pytest.raises(ValueError, match="--song_dir"):
        run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav", "--song_dir", "s"]))
    with pytest.raises(ValueError, match="--synthetic"):
        run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav", "--synthetic"]))
    for bad in ("32", "-1"):
        with pytest.raises(ValueError, match="overlap_frames"):
            run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav", "--overlap_frames", bad]))
    run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav", "--overlap_frames", "31"]))
    run_basis_sep.check_mix_args(_args(["a", "b", "--mix", "m.wav", "--overlap_frames", "0"]))
    with pytest.raises(ValueError):
        track.segment_starts(100, 32)
    # a --sources list of the wrong length fails before the separation runs, not after it
    with pytest.raises(ValueError, match="--sources"):
        run_basis_sep.check_mix_args(_args(["a", "b", "c", "--mix", "m.wav", "--sources", "x,y"]))


def test_mix_output_names():
    assert run_basis_sep.source_names(_args(["a", "b", "--mix", "m.wav"])) == ["piano", "violin"]
    assert run_basis_sep.source_names(_args(["a", "b", "c", "--mix", "m.wav"])) == ["source1", "source2", "source3"]
    assert run_basis_sep.source_names(_args(["a", "b", "c", "--mix", "m.wav", "--sources", "bass,drums,vocals"])) == \
        ["bass", "drums", "vocals"]
    with pytest.raises(ValueError, match="--sources"):
        run_basis_sep.source_names(_args(["a", "b", "c", "--mix", "m.wav", "--sources", "x,y"]))


def test_merge_config_keeps_the_mix_fields(tmp_path):
    yml = tmp_path / "c.yml"
    yml.write_text("T: 7\noverlap_frames: 3\n")
    merged = run_basis_sep.merge_config(_args(["a", "b", "--config", str(yml), "--mix", "m.wav", "--overlap_frames", "5",
                                               "--wiener_filter"]))
    assert merged.mix == "m.wav" and merged.overlap_frames == 5 and merged.wiener_filter and merged.T == 7
