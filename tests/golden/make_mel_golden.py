"""Real-data fixture for the mel front / back end, cut from artefacts THE REFERENCE SHIPS
(basis_sep_results/beethoven_sonata_1_sep_1min of SamArgt/AudioSourceSep): ``mix.wav`` is the output of the reference's own
melspec_inversion_basis.py (librosa mel_to_stft + mixture phase + istft, one 2.016 s chunk per extract) for the ``mixed``
mel spectrograms stored in ``results.npz`` (librosa stft / melspectrogram / power_to_db of the real recording).
Two extracts are kept: the int16 audio chunks and their mel spectrograms.
    python tests/golden/make_mel_golden.py <reference checkout>"""
import os
import sys
import wave

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    base = os.path.join(ref, "basis_sep_results", "beethoven_sonata_1_sep_1min")
    d = np.load(os.path.join(base, "results.npz"))
    with wave.open(os.path.join(base, "mix.wav"), "rb") as w:
        assert w.getframerate() == 16000 and w.getnchannels() == 1 and w.getsampwidth() == 2
        a = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
    n = 512 * 63                                         # hop * (frames - 1): what librosa.istft returns per extract
    assert a.size == 30 * n
    keep = [0, 7]
    np.savez_compressed(os.path.join(HERE, "real_inversion.npz"), extracts=np.array(keep),
                        mix_audio_int16=np.stack([a[i * n:(i + 1) * n] for i in keep]),
                        mixed_db=np.stack([d["mixed"][i] for i in keep]).astype(np.float32))


if __name__ == "__main__":
    main(sys.argv[1])
