"""Regenerates the fixtures of tests/golden/ from a READ-ONLY checkout of the reference (SamArgt/AudioSourceSep):
    python tests/golden/make_golden.py <reference checkout>
Produces
  sigmas_v1.json     the noise schedule printed by the reference's own BASIS run
                     (basis_sep_results/beethoven_sonata_1_sep_1min/out.log:44-116)
  real_patches.npz   the first 4 of the 30 real mel patches (gt1, gt2, mixed; dB) and the
                     reference's separated outputs (x1, x2) from
                     basis_sep_results/beethoven_sonata_1_sep_1min/results.npz
  param_counts.json  trainable-parameter known answers (trained_ncsn/.../out.log:35)
"""
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    run = os.path.join(ref, "basis_sep_results", "beethoven_sonata_1_sep_1min")
    sig = []
    dur = None
    with open(os.path.join(run, "out.log")) as f:
        for line in f:
            m = re.match(r"Sigma = ([0-9.eE+-]+) \((\d+) / (\d+)\)", line)
            if m:
                sig.append(float(m.group(1)))
            m = re.match(r"Duration: ([0-9.]+) seconds", line)
            if m:
                dur = float(m.group(1))
    with open(os.path.join(HERE, "sigmas_v1.json"), "w") as f:
        json.dump({"source": "basis_sep_results/beethoven_sonata_1_sep_1min/out.log:44-116",
                   "sigma1": 1.0, "sigmaL": 0.01, "num_classes": 10, "progression": "logarithmic",
                   "printed": sig, "duration_s": dur, "n_mixed": 30, "T": 100}, f, indent=1)
    d = np.load(os.path.join(run, "results.npz"))
    np.savez_compressed(os.path.join(HERE, "real_patches.npz"), **{k: d[k][:4] for k in ("gt1", "gt2", "mixed", "x1", "x2")})
    with open(os.path.join(ref, "trained_ncsn", "ncsn_piano_192_32_dB_custom_loop", "out.log")) as f:
        txt = f.read()
    m = re.search(r"([0-9][0-9,]{6,})", txt.split("\n")[34])
    with open(os.path.join(HERE, "param_counts.json"), "w") as f:
        json.dump({"source": "trained_ncsn/ncsn_piano_192_32_dB_custom_loop/out.log:35", "line": txt.split("\n")[34],
                   "ncsn_v1_ngf192_classes10": 67464769}, f, indent=1)
    print(sig, dur, txt.split("\n")[34])


if __name__ == "__main__":
    main(sys.argv[1])
