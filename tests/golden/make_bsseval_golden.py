"""Golden vectors of BSS Eval v4 and the ideal-mask systems, produced by RUNNING THE REFERENCE ITSELF
(bsseval_v4.py, oracle_systems.py of SamArgt/AudioSourceSep: pure numpy / scipy, importable with the ``np.float``
alias that NumPy >= 1.24 removed).   python tests/golden/make_bsseval_golden.py <reference checkout>
"""
import os
import sys
import types

import numpy as np

np.float = float                                      # bsseval_v4.py:507, oracle_systems.py use the removed alias
sys.path.insert(0, sys.argv[1])
import bsseval_v4 as bv  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def signals(seed, n):
    rng = np.random.default_rng(seed)
    s = rng.standard_normal((2, n))
    s[0] = np.convolve(s[0], np.hanning(32), "same")
    s[1] = np.convolve(s[1], np.ones(8) / 8, "same")
    est = np.stack([0.8 * s[0] + 0.2 * s[1] + 0.05 * rng.standard_normal(n),
                    0.7 * s[1] + 0.1 * s[0] + 0.05 * rng.standard_normal(n)])
    return s, est


def main():
    out = {}
    # 1. synthetic signals, framed evaluation with global filters (the v4 default)
    s, e = signals(0, 20000)
    for name, kw in (("v4_framed", dict(window=8000, hop=6000, filters_len=64)),
                     ("v4_whole_512", dict(window=np.inf, hop=np.inf, filters_len=512)),
                     ("v4_framewise", dict(window=8000, hop=6000, filters_len=64, framewise_filters=True)),
                     ("v4_perm", dict(window=8000, hop=6000, filters_len=64, compute_permutation=True))):
        est = e[::-1].copy() if name == "v4_perm" else e             # swapped estimates: the permutation must undo it
        r = bv.bss_eval(s[..., None], est[..., None], **kw)
        for k, v in zip(("sdr", "isr", "sir", "sar", "perm"), r):
            out[f"{name}/{k}"] = np.asarray(v, dtype=np.float64)
    r = bv.bss_eval_sources(s[..., None], e[..., None], compute_permutation=False)      # v3 criteria, framewise filters
    for k, v in zip(("sdr", "sir", "sar", "perm"), r):
        out[f"v3_sources/{k}"] = np.asarray(v, dtype=np.float64)
    # 2. a silent estimate in the second window -> NaN row
    e2 = e.copy()
    e2[1, 6000:14000] = 0.0
    r = bv.bss_eval(s[..., None], e2[..., None], window=8000, hop=6000, filters_len=64)
    for k, v in zip(("sdr", "isr", "sir", "sar", "perm"), r):
        out[f"v4_silent/{k}"] = np.asarray(v, dtype=np.float64)
    # 3. the mel-domain SDR of SURVEY 8(d): flattened normalised patches of the shipped results.npz
    d = np.load(os.path.join(HERE, "real_patches.npz"))
    norm = lambda x: ((x.astype(np.float64) + 100.0) / 120.0).reshape(-1)
    refs = np.stack([norm(d["gt1"]), norm(d["gt2"])])
    ests = np.stack([norm(d["x1"]), norm(d["x2"])])
    r = bv.bss_eval(refs[..., None], ests[..., None], window=np.inf, hop=np.inf, filters_len=512)
    for k, v in zip(("sdr", "isr", "sir", "sar", "perm"), r):
        out[f"mel_real/{k}"] = np.asarray(v, dtype=np.float64)
    # 4. ideal masks (oracle_systems.py:264-350); the module imports plotting / audio packages at the top, stub them
    for mod in ("soundfile", "librosa", "librosa.display", "matplotlib", "matplotlib.pyplot", "museval", "musdb", "norbert"):
        sys.modules.setdefault(mod, types.ModuleType(mod))
    try:
        import oracle_systems as osys
        rng = np.random.default_rng(1)
        srcs = rng.random((2, 3, 96, 64)).astype(np.float64) ** 2
        mix = srcs.sum(0) * (1.0 + 0.05 * rng.standard_normal((3, 96, 64)))
        out["mask/sources"] = srcs
        out["mask/mixture"] = mix
        out["mask/irm"] = osys.IRM_melspec(mix, srcs)
        out["mask/ibm"] = osys.IBM_melspec(mix, srcs, theta=0.5)
    except Exception as ex:                           # pragma: no cover
        print("oracle_systems could not be imported:", ex)
    np.savez_compressed(os.path.join(HERE, "bsseval_v4.npz"), **out)
    for k in sorted(out):
        if out[k].size <= 12:
            print(k, out[k].tolist())


if __name__ == "__main__":
    main()
