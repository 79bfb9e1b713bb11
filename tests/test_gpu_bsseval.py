"""GPU parity tests of BSS Eval v4 and the ideal masks against outputs of THE REFERENCE ITSELF
(tests/golden/bsseval_v4.npz, written by tests/golden/make_bsseval_golden.py from the reference's bsseval_v4.py and
oracle_systems.py) -- a reference-pinned oracle, not a restatement."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "bsseval_v4.npz"))


def _signals(seed, n):
    rng = np.random.default_rng(seed)
    s = rng.standard_normal((2, n))
    s[0] = np.convolve(s[0], np.hanning(32), "same")
    s[1] = np.convolve(s[1], np.ones(8) / 8, "same")
    est = np.stack([0.8 * s[0] + 0.2 * s[1] + 0.05 * rng.standard_normal(n),
                    0.7 * s[1] + 0.1 * s[0] + 0.05 * rng.standard_normal(n)])
    return s, est


def _check(name, got, keys=("sdr", "isr", "sir", "sar", "perm"), tol=1e-6):
    for k, g in zip(keys, got):
        want = GOLD[f"{name}/{k}"]
        g = np.asarray(g, dtype=np.float64)
        assert g.shape == want.shape, (name, k, g.shape, want.shape)
        assert np.array_equal(np.isnan(g), np.isnan(want)), (name, k)
        err = np.nanmax(np.abs(g - want)) if np.any(~np.isnan(want)) else 0.0
        print(f"{name}/{k}: max |delta| = {err:.3e} dB")
        assert err <= tol, (name, k, g, want)


@pytest.mark.parametrize("name,kw", [
    ("v4_framed", dict(window=8000, hop=6000, filters_len=64)),
    ("v4_whole_512", dict(window=np.inf, hop=np.inf, filters_len=512)),
    ("v4_framewise", dict(window=8000, hop=6000, filters_len=64, framewise_filters=True)),
    ("v4_perm", dict(window=8000, hop=6000, filters_len=64, compute_permutation=True)),
])
def test_bss_eval_matches_the_reference(name, kw):
    from audiosourcesep_b200 import bsseval_v4 as bv
    s, e = _signals(0, 20000)
    est = e[::-1].copy() if name == "v4_perm" else e
    _check(name, bv.bss_eval(s[..., None], est[..., None], **kw))


def test_bss_eval_sources_v3_criteria_and_silent_windows():
    from audiosourcesep_b200 import bsseval_v4 as bv
    s, e = _signals(0, 20000)
    _check("v3_sources", bv.bss_eval_sources(s[..., None], e[..., None], compute_permutation=False), keys=("sdr", "sir", "sar", "perm"))
    e2 = e.copy()
    e2[1, 6000:14000] = 0.0
    _check("v4_silent", bv.bss_eval(s[..., None], e2[..., None], window=8000, hop=6000, filters_len=64))
    with pytest.raises(ValueError):
        bv.bss_eval(s[..., None], e[:, :100, None])
    assert all(v.size == 0 for v in bv.bss_eval(np.zeros((0, 0, 1)), np.zeros((0, 0, 1))))


def test_mel_domain_sdr_of_the_shipped_separation():
    """SURVEY 8(d): mel-domain SDR on the flattened normalised patches of the reference's own results.npz."""
    from audiosourcesep_b200 import bsseval_v4 as bv
    d = np.load(os.path.join(HERE, "golden", "real_patches.npz"))
    norm = lambda x: ((x.astype(np.float64) + 100.0) / 120.0).reshape(-1)
    refs = np.stack([norm(d["gt1"]), norm(d["gt2"])])
    ests = np.stack([norm(d["x1"]), norm(d["x2"])])
    _check("mel_real", bv.bss_eval(refs[..., None], ests[..., None], window=np.inf, hop=np.inf, filters_len=512), tol=1e-5)


def test_ideal_masks_match_the_reference():
    from audiosourcesep_b200 import oracle_systems as osys
    if "mask/irm" not in GOLD.files:
        pytest.skip("mask goldens were not generated")
    srcs, mix = GOLD["mask/sources"], GOLD["mask/mixture"]
    irm = osys.IRM_melspec(mix, srcs)
    ibm = osys.IBM_melspec(mix, srcs, theta=0.5)
    assert np.max(np.abs(irm - GOLD["mask/irm"])) <= 2e-6 * np.max(np.abs(GOLD["mask/irm"]))
    # the binary decision is taken on float32 inputs here and float64 in the reference: bins within 1e-6 of the threshold may flip
    want = GOLD["mask/ibm"]
    ratio = srcs / (np.finfo(float).eps + mix)
    decided = np.abs(ratio - 0.5) > 1e-6
    assert np.max(np.abs(ibm - want)[decided]) <= 2e-6 * np.max(np.abs(want))
    assert decided.mean() > 0.999
