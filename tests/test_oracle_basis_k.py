"""CPU checks of the K-source BASIS restatement (oracle/basis_oracle.py) and of the K-source CLI logic of run_basis_sep."""
import argparse

import numpy as np
import pytest

from audiosourcesep_b200 import run_basis_sep, synthetic
from oracle import basis_k_oracle as bko
from oracle import basis_oracle as bo


def _states(K, shape, seed):
    rng = np.random.default_rng(seed)
    return [rng.uniform(-0.5, 1.5, shape).astype(np.float32) for _ in range(K)]


def test_k2_update_and_run_equal_the_two_source_oracle_bitwise():
    g, grad_g = bo.mixing_process("melspec", "dB")
    sig = bo.get_sigmas(1.0, 0.01, 4, "logarithmic")
    shp = (2, 12, 8, 1)
    rng = np.random.default_rng(0)
    x1, x2, mixed = _states(3, shp, 1)
    for i in range(len(sig)):
        eta, lam, ns = bo.step_constants(sig, i)
        s1, s2, n1, n2 = (rng.standard_normal(shp).astype(np.float32) for _ in range(4))
        a1, a2 = bo.langevin_update(x1, x2, s1, s2, mixed, n1, n2, eta, lam, ns, g, grad_g)
        b1, b2 = bko.langevin_update_k([x1, x2], [s1, s2], mixed, [n1, n2], eta, lam, ns, g, grad_g)
        assert np.array_equal(a1, b1) and np.array_equal(a2, b2)
        x1, x2 = a1, a2
    # whole sigma x T loop with nonlinear scores and per-step states
    noise = {(i, t): [rng.standard_normal(shp).astype(np.float32) for _ in range(2)] for i in range(4) for t in range(3)}
    score1 = lambda x, i: np.tanh(x * np.float32(i + 1)).astype(np.float32)
    score2 = lambda x, i: (np.float32(0.5) - x).astype(np.float32)
    y1, y2 = _states(2, shp, 5)
    ps2, psk = [], []
    r1, r2, arr2 = bo.basis_run(mixed, y1, y2, score1, score2, sig, 3, lambda i, t: tuple(noise[(i, t)]), per_step=ps2)
    rk, arrk = bko.basis_run_k(mixed, [y1, y2], [score1, score2], sig, 3, lambda i, t: noise[(i, t)], per_step=psk)
    assert np.array_equal(r1, rk[0]) and np.array_equal(r2, rk[1])
    for key in ("x1", "x2"):
        assert len(arr2[key]) == len(arrk[key]) == len(sig) + 1
        assert all(np.array_equal(a, b) for a, b in zip(arr2[key], arrk[key]))
    assert all(np.array_equal(a[k], b[k]) for a, b in zip(ps2, psk) for k in range(2))


@pytest.mark.parametrize("K", [3, 5])
def test_k_source_mixing_properties(K):
    g, grad_g = bo.mixing_process("melspec", "dB")
    shp = (2, 6, 4, 1)
    x = _states(1, shp, K)[0]
    # equal sources: the power mean of identical sources is the source, each gets weight 1/K
    np.testing.assert_allclose(g(*([x] * K)), x, rtol=0, atol=2e-5)
    for w in grad_g(*([x] * K)):
        np.testing.assert_allclose(w, np.float32(1.0 / K), rtol=1e-6)
    xs = _states(K, shp, 10 + K)
    ws = grad_g(*xs)
    np.testing.assert_allclose(np.sum(np.stack(ws), 0, dtype=np.float64), 1.0, rtol=0, atol=1e-6)
    # grad g against central differences of g in float64
    x64 = [v.astype(np.float64) for v in xs]

    def g64(vs):
        a = np.stack(vs) * np.log(10.0) / 10.0
        m = a.max(0)
        return (10.0 / np.log(10.0)) * (m + np.log(np.exp(a - m).sum(0)) - np.log(K))

    np.testing.assert_allclose(g(*xs), g64(x64), rtol=0, atol=5e-5)
    h = 1e-6
    for k in range(K):
        up = [v.copy() for v in x64]
        dn = [v.copy() for v in x64]
        up[k] += h
        dn[k] -= h
        fd = (g64(up) - g64(dn)) / (2 * h)
        np.testing.assert_allclose(ws[k], fd, rtol=0, atol=1e-5)


def test_mixture_db_is_the_power_sum_of_any_number_of_sources():
    a, b, c, d = (synthetic.mel_patches_db(2, s) for s in range(4))
    p2 = np.power(10.0, a.astype(np.float64) / 10.0) + np.power(10.0, b.astype(np.float64) / 10.0)
    assert np.array_equal(synthetic.mixture_db(a, b), np.clip(10.0 * np.log10(p2), -100.0, 20.0).astype(np.float32))
    p4 = sum(np.power(10.0, v.astype(np.float64) / 10.0) for v in (a, b, c, d))
    np.testing.assert_allclose(synthetic.mixture_db(a, b, c, d), np.clip(10.0 * np.log10(p4), -100.0, 20.0), rtol=0, atol=1e-4)
    with pytest.raises(ValueError):
        synthetic.mixture_db(a)


def _args(argv):
    return run_basis_sep.build_parser().parse_args(argv)


def test_number_of_sources_comes_from_the_restore_directories():
    assert run_basis_sep.restore_dirs(_args(["a", "b"])) == ["a", "b"]
    assert run_basis_sep.source_names(_args(["a", "b"])) == ["piano", "violin"]
    args = _args(["a", "b", "c", "d", "--synthetic"])
    assert run_basis_sep.restore_dirs(args) == ["a", "b", "c", "d"]
    assert len(run_basis_sep.source_names(args)) == 4
    args = _args(["a", "b", "c", "--song_dir", "song", "--sources", "bass, drums,vocals"])
    assert run_basis_sep.source_names(args) == ["bass", "drums", "vocals"]


def test_sources_flag_is_required_and_checked():
    with pytest.raises(ValueError, match="--sources"):
        run_basis_sep.source_names(_args(["a", "b", "c", "--song_dir", "song"]))
    with pytest.raises(ValueError, match="--sources"):
        run_basis_sep.source_names(_args(["a", "b", "c", "--song_dir", "song", "--sources", "x,y"]))
    with pytest.raises(ValueError, match="--sources"):
        run_basis_sep.source_names(_args(["a", "b", "--song_dir", "song", "--sources", "x,y,z"]))
    with pytest.raises(ValueError, match="at most 8"):
        run_basis_sep.restore_dirs(_args([f"r{k}" for k in range(9)] + ["--synthetic"]))
    assert len(run_basis_sep.restore_dirs(_args([f"r{k}" for k in range(8)]))) == 8


def test_merge_config_keeps_the_k_source_fields(tmp_path):
    yml = tmp_path / "c.yml"
    yml.write_text("T: 7\nRESTORE: [x]\nsources: nope\n")
    args = _args(["a", "b", "c", "--config", str(yml), "--sources", "p,q,r"])
    merged = run_basis_sep.merge_config(args)
    assert merged.RESTORE == ["c"] and merged.sources == "p,q,r" and merged.T == 7
    assert isinstance(merged, argparse.Namespace)
