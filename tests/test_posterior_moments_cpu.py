"""hiddengem posterior moments: the oracle of the posterior mean and covariance of the bins per IBD state, checked
against enumeration of every path (float64 on the tiny tables of test_posterior_cpu.py, 60-digit mpmath on the edge
tables of test_hiddengem_edges_cpu.py), its exact invariants, and the command-line surface of --share-sd that needs no
GPU.

For one table, N_s(x) = #{i : x_i = s} under the path weights W(x) of the posterior.  The recursion: conditioned on
x_i = k the rest of the path is Markov, P(x_{i+1} = l | x_i = k) = pen(k, l) nrm[i+1][l] beta[i+1][l] / t_k;
    h_i^t[k] = E[#{j > i : x_j = t} | x_i = k] = sum_l P(l | k) (delta_lt + h_{i+1}^t[l]),   h_{n-1} = 0 (0 where t_k = 0),
    H_i^t = sum_k gamma_i(k) h_i^t[k],
    Cov(N_s, N_t) = sum_i gamma_i(s) (delta_st - gamma_i(t)) + gamma_i(s) (h_i^t[s] - H_i^t) + gamma_i(t) (h_i^s[t] - H_i^s)."""
import os
import subprocess

import numpy as np
import pytest

import hostlib
from test_posterior_cpu import PENALTIES, _lse3, _shift, brute_force, log_emissions, posterior_oracle, tiny_tables


def moments_oracle(lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3, dtype=np.float64, with_h=False):
    """Log-space forward-backward as posterior_oracle, and the moment recursion above, vectorised across tables and
    looped over bins, in `dtype` (np.float64, or np.longdouble for an x87 reference).  NaN mean and covariance for a
    table of total weight 0.  Returns (expected [T, 3], cov [T, 3, 3]) and with with_h also (gamma [T, nmax, 3],
    h [T, nmax, 3 (k), 3 (t)])."""
    off = np.asarray(bin_offsets, np.int64)
    T = len(off) - 1
    lens = np.diff(off)
    nmax = int(lens.max()) if T else 0
    rows = np.asarray(lik, np.float64).reshape(-1, 3)[off[0]: off[-1]] if off[-1] > off[0] else np.zeros((0, 3))
    le = log_emissions(rows, is_log).astype(dtype)
    E = np.zeros((T, nmax, 3), dtype)
    idx = np.arange(nmax)[None, :] < lens[:, None]
    E[idx] = le
    with np.errstate(divide="ignore"):
        lp = np.log(np.array([[1.0, p01, p02], [p01, 1.0, p12], [p02, p12, 1.0]], dtype))
    fa = np.zeros((T, nmax, 3), dtype)
    fb = np.zeros((T, nmax, 3), dtype)
    if nmax:
        fa[:, 0] = E[:, 0]
    for i in range(1, nmax):
        fa[:, i] = _shift(E[:, i] + _lse3(fa[:, i - 1][:, :, None] + lp[None], axis=1))
    h = np.zeros((T, nmax, 3, 3), dtype)
    eye = np.eye(3, dtype=dtype)
    with np.errstate(all="ignore"):
        for i in range(nmax - 2, -1, -1):
            x = lp[None] + (E[:, i + 1] + fb[:, i + 1])[:, None, :]  # [T, k, l]
            t = _lse3(x, axis=2)  # [T, k]
            live = (i < lens - 1)[:, None]
            fb[:, i] = np.where(live, _shift(t), 0.0)
            P = np.where(np.isfinite(t)[:, :, None], np.exp(x - t[:, :, None]), 0.0)
            hn = np.einsum("zkl,zlt->zkt", P, eye[None] + h[:, i + 1])
            h[:, i] = np.where(live[:, :, None], hn, 0.0)
        last = fa[np.arange(T), np.maximum(lens - 1, 0)]
        dead = np.isneginf(last).all(axis=1)
        hh = fa + fb
        g = np.exp(hh - _lse3(hh, axis=2)[:, :, None])
    g = np.where(idx[:, :, None], g, 0.0)
    H = np.einsum("zik,zikt->zit", g, h)  # [T, i, t]
    D = np.einsum("zis,zist->zist", g, h - H[:, :, None, :])  # gamma_i(s) (h_i^t[s] - H_i^t), [T, i, s, t]
    cov = (np.einsum("zis,st->zst", g, eye) - np.einsum("zis,zit->zst", g, g) + D.sum(axis=1) + D.sum(axis=1).transpose(0, 2, 1))
    expected = g.sum(axis=1)
    expected[dead] = np.nan
    cov[dead] = np.nan
    if with_h:
        return expected, cov, g, h
    return expected, cov


def enumerate_moments(lik, is_log, p01, p02, p12):
    """E[N] and Cov(N) of one table from the weights of every one of its 3^n paths (NaN for total weight 0)."""
    _, w, paths = brute_force(lik, is_log, p01, p02, p12)
    z = w.sum()
    if not z > 0:
        return np.full(3, np.nan), np.full((3, 3), np.nan)
    N = np.stack([(paths == s).sum(axis=1) for s in range(3)], axis=1).astype(np.float64)
    mean = (w[:, None] * N).sum(axis=0) / z
    d = N - mean
    return mean, (w[:, None, None] * d[:, :, None] * d[:, None, :]).sum(axis=0) / z


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_oracle_equals_enumeration_of_every_path(is_log, pen):
    rng = np.random.default_rng(5 + is_log)
    tables = tiny_tables(rng, is_log)
    off = np.concatenate([[0], np.cumsum([len(t) for t in tables])])
    p = PENALTIES[pen]
    expected, cov = moments_oracle(np.concatenate(tables), off, is_log, *p)
    _, want_e = posterior_oracle(np.concatenate(tables), off, is_log, *p)
    np.testing.assert_allclose(expected, want_e, rtol=0, atol=1e-12, equal_nan=True)  # the posterior entry's mean
    for t, l in enumerate(tables):
        m, c = enumerate_moments(l, is_log, *p)
        np.testing.assert_allclose(expected[t], m, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(cov[t], c, rtol=0, atol=1e-12, equal_nan=True)
    assert np.isnan(cov[-1]).all() == (p[0] == 0)  # the forced table has weight p01


def test_oracle_edge_rules():
    l = np.array([[1e-3, 3e-3, 4e-3]])
    expected, cov = moments_oracle(l, [0, 0, 1, 1])
    for t in (0, 2):  # empty tables: mean 0, covariance 0
        np.testing.assert_array_equal(expected[t], 0.0)
        np.testing.assert_array_equal(cov[t], 0.0)
    g = l[0] / l[0].sum()  # one bin: diag(gamma) - gamma gamma^T
    np.testing.assert_allclose(cov[1], np.diag(g) - np.outer(g, g), rtol=0, atol=1e-15)
    expected, cov = moments_oracle(np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]), [0, 2], False, 0.0, 0.0, 0.0)
    assert np.isnan(expected).all() and np.isnan(cov).all()  # total weight 0


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_invariants(is_log, pen):
    """sum_t h_i^t[k] = n - 1 - i wherever state k can continue; H_i^t = sum_{j>i} gamma_j(t); rows of Cov sum to 0;
    Cov is positive semi-definite."""
    rng = np.random.default_rng(40 + is_log)
    lens = [1, 2, 17, 60, 0, 33]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    lik = rng.normal(-30, 3, (off[-1], 3)) if is_log else np.exp(rng.normal(-10, 1.5, (off[-1], 3)))
    p = PENALTIES[pen]
    expected, cov, g, h = moments_oracle(lik, off, is_log, *p, with_h=True)
    for t, n in enumerate(lens):
        if np.isnan(cov[t]).any():
            continue
        for i in range(n):
            reach = g[t, i] > 1e-300
            np.testing.assert_allclose(h[t, i].sum(axis=1)[reach], n - 1 - i, rtol=1e-12, atol=1e-12)
            H = np.einsum("k,kt->t", g[t, i], h[t, i])
            np.testing.assert_allclose(H, g[t, i + 1: n].sum(axis=0), rtol=0, atol=1e-10 * n)
        np.testing.assert_allclose(cov[t].sum(axis=1), 0.0, rtol=0, atol=1e-10 * max(n, 1))
        np.testing.assert_allclose(cov[t], cov[t].T, rtol=0, atol=1e-12 * max(n, 1))
        assert np.linalg.eigvalsh(cov[t]).min() >= -1e-10 * max(n, 1)


def test_longdouble_oracle_agrees_with_float64():
    rng = np.random.default_rng(12)
    lens = rng.integers(0, 300, 20)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    lik = rng.normal(-30, 3, (off[-1], 3))
    e1, c1 = moments_oracle(lik, off, True)
    e2, c2 = moments_oracle(lik, off, True, dtype=np.longdouble)
    np.testing.assert_allclose(e1, e2.astype(np.float64), rtol=0, atol=1e-11)
    np.testing.assert_allclose(c1, c2.astype(np.float64), rtol=0, atol=1e-9)


# ---- 60-digit enumeration on the edge tables -----------------------------------------------------------------------
def mp_moments(rows, is_log, pen, dps=60):
    """E[N] and Cov(N) of one table by enumeration of every path in dps-digit arithmetic (emissions as
    test_hiddengem_edges_cpu.mp_posterior defines them); NaN where the total weight is 0."""
    mp = pytest.importorskip("mpmath").mp
    rows = np.asarray(rows, np.float64)
    n = len(rows)
    with mp.workdps(dps):
        nrm = []
        for r in rows:
            if is_log:
                m = np.max(r) if not np.isnan(r).any() else np.nan
                bad = np.isnan(r).any() or not np.isfinite(m)
                nrm.append([mp.mpf(1)] * 3 if bad else [mp.mpf(0) if x == -np.inf else mp.exp(mp.mpf(x) - mp.mpf(m)) for x in r])
            else:
                with np.errstate(all="ignore"):
                    tot = (r[0] + r[1]) + r[2]
                bad = not (tot > 0) or not np.isfinite(tot)
                nrm.append([mp.mpf(1)] * 3 if bad else [mp.mpf(x) / mp.mpf(tot) for x in r])
        P = [[mp.mpf(1), mp.mpf(pen[0]), mp.mpf(pen[1])], [mp.mpf(pen[0]), mp.mpf(1), mp.mpf(pen[2])],
             [mp.mpf(pen[1]), mp.mpf(pen[2]), mp.mpf(1)]]
        level = [((s,), nrm[0][s]) for s in range(3) if nrm[0][s] != 0]
        for i in range(1, n):
            level = [(x + (s,), w * P[x[-1]][s] * nrm[i][s]) for x, w in level for s in range(3)]
            level = [(x, w) for x, w in level if w != 0]
        z = mp.fsum(w for _, w in level)
        if z == 0:
            return np.full(3, np.nan), np.full((3, 3), np.nan)
        cnt = [[x.count(s) for s in range(3)] for x, _ in level]
        mean = [mp.fsum(w * c[s] for (_, w), c in zip(level, cnt)) / z for s in range(3)]
        cov = [[float(mp.fsum(w * (c[s] - mean[s]) * (c[t] - mean[t]) for (_, w), c in zip(level, cnt)) / z) for t in range(3)]
               for s in range(3)]
        return np.array([float(m) for m in mean]), np.array(cov)


def _check_against_mp(tables, is_log, p):
    off = np.concatenate([[0], np.cumsum([len(r) for r in tables])]).astype(np.int64)
    expected, cov = moments_oracle(np.concatenate(tables), off, is_log, *p)
    for t, rows in enumerate(tables):
        want_e, want_c = mp_moments(rows, is_log, p)
        assert np.isnan(cov[t]).all() == np.isnan(want_c).all() and np.isnan(cov[t]).any() == np.isnan(want_c).any()
        np.testing.assert_allclose(expected[t], want_e, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(cov[t], want_c, rtol=0, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("pen", ["default", "p02_zero", "all_zero", "subnormal", "1.7e308", "all_1e-300", "all_1", "p02_1e+300"])
def test_oracle_equals_60_digit_enumeration(pen):
    from test_hiddengem_edges_cpu import ALL_PENALTIES, _cpu_tables
    p = ALL_PENALTIES[pen]
    for is_log in (False, True):
        _check_against_mp([rows for _, rows, lg in _cpu_tables() if lg == is_log], is_log, p)


@pytest.mark.parametrize("name", ["gap800_p02_zero", "gap700_p02_zero", "gap650_tiny_penalties", "meet_below_range",
                                  "huge_penalties", "gap800_default"])
def test_oracle_on_the_named_cases(name):
    from test_hiddengem_edges_cpu import LOG_CASES, to_text
    rows, p = LOG_CASES[name]
    _check_against_mp([np.array(rows, np.float64)], True, p)
    _check_against_mp([to_text(rows)], False, p)


@pytest.mark.parametrize("pen", ["default", "p02_zero", "all_zero", "subnormal", "1.7e308"])
def test_oracle_on_the_gap_sweep(pen):
    from test_hiddengem_edges_cpu import GAPS, PENALTY_SETS, gap_rows, to_text
    p = PENALTY_SETS[pen]
    _check_against_mp([gap_rows(g) for g in GAPS], True, p)
    _check_against_mp([to_text(gap_rows(g)) for g in GAPS], False, p)


def test_zero_weight_is_nan_only_where_real_weight_is_zero():
    rows = np.array([[0.0, -np.inf, -np.inf], [-np.inf, -np.inf, 0.0]])
    expected, cov = moments_oracle(rows, [0, 2], True, 1.0, 0.0, 1.0)
    assert np.isnan(expected).all() and np.isnan(cov).all()
    expected, cov = moments_oracle(rows, [0, 2], True, 1.0, 5e-324, 1.0)
    np.testing.assert_array_equal(expected[0], [1, 0, 1])
    np.testing.assert_array_equal(cov[0], 0.0)  # one path


# ---- command lines -------------------------------------------------------------------------------------------------
def test_share_sd_without_posterior_is_rejected(fixture_dir, tmp_path):
    hostlib.build()
    r = subprocess.run([os.path.join(hostlib.BIN, "hiddengem"), "-s", "missing.summary.txt", "--share-sd"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == ""
    assert r.stderr == "[::] ERROR: --share-sd needs --posterior (the standard deviations are those of the posterior counts).\n"
    inp = os.path.join(fixture_dir, "input")
    r = subprocess.run([os.path.join(hostlib.BIN, "ibdgem"), "-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"),
                        "-I", os.path.join(inp, "test.indv"), "-P", os.path.join(inp, "test1.pileup"), "-O", str(tmp_path),
                        "--hiddengem", "--share-sd"], capture_output=True, text=True)
    assert r.returncode == 0
    assert r.stderr == "[::] ERROR: --share-sd needs --posterior (the standard deviations are those of the posterior counts).\n"
    assert not list(tmp_path.iterdir())


def test_help_lists_share_sd():
    hostlib.build()
    for binary in ("hiddengem", "ibdgem"):
        r = subprocess.run([os.path.join(hostlib.BIN, binary), "--help"], capture_output=True, text=True)
        assert "--share-sd" in r.stderr and "kinship" in r.stderr, binary
