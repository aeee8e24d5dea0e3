"""hiddengem posterior tract counts: the oracle of the expected switches between IBD states, the expected number of
IBD tracts per state and the covariance of the tract counts, checked against enumeration of every path (float64 on
the tiny tables of test_posterior_cpu.py, 60-digit mpmath on the edge tables of test_hiddengem_edges_cpu.py), its
exact invariants, and the command-line surface of --tract-counts that needs no GPU.

For one table of n bins and a path x, S_kl = #{1 <= i < n : x_{i-1} = k, x_i = l} and T_s = [x_0 = s] +
#{1 <= i < n : x_i = s, x_{i-1} != s}, the number of maximal runs of state s.  With xi_i(k, l) = P(x_{i-1} = k, x_i = l)
= gamma_i(l) alpha_{i-1}(k) pen(k, l) / sum_k' alpha_{i-1}(k') pen(k', l), phi_i(s) = sum_{k != s} xi_i(k, s) (phi_0 =
gamma_0) and the posterior Markov chain P(x_{i+1} = l | x_i = k) = pen(k, l) nrm[i+1][l] beta[i+1][l] / t_k,
    g_i^t[k] = E[#{j > i : x_j = t, x_{j-1} != t} | x_i = k] = sum_l P(l | k) ([l = t][k != t] + g_{i+1}^t[l]),  g_{n-1} = 0,
    G_i^t = sum_k gamma_i(k) g_i^t[k],
    Cov(T_s, T_t) = sum_i phi_i(s) (delta_st - phi_i(t)) + phi_i(s) (g_i^t[s] - G_i^t) + phi_i(t) (g_i^s[t] - G_i^s)."""
import os
import subprocess

import numpy as np
import pytest

import hostlib
from test_posterior_cpu import PENALTIES, _lse3, _shift, brute_force, log_emissions, tiny_tables
from test_posterior_moments_cpu import moments_oracle


def tract_counts_oracle(lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3, dtype=np.float64, with_gamma=False):
    """Log-space forward-backward as posterior_oracle, the switch terms and the g-recursion above, vectorised across
    tables and looped over bins, in `dtype` (np.float64, or np.longdouble for an x87 reference).  NaN everywhere for
    a table of total weight 0.  Returns (expected [T, 3], switches [T, 3, 3], tracts [T, 3], tract_cov [T, 3, 3]) and
    with with_gamma also gamma [T, nmax, 3]."""
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
    eye = np.eye(3, dtype=dtype)
    M = ((np.arange(3)[None, :, None] == np.arange(3)[None, None, :]) &
         (np.arange(3)[:, None, None] != np.arange(3)[None, None, :])).astype(dtype)  # [k, l, t]: [l = t][k != t]
    gr = np.zeros((T, nmax, 3, 3), dtype)  # g_i^t[k] as [T, i, k, t]
    with np.errstate(all="ignore"):
        for i in range(nmax - 2, -1, -1):
            x = lp[None] + (E[:, i + 1] + fb[:, i + 1])[:, None, :]  # [T, k, l]
            t = _lse3(x, axis=2)  # [T, k]
            live = (i < lens - 1)[:, None]
            fb[:, i] = np.where(live, _shift(t), 0.0)
            P = np.where(np.isfinite(t)[:, :, None], np.exp(x - t[:, :, None]), 0.0)
            gn = np.einsum("zkl,klt->zkt", P, M) + np.einsum("zkl,zlt->zkt", P, gr[:, i + 1])
            gr[:, i] = np.where(live[:, :, None], gn, 0.0)
        last = fa[np.arange(T), np.maximum(lens - 1, 0)]
        dead = np.isneginf(last).all(axis=1)
        hh = fa + fb
        g = np.exp(hh - _lse3(hh, axis=2)[:, :, None])
        g = np.where(idx[:, :, None], g, 0.0)
        xi = np.zeros((T, nmax, 3, 3), dtype)  # xi_i(k, l) as [T, i, k, l]; 0 for i = 0
        for i in range(1, nmax):
            w = fa[:, i - 1][:, :, None] + lp[None]  # [T, k, l]
            D = _lse3(w, axis=1)  # [T, l]
            r = np.where(np.isfinite(D)[:, None, :], np.exp(w - D[:, None, :]), 0.0)
            xi[:, i] = np.where(g[:, i][:, None, :] > 0, g[:, i][:, None, :] * r, 0.0)
    xi = np.where(idx[:, :, None, None], xi, 0.0)
    phi = np.einsum("zikl,kl->zil", xi, 1 - eye)
    if nmax:
        phi[:, 0] = g[:, 0]
    G = np.einsum("zik,zikt->zit", g, gr)  # [T, i, t]
    D = np.einsum("zis,zist->zist", phi, gr - G[:, :, None, :])  # phi_i(s) (g_i^t[s] - G_i^t), [T, i, s, t]
    tract_cov = (np.einsum("zis,st->zst", phi, eye) - np.einsum("zis,zit->zst", phi, phi) + D.sum(axis=1)
                 + D.sum(axis=1).transpose(0, 2, 1))
    switches = xi.sum(axis=1)
    tracts = phi.sum(axis=1)
    expected = g.sum(axis=1)
    for a in (expected, switches, tracts, tract_cov):
        a[dead] = np.nan
    if with_gamma:
        return expected, switches, tracts, tract_cov, g
    return expected, switches, tracts, tract_cov


def path_counts(paths):
    """S [P, 3, 3] and T [P, 3] of every path (rows of `paths`)."""
    paths = np.asarray(paths)
    P, n = paths.shape
    S = np.zeros((P, 3, 3))
    for k in range(3):
        for l in range(3):
            S[:, k, l] = ((paths[:, :-1] == k) & (paths[:, 1:] == l)).sum(axis=1)
    first = np.stack([(paths[:, 0] == s) for s in range(3)], axis=1) if n else np.zeros((P, 3))
    T = first + S.sum(axis=1) - S[:, np.arange(3), np.arange(3)]
    return S, T


def enumerate_tract_counts(lik, is_log, p01, p02, p12):
    """E[S], E[T] and Cov(T) of one table from the weights of every one of its 3^n paths (NaN for total weight 0)."""
    _, w, paths = brute_force(lik, is_log, p01, p02, p12)
    z = w.sum()
    if not z > 0:
        return np.full((3, 3), np.nan), np.full(3, np.nan), np.full((3, 3), np.nan)
    S, T = path_counts(paths)
    ms = (w[:, None, None] * S).sum(axis=0) / z
    mt = (w[:, None] * T).sum(axis=0) / z
    d = T - mt
    return ms, mt, (w[:, None, None] * d[:, :, None] * d[:, None, :]).sum(axis=0) / z


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_oracle_equals_enumeration_of_every_path(is_log, pen):
    rng = np.random.default_rng(5 + is_log)
    tables = tiny_tables(rng, is_log)
    off = np.concatenate([[0], np.cumsum([len(t) for t in tables])])
    p = PENALTIES[pen]
    expected, switches, tracts, tcov = tract_counts_oracle(np.concatenate(tables), off, is_log, *p)
    want_e, _ = moments_oracle(np.concatenate(tables), off, is_log, *p)
    np.testing.assert_array_equal(expected, want_e)  # the same forward-backward
    for t, l in enumerate(tables):
        ms, mt, c = enumerate_tract_counts(l, is_log, *p)
        np.testing.assert_allclose(switches[t], ms, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(tracts[t], mt, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(tcov[t], c, rtol=0, atol=1e-12, equal_nan=True)
    assert np.isnan(tcov[-1]).all() == (p[0] == 0)  # the forced table has weight p01


def test_oracle_edge_rules():
    l = np.array([[1e-3, 3e-3, 4e-3]])
    expected, switches, tracts, tcov = tract_counts_oracle(l, [0, 0, 1, 1])
    for t in (0, 2):  # empty tables: everything 0
        for a in (expected, switches, tracts, tcov):
            np.testing.assert_array_equal(a[t], 0.0)
    g = l[0] / l[0].sum()  # one bin: no switches, one tract in the state of the bin
    np.testing.assert_array_equal(switches[1], 0.0)
    np.testing.assert_allclose(tracts[1], g, rtol=0, atol=1e-15)
    np.testing.assert_allclose(tcov[1], np.diag(g) - np.outer(g, g), rtol=0, atol=1e-15)
    out = tract_counts_oracle(np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]), [0, 2], False, 0.0, 0.0, 0.0)
    assert all(np.isnan(a).all() for a in out)  # total weight 0


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_invariants(is_log, pen):
    """sum S = n - 1; column sums of S = E[N] - gamma_0, row sums = E[N] - gamma_{n-1}; E[T_s] = gamma_0(s) + the
    switches into s from another state; Cov(T) symmetric and positive semi-definite."""
    rng = np.random.default_rng(40 + is_log)
    lens = [1, 2, 17, 60, 0, 33]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    lik = rng.normal(-30, 3, (off[-1], 3)) if is_log else np.exp(rng.normal(-10, 1.5, (off[-1], 3)))
    p = PENALTIES[pen]
    expected, switches, tracts, tcov, g = tract_counts_oracle(lik, off, is_log, *p, with_gamma=True)
    for t, n in enumerate(lens):
        if np.isnan(tcov[t]).any():
            continue
        tol = 1e-12 * max(n, 1)
        np.testing.assert_allclose(switches[t].sum(), max(n - 1, 0), rtol=0, atol=tol)
        if n == 0:
            continue
        np.testing.assert_allclose(switches[t].sum(axis=0), expected[t] - g[t, 0], rtol=0, atol=tol)
        np.testing.assert_allclose(switches[t].sum(axis=1), expected[t] - g[t, n - 1], rtol=0, atol=tol)
        into = switches[t].sum(axis=0) - np.diag(switches[t])
        np.testing.assert_allclose(tracts[t], g[t, 0] + into, rtol=0, atol=tol)
        np.testing.assert_allclose(tcov[t], tcov[t].T, rtol=0, atol=tol)
        assert np.linalg.eigvalsh(tcov[t]).min() >= -1e-10 * max(n, 1)


def test_clear_cut_table_keeps_its_digits():
    """A planted 10^4-bin table with strong evidence: E[T_s] is the planted count of runs and its sd near 0, where
    E[N_s] - sum_i xi_i(s, s) would have lost the digits."""
    rng = np.random.default_rng(3)
    runs = np.cumsum(rng.integers(1, 3, 40)) % 3  # neighbouring runs differ
    seg = np.repeat(runs, 250)
    ll = rng.normal(-150, 1, (len(seg), 3))
    ll[np.arange(len(seg)), seg] += 60.0
    expected, switches, tracts, tcov = tract_counts_oracle(ll, [0, len(seg)], True)
    want = np.bincount(runs, minlength=3)
    np.testing.assert_allclose(tracts[0], want, rtol=0, atol=1e-9)
    assert (np.sqrt(np.maximum(np.diag(tcov[0]), 0)) < 1e-4).all()
    S, _ = path_counts(seg[None])
    np.testing.assert_allclose(switches[0], S[0], rtol=0, atol=1e-9)


def test_longdouble_oracle_agrees_with_float64():
    rng = np.random.default_rng(12)
    lens = rng.integers(0, 300, 20)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    lik = rng.normal(-30, 3, (off[-1], 3))
    a = tract_counts_oracle(lik, off, True)
    b = tract_counts_oracle(lik, off, True, dtype=np.longdouble)
    for x, y in zip(a, b):
        np.testing.assert_allclose(x, y.astype(np.float64), rtol=0, atol=1e-9)


# ---- 60-digit enumeration on the edge tables -----------------------------------------------------------------------
def mp_tract_counts(rows, is_log, pen, dps=60):
    """E[S], E[T] and Cov(T) of one table by enumeration of every path in dps-digit arithmetic (emissions as
    test_hiddengem_edges_cpu.mp_posterior defines them); NaN where the total weight is 0."""
    mp = pytest.importorskip("mpmath").mp
    rows = np.asarray(rows, np.float64)
    n = len(rows)
    nan3, nan33 = np.full(3, np.nan), np.full((3, 3), np.nan)
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
            return nan33, nan3, nan33
        S, T = path_counts(np.array([x for x, _ in level]))
        ms = np.array([[float(mp.fsum(w * int(c[k, l]) for (_, w), c in zip(level, S)) / z) for l in range(3)] for k in range(3)])
        mt = [mp.fsum(w * int(c[s]) for (_, w), c in zip(level, T)) / z for s in range(3)]
        cov = [[float(mp.fsum(w * (int(c[s]) - mt[s]) * (int(c[t]) - mt[t]) for (_, w), c in zip(level, T)) / z) for t in range(3)]
               for s in range(3)]
        return ms, np.array([float(m) for m in mt]), np.array(cov)


def _check_against_mp(tables, is_log, p):
    off = np.concatenate([[0], np.cumsum([len(r) for r in tables])]).astype(np.int64)
    _, switches, tracts, tcov = tract_counts_oracle(np.concatenate(tables), off, is_log, *p)
    for t, rows in enumerate(tables):
        ms, mt, mc = mp_tract_counts(rows, is_log, p)
        assert np.isnan(tcov[t]).all() == np.isnan(mc).all() and np.isnan(tcov[t]).any() == np.isnan(mc).any()
        np.testing.assert_allclose(switches[t], ms, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(tracts[t], mt, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(tcov[t], mc, rtol=0, atol=1e-12, equal_nan=True)


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


# ---- command lines -------------------------------------------------------------------------------------------------
def test_tract_counts_without_posterior_is_rejected(fixture_dir, tmp_path):
    hostlib.build()
    msg = "[::] ERROR: --tract-counts needs --posterior (the tract counts are those of the posterior paths).\n"
    r = subprocess.run([os.path.join(hostlib.BIN, "hiddengem"), "-s", "missing.summary.txt", "--tract-counts"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "" and r.stderr == msg
    inp = os.path.join(fixture_dir, "input")
    r = subprocess.run([os.path.join(hostlib.BIN, "ibdgem"), "-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"),
                        "-I", os.path.join(inp, "test.indv"), "-P", os.path.join(inp, "test1.pileup"), "-O", str(tmp_path),
                        "--hiddengem", "--tract-counts"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stderr == msg
    assert not list(tmp_path.iterdir())


def test_help_lists_tract_counts():
    hostlib.build()
    for binary in ("hiddengem", "ibdgem"):
        r = subprocess.run([os.path.join(hostlib.BIN, binary), "--help"], capture_output=True, text=True)
        assert "--tract-counts" in r.stderr and "switches" in r.stderr, binary
