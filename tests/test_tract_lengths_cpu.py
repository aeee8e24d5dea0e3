"""hiddengem posterior tract-length spectrum: the oracle of E[R_s(X)], the expected number of maximal runs of state s at
least X long, checked against enumeration of every path (float64 on the tiny tables of test_posterior_cpu.py, 60-digit
mpmath on the edge tables of test_hiddengem_edges_cpu.py), its invariants, a long table that needs the window sums to
be formed from the window's own terms, and the command-line surface of --tract-lengths that needs no GPU.

For a table of n bins, J(i, X) is the first bin J >= i whose run [i, J] is X long (end[J] - start[i] + 1 with
coordinates, J - i + 1 in bins), and
    E[R_s(X)] = sum_i d_i(s) prod_{m=i+1}^{J} c_m(s) gamma_J(s),
    c_m(s) = alpha_{m-1}(s) pen(s, s) / sum_k alpha_{m-1}(k) pen(k, s),  d_i(s) = 1 - c_i(s) (the other two), d_0 = 1.
The product is exp of a sum of ln c_m (clamped at -750, and -750 where gamma_m(s) = 0) formed as the kernel forms it:
within one 32-bin stride from the terms, otherwise from the rest of i's stride, whole strides (or, across 1,024-bin
blocks, the block-suffix, whole blocks and block-prefix of stride totals) and the in-stride prefix of J's stride."""
import os
import subprocess

import numpy as np
import pytest

import hostlib
from test_posterior_cpu import PENALTIES, _lse3, _shift, brute_force, log_emissions, tiny_tables
from test_tract_counts_cpu import tract_counts_oracle

CLAMP = -750.0


def run_terms(lik, is_log, p01, p02, p12, dtype=np.float64):
    """(gamma [n, 3], d [n, 3], ln c [n, 3], dead) of one table by log-space forward-backward, in `dtype`."""
    le = log_emissions(np.asarray(lik, np.float64).reshape(-1, 3), is_log).astype(dtype)
    n = len(le)
    with np.errstate(divide="ignore"):
        lp = np.log(np.array([[1.0, p01, p02], [p01, 1.0, p12], [p02, p12, 1.0]], dtype))
    fa = np.zeros((n, 3), dtype)
    fb = np.zeros((n, 3), dtype)
    if n:
        fa[0] = le[0]
    with np.errstate(all="ignore"):
        for i in range(1, n):
            fa[i] = _shift(le[i] + _lse3(fa[i - 1][:, None] + lp, axis=0))
        for i in range(n - 2, -1, -1):
            fb[i] = _shift(_lse3(lp + (le[i + 1] + fb[i + 1])[None, :], axis=1))
        dead = n > 0 and np.isneginf(fa[n - 1]).all()
        hh = fa + fb
        g = np.exp(hh - _lse3(hh, axis=1)[:, None]) if n else np.zeros((0, 3), dtype)
        d = np.ones((n, 3), dtype)
        lc = np.zeros((n, 3), dtype)
        if n > 1:
            w = fa[:-1][:, :, None] + lp[None]  # [i - 1, k, l]
            D = _lse3(w, axis=1)  # [i - 1, l]
            r = np.where(np.isfinite(D)[:, None, :], np.exp(w - D[:, None, :]), 0.0)
            ok = g[1:] > 0
            diag = w[:, [0, 1, 2], [0, 1, 2]] - D
            lc[1:] = np.where(ok, np.maximum(np.where(np.isfinite(D), diag, -np.inf), CLAMP), CLAMP)
            d[1:] = np.where(ok, r.sum(axis=1) - r[:, [0, 1, 2], [0, 1, 2]], 0.0)
    return g, d, lc, dead


def window_sums(lc, i, J):
    """sum of lc[m] over m in (i, J], per state, from pieces inside the window (the kernel's decomposition); i, J
    arrays of equal length with i <= J."""
    n = len(lc)
    dt = lc.dtype
    z = np.zeros((len(i), 3), dt)
    if len(i) == 0:
        return z
    ns = (n + 31) // 32
    pad = np.zeros((ns * 32, 3), dt)
    pad[:n] = lc
    strides = pad.reshape(ns, 32, 3)
    pf = np.cumsum(strides, axis=1).reshape(-1, 3)[:n]  # in-stride inclusive prefix
    sx = np.flip(np.cumsum(np.flip(strides, 1), axis=1), 1)  # in-stride inclusive suffix
    sx = np.concatenate([sx[:, 1:], np.zeros((ns, 1, 3), dt)], axis=1).reshape(-1, 3)[:n]  # exclusive: m > i
    st = strides.sum(axis=1)
    nb = (ns + 31) // 32
    padb = np.zeros((nb * 32, 3), dt)
    padb[:ns] = st
    blocks = padb.reshape(nb, 32, 3)
    sp = np.cumsum(blocks, axis=1).reshape(-1, 3)[:ns]
    ss = np.flip(np.cumsum(np.flip(blocks, 1), axis=1), 1).reshape(-1, 3)[:ns]
    bt = blocks.sum(axis=1)
    si, sj = i >> 5, J >> 5
    w = np.zeros((len(i), 3), dt)
    same = si == sj
    for o in range(1, 32):  # within one stride: the terms themselves
        m = same & (i + o <= J)
        w[m] += lc[(i + o)[m]]
    far = ~same
    mid = np.zeros((len(i), 3), dt)
    qa, qb = si + 1, sj - 1
    inblock = far & (qa <= qb) & ((qa >> 5) == (qb >> 5))
    for o in range(0, 31):
        m = inblock & (qa + o <= qb)
        mid[m] += st[(qa + o)[m]]
    across = far & (qa <= qb) & ((qa >> 5) != (qb >> 5))
    mid[across] = ss[qa[across]]
    nbt = int(((qb >> 5) - (qa >> 5) - 1)[across].max()) if across.any() else 0
    for o in range(nbt):
        m = across & ((qa >> 5) + 1 + o < (qb >> 5))
        mid[m] += bt[((qa >> 5) + 1 + o)[m]]
    mid[across] += sp[qb[across]]
    w[far] = (sx[i[far]] + mid[far]) + pf[J[far]]
    return w


def first_reaching(n, thr, start=None, end=None):
    """J(i, X) for every start bin i (n where no J exists)."""
    i = np.arange(n)
    if start is None:
        return np.where(thr - 1 < n - i, i + (int(thr) - 1), n)
    target = np.asarray(start, np.float64) + (float(thr) - 1)
    return np.maximum(i, np.searchsorted(np.asarray(end, np.float64), target, side="left"))


def tract_lengths_oracle(lik, bin_offsets, thresholds, start=None, end=None, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3,
                         dtype=np.float64):
    """E[R_s(X)] per table, threshold and state, [T, K, 3] (float64); start / end per bin, packed like lik (None:
    lengths in bins)."""
    off = np.asarray(bin_offsets, np.int64)
    rows = np.asarray(lik, np.float64).reshape(-1, 3)
    out = np.zeros((len(off) - 1, len(thresholds), 3))
    for t in range(len(off) - 1):
        a, b = int(off[t]), int(off[t + 1])
        n = b - a
        if n == 0:
            continue
        g, d, lc, dead = run_terms(rows[a:b], is_log, p01, p02, p12, dtype)
        if dead:
            out[t] = np.nan
            continue
        for k, x in enumerate(thresholds):
            J = first_reaching(n, x, None if start is None else start[a:b], None if end is None else end[a:b])
            i = np.nonzero(J < n)[0]
            J = J[i]
            w = window_sums(lc, i, J)
            with np.errstate(under="ignore"):
                out[t, k] = (g[J] * d[i] * np.exp(w)).sum(axis=0).astype(np.float64)
    return out


def enumerate_runs(lik, is_log, p, thresholds, start=None, end=None):
    """E[R_s(X)] [K, 3] of one table from the weights of every one of its 3^n paths (NaN for total weight 0)."""
    _, w, paths = brute_force(lik, is_log, *p)
    z = w.sum()
    if not z > 0:
        return np.full((len(thresholds), 3), np.nan)
    return (w[:, None, None] * path_runs(paths, thresholds, start, end)).sum(axis=0) / z


def path_runs(paths, thresholds, start=None, end=None):
    """R_s(X) [P, K, 3] of every path (rows of `paths`), counted run by run."""
    paths = np.asarray(paths)
    P, n = paths.shape
    R = np.zeros((P, len(thresholds), 3))
    for p in range(P):
        i = 0
        while i < n:
            j = i
            while j + 1 < n and paths[p, j + 1] == paths[p, i]:
                j += 1
            length = (int(end[j]) - int(start[i]) + 1) if start is not None else j - i + 1
            for k, x in enumerate(thresholds):
                if length >= x:
                    R[p, k, paths[p, i]] += 1
            i = j + 1
    return R


def irregular_coords(rng, n):
    s = np.cumsum(rng.integers(0, 40, n)).astype(np.uint64) + 100
    e = s + rng.integers(0, 30, n).astype(np.uint64)
    return s, np.maximum.accumulate(e)


@pytest.mark.parametrize("coords", [False, True])
@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_oracle_equals_enumeration_of_every_path(coords, is_log, pen):
    rng = np.random.default_rng(11 + is_log + 2 * coords)
    tables = [l for l in tiny_tables(rng, is_log) if len(l) <= 7]
    off = np.concatenate([[0], np.cumsum([len(t) for t in tables])]).astype(np.int64)
    p = PENALTIES[pen]
    lik = np.concatenate(tables)
    start = end = None
    if coords:
        parts = [irregular_coords(rng, len(t)) for t in tables]
        start, end = np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])
    for t, l in enumerate(tables):
        a, b = off[t], off[t + 1]
        span = int(end[b - 1] - start[a] + 1) if coords else len(l)
        th = sorted({1, 2, max(1, span // 2), span, span + 1})
        got = tract_lengths_oracle(l, [0, len(l)], th, None if not coords else start[a:b], None if not coords else end[a:b],
                                   is_log, *p)
        want = enumerate_runs(l, is_log, p, th, None if not coords else start[a:b], None if not coords else end[a:b])
        np.testing.assert_allclose(got[0], want, rtol=0, atol=1e-12, equal_nan=True)
        assert np.isnan(want).any() or (got[0][-1] == 0).all()  # past the table's span


def test_oracle_edge_rules():
    l = np.array([[1e-3, 3e-3, 4e-3]])
    got = tract_lengths_oracle(l, [0, 0, 1, 1], [1, 2])
    assert (got[0] == 0).all() and (got[2] == 0).all()  # empty tables
    np.testing.assert_allclose(got[1, 0], l[0] / l[0].sum(), rtol=0, atol=1e-15)  # one bin: gamma_0 when it reaches X
    assert (got[1, 1] == 0).all()
    got = tract_lengths_oracle(l, [0, 1], [5, 6], np.array([10], np.uint64), np.array([14], np.uint64))
    np.testing.assert_allclose(got[0, 0], l[0] / l[0].sum(), rtol=0, atol=1e-15)  # the bin spans 5 bp
    assert (got[0, 1] == 0).all()
    dead = tract_lengths_oracle(np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]), [0, 2], [1, 5], is_log=False, p01=0.0, p02=0.0, p12=0.0)
    assert np.isnan(dead).all()  # total weight 0


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_invariants(is_log, pen):
    """Non-increasing in X; X = 1 bin is tract_counts_oracle's E[T_s] to 1e-12 relative."""
    rng = np.random.default_rng(60 + is_log)
    lens = [1, 2, 17, 60, 0, 33, 1500]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    lik = rng.normal(-30, 3, (off[-1], 3)) if is_log else np.exp(rng.normal(-10, 1.5, (off[-1], 3)))
    p = PENALTIES[pen]
    th = [1, 2, 3, 16, 33, 40, 1100]
    got = tract_lengths_oracle(lik, off, th, is_log=is_log, p01=p[0], p02=p[1], p12=p[2])
    _, _, tracts, _ = tract_counts_oracle(lik, off, is_log, *p)
    live = ~np.isnan(tracts).any(axis=1)
    np.testing.assert_allclose(got[live, 0], tracts[live], rtol=1e-12, atol=1e-300)
    assert (np.diff(got[live], axis=1) <= 1e-12 * np.maximum(1, got[live, :-1])).all()


def conditioning_table(n=100_000):
    """IBD2 very unlikely (about 40 nats per bin behind) for most of the table, then a long IBD2 run at the end."""
    rng = np.random.default_rng(8)
    ll = rng.normal(-100, 1, (n, 3))
    ll[:, 2] -= 40.0
    ll[: n - 3000, rng.integers(0, 2)] += 5.0
    ll[n - 3000:, 2] += 80.0
    return ll


def test_conditioning_table_keeps_its_digits():
    """Over the unlikely stretch ln c of IBD2 sums to millions of nats; the windows are formed from their own terms,
    so the float64 oracle matches its long double run."""
    ll = conditioning_table()
    th = [1, 100, 2000, 2999, 3000, 3001]
    a = tract_lengths_oracle(ll, [0, len(ll)], th, is_log=True)
    b = tract_lengths_oracle(ll, [0, len(ll)], th, is_log=True, dtype=np.longdouble)
    np.testing.assert_allclose(a, b, rtol=1e-10, atol=1e-300)
    assert abs(a[0, 4, 2] - 1) < 1e-6 and a[0, 5, 2] < 1e-6  # the planted 3000-bin run, counted once
    _, _, lc, _ = run_terms(ll, True, 1e-3, 1e-6, 1e-3)
    assert -lc[:, 2].sum() > 1e6  # where prefix sums over the table would have lost the digits


# ---- 60-digit enumeration on the edge tables -----------------------------------------------------------------------
def mp_runs(rows, is_log, pen, thresholds, dps=60):
    """E[R_s(X)] [K, 3] of one table by enumeration of every path in dps-digit arithmetic; NaN for total weight 0."""
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
            return np.full((len(thresholds), 3), np.nan)
        R = path_runs(np.array([x for x, _ in level]), thresholds)
        return np.array([[float(mp.fsum(w * int(r[k, s]) for (_, w), r in zip(level, R)) / z) for s in range(3)]
                         for k in range(len(thresholds))])


def _check_against_mp(tables, is_log, p):
    for rows in tables:
        n = len(rows)
        th = sorted({1, 2, max(1, n // 2), n, n + 1})
        got = tract_lengths_oracle(rows, [0, n], th, is_log=is_log, p01=p[0], p02=p[1], p12=p[2])[0]
        want = mp_runs(rows, is_log, p, th)
        assert np.isnan(got).all() == np.isnan(want).all()
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12, equal_nan=True)


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


# ---- command lines -------------------------------------------------------------------------------------------------
def test_tract_lengths_rejections(fixture_dir, tmp_path):
    hostlib.build()
    hg = os.path.join(hostlib.BIN, "hiddengem")
    msg = "[::] ERROR: --tract-lengths needs --posterior (the run lengths are those of the posterior paths).\n"
    r = subprocess.run([hg, "-s", "missing.summary.txt", "--tract-lengths", "100"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "" and r.stderr == msg
    inp = os.path.join(fixture_dir, "input")
    base = [os.path.join(hostlib.BIN, "ibdgem"), "-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"),
            "-I", os.path.join(inp, "test.indv"), "-P", os.path.join(inp, "test1.pileup"), "-O", str(tmp_path), "--hiddengem"]
    r = subprocess.run(base + ["--tract-lengths", "100"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stderr == msg
    bad = "[::] ERROR: --tract-lengths takes 1 to 16 positive integers (bp), strictly increasing, separated by commas.\n"
    for arg in ("0", "100,100", "200,100", "10,x", "abc", "", "10,", "-5", ",".join(str(10 * (k + 1)) for k in range(17))):
        r = subprocess.run([hg, "-s", "missing.summary.txt", "--posterior", "--tract-lengths", arg], capture_output=True, text=True)
        assert r.returncode == 0 and r.stdout == "" and r.stderr == bad, arg
        r = subprocess.run(base + ["--posterior", "--tract-lengths", arg], capture_output=True, text=True)
        assert r.returncode == 0 and r.stderr == bad, arg
    assert not list(tmp_path.iterdir())


def test_help_lists_tract_lengths():
    hostlib.build()
    for binary in ("hiddengem", "ibdgem"):
        r = subprocess.run([os.path.join(hostlib.BIN, binary), "--help"], capture_output=True, text=True)
        assert "--tract-lengths" in r.stderr and "at least" in r.stderr, binary
