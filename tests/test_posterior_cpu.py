"""hiddengem posterior: the float64 log-space oracle of the per-bin posterior state probabilities, checked against
brute-force enumeration of every path on tiny tables, and the command-line surface of --posterior that needs no GPU.

The model is the path weight hiddengem maximises (src/hiddengem.c:108-147):
    W(x) = prod_i nrm[i][x_i] * prod_{i>0} pen(x_{i-1}, x_i),   posterior[i][s] = sum_{x: x_i = s} W(x) / sum_x W(x)
with pen = 1 on the diagonal, p01 / p02 / p12 off it, and no prior on bin 0.  A bin whose normalised row is undefined
gets the uniform emission; a table of total weight 0 has NaN posteriors."""
import itertools
import os
import subprocess

import numpy as np
import pytest

import hostlib

PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "zero_and_above_one": (0.0, 1e-3, 2.5), "above_one": (1.5, 3.0, 1.2),
             "loose": (0.2, 0.05, 0.3), "one": (1.0, 1.0, 1.0)}


def log_emissions(lik, is_log):
    """ln nrm per bin, [n, 3]; undefined rows (text: total not a positive finite number; log: a NaN score or a row
    maximum that is not finite) are uniform (ln 1 = 0)."""
    lik = np.asarray(lik, np.float64).reshape(-1, 3)
    with np.errstate(all="ignore"):
        if is_log:
            m = lik.max(axis=1, keepdims=True)
            bad = np.isnan(lik).any(axis=1) | ~np.isfinite(m[:, 0])
            out = lik - m - np.log(np.exp(lik - m).sum(axis=1, keepdims=True))
        else:
            tot = (lik[:, 0] + lik[:, 1]) + lik[:, 2]
            bad = ~(tot > 0) | ~np.isfinite(tot)
            out = np.log(lik) - np.log(tot)[:, None]  # not log(lik / tot): that quotient can underflow to 0
    out[bad] = 0.0
    return out


def _lse3(x, axis):
    with np.errstate(all="ignore"):
        m = x.max(axis=axis, keepdims=True)
        ms = np.where(np.isfinite(m), m, 0.0)
        return (ms + np.log(np.exp(x - ms).sum(axis=axis, keepdims=True))).squeeze(axis)


def _shift(x):
    """Rows of log weights shifted so their maximum is 0 (a row of -inf stays -inf): magnitudes, and with them the
    rounding of the sums, stay those of one row's spread however long the table."""
    m = x.max(axis=-1, keepdims=True)
    return x - np.where(np.isfinite(m), m, 0.0)


def posterior_oracle(lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3):
    """Log-space forward-backward (np.logaddexp-style log-sum-exp), vectorised across tables, looped over bins; each
    row of log alpha / log beta shifted to maximum 0, each bin's posterior normalised on its own.  NaN for a table
    whose final alpha is all -inf (total weight 0).  Returns (posterior [n_bins, 3], expected [n_tables, 3])."""
    off = np.asarray(bin_offsets, np.int64)
    T = len(off) - 1
    lens = np.diff(off)
    nmax = int(lens.max()) if T else 0
    le = log_emissions(np.asarray(lik, np.float64).reshape(-1, 3)[off[0]: off[-1]], is_log) if off[-1] > off[0] else np.zeros((0, 3))
    E = np.zeros((T, nmax, 3))
    idx = np.arange(nmax)[None, :] < lens[:, None]
    E[idx] = le
    with np.errstate(divide="ignore"):
        lp = np.log(np.array([[1.0, p01, p02], [p01, 1.0, p12], [p02, p12, 1.0]]))
    fa = np.zeros((T, nmax, 3))
    fb = np.zeros((T, nmax, 3))
    if nmax:
        fa[:, 0] = E[:, 0]
    for i in range(1, nmax):
        fa[:, i] = _shift(E[:, i] + _lse3(fa[:, i - 1][:, :, None] + lp[None], axis=1))
    for i in range(nmax - 2, -1, -1):
        nxt = _shift(_lse3(lp[None] + (E[:, i + 1] + fb[:, i + 1])[:, None, :], axis=2))
        fb[:, i] = np.where((i < lens - 1)[:, None], nxt, 0.0)
    last = fa[np.arange(T), np.maximum(lens - 1, 0)]
    dead = np.isneginf(last).all(axis=1)
    h = fa + fb
    with np.errstate(all="ignore"):
        g = np.exp(h - _lse3(h, axis=2)[:, :, None])
    g[dead] = np.nan
    post = g[idx]
    expected = np.where(idx[:, :, None], g, 0.0).sum(axis=1)
    return post, expected


def brute_force(lik, is_log, p01, p02, p12):
    """Every one of the 3^n paths of one table: (posterior [n, 3], path weights W [3^n], paths [3^n, n])."""
    nrm = np.exp(log_emissions(lik, is_log))
    n = len(nrm)
    pen = np.array([[1.0, p01, p02], [p01, 1.0, p12], [p02, p12, 1.0]])
    paths = np.array(list(itertools.product(range(3), repeat=n)), np.int64)
    w = nrm[np.arange(n)[None, :], paths].prod(axis=1)
    if n > 1:
        w = w * pen[paths[:, :-1], paths[:, 1:]].prod(axis=1)
    z = w.sum()
    post = np.full((n, 3), np.nan)
    if z > 0:
        for s in range(3):
            post[:, s] = ((paths == s) * w[:, None]).sum(axis=0) / z
    return post, w, paths


def tiny_tables(rng, is_log):
    """Tables of 1-8 bins: random rows, and rows with zeros or NaN."""
    tables = []
    for k in range(24):
        n = 1 + k % 8
        if is_log:
            l = rng.normal(-30, 4, (n, 3))
            if k % 3 == 1:
                l[rng.integers(0, n)] = np.nan
            if k % 5 == 2:
                l[rng.integers(0, n)] = -np.inf
            if k % 7 == 3:
                l[rng.integers(0, n), 1] = -np.inf
        else:
            l = np.exp(rng.normal(-10, 2, (n, 3)))
            if k % 3 == 1:
                l[rng.integers(0, n)] = 0.0
            if k % 5 == 2:
                l[rng.integers(0, n)] = np.nan
            if k % 4 == 3:
                l[rng.integers(0, n), rng.integers(0, 3)] = 0.0
        tables.append(l)
    # a zero penalty can leave no path of positive weight: IBD0, then IBD1, weighted p01
    forced = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])
    with np.errstate(divide="ignore"):
        tables.append(np.log(forced) if is_log else forced)
    return tables


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_oracle_equals_enumeration_of_every_path(is_log, pen):
    rng = np.random.default_rng(5 + is_log)
    tables = tiny_tables(rng, is_log)
    off = np.concatenate([[0], np.cumsum([len(t) for t in tables])])
    with np.errstate(divide="ignore"):
        post, expected = posterior_oracle(np.concatenate(tables), off, is_log, *PENALTIES[pen])
    for t, l in enumerate(tables):
        want, _, _ = brute_force(l, is_log, *PENALTIES[pen])
        got = post[off[t]: off[t + 1]]
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(expected[t], want.sum(axis=0), rtol=0, atol=1e-12, equal_nan=True)
    assert np.isnan(post[off[-2]:]).all() == (PENALTIES[pen][0] == 0)  # the forced table has weight p01


def test_oracle_edge_rules():
    # an empty table: no bins, expected occupancy 0; one bin: the normalised row
    l = np.array([[1e-3, 3e-3, 4e-3]])
    post, expected = posterior_oracle(l, [0, 0, 1, 1])
    np.testing.assert_array_equal(expected[0], 0.0)
    np.testing.assert_array_equal(expected[2], 0.0)
    np.testing.assert_allclose(post[0], l[0] / l[0].sum(), rtol=1e-14)
    # an uninformative bin is the uniform emission
    a, _ = posterior_oracle(np.array([[1e-3, 2e-3, 1e-4], [0.0, 0.0, 0.0], [5e-4, 1e-4, 1e-3]]), [0, 3])
    b, _ = posterior_oracle(np.array([[1e-3, 2e-3, 1e-4], [1.0, 1.0, 1.0], [5e-4, 1e-4, 1e-3]]), [0, 3])
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-15)
    # zero total weight: NaN posteriors and counts
    post, expected = posterior_oracle(np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]), [0, 2], False, 0.0, 0.0, 0.0)
    assert np.isnan(post).all() and np.isnan(expected).all()


@pytest.mark.parametrize("pen", list(PENALTIES))
def test_mode_of_the_path_weights_is_the_hiddengem_path(pen):
    """The posterior is over the weights hiddengem maximises: wherever the heaviest path is unique, it is the path the
    reference's recurrence (C oracle) infers."""
    import oracle
    rng = np.random.default_rng(11)
    p = PENALTIES[pen]
    checked = 0
    for k in range(40):
        n = 1 + k % 8
        l = np.exp(rng.normal(-10, 1.5, (n, 3)))
        _, w, paths = brute_force(l, False, *p)
        order = np.sort(w)
        if len(order) > 1 and not order[-1] > order[-2] * (1 + 1e-9):
            continue  # no unique maximum
        st, _, _ = oracle.hiddengem(l, *p)
        np.testing.assert_array_equal(st, paths[int(np.argmax(w))])
        checked += 1
    assert checked >= 30


def test_hiddengem_help_lists_posterior():
    hostlib.build()
    r = subprocess.run([os.path.join(hostlib.BIN, "hiddengem"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--posterior" in r.stderr
    assert "P_IBD0, P_IBD1, P_IBD2" in r.stderr


def test_ibdgem_posterior_without_hiddengem_is_rejected(fixture_dir, tmp_path):
    hostlib.build()
    inp = os.path.join(fixture_dir, "input")
    r = subprocess.run([os.path.join(hostlib.BIN, "ibdgem"), "-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"),
                        "-I", os.path.join(inp, "test.indv"), "-P", os.path.join(inp, "test1.pileup"), "-O", str(tmp_path),
                        "--posterior"], capture_output=True, text=True)
    assert r.returncode == 0  # the front-end's option validation exits with status 0, as the reference's does
    assert r.stderr == "[::] ERROR: --posterior needs --hiddengem (the posteriors are written to the hiddengem files).\n"
    assert not list(tmp_path.iterdir())
    r = subprocess.run([os.path.join(hostlib.BIN, "ibdgem"), "--help"], capture_output=True, text=True)
    assert "--posterior" in r.stderr and "--hiddengem" in r.stderr
