"""hiddengem IBD tracts, the parts that need no GPU: the numpy run-length oracle the GPU tests use, the record layout
of include/ibdgem_b200.h, and the command-line checks."""
import os
import re
import subprocess

import numpy as np
import pytest

import hostlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def tract_dtype():
    from ibdgem_b200.engine import TRACT_DTYPE
    return TRACT_DTYPE


def tract_oracle(states, lik, off, is_log, post=None, starts=None):
    """Run-length encoding of each table's states: (tract_offsets, records, scale), with records as
    hiddengem_tract and scale[k] = sum over tract k of |ln l| per state (the tolerance of the log-likelihood sums).
    starts[t] is where table t's bins sit in states / lik / post (default: off[t], the packed layout)."""
    off = np.asarray(off, np.int64)
    nt = len(off) - 1
    starts = off[:-1] if starts is None else np.asarray(starts, np.int64)
    toff = np.zeros(nt + 1, np.int64)
    recs, scales = [], []
    for t in range(nt):
        n = int(off[t + 1] - off[t])
        a = int(starts[t])
        if n == 0:
            toff[t + 1] = toff[t]
            continue
        x = np.asarray(states[a: a + n]).astype(np.int64)
        first = np.concatenate([[0], np.flatnonzero(x[1:] != x[:-1]) + 1])
        last = np.concatenate([first[1:], [n]])
        l = np.asarray(lik[a: a + n], np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            ll = l if is_log else np.log(l)
        r = np.zeros(len(first), tract_dtype())
        r["first_bin"], r["n_bins"], r["state"] = first, last - first, x[first]
        with np.errstate(invalid="ignore"):
            r["loglik"] = [ll[f:e].sum(axis=0) for f, e in zip(first, last)]
            sc = [np.abs(ll[f:e]).sum(axis=0) for f, e in zip(first, last)]
        if post is None:
            r["post_mean"] = r["post_min"] = np.nan
        else:
            p = np.asarray(post[a: a + n], np.float64)
            own = p[np.arange(n), x]
            r["post_mean"] = [own[f:e].mean() for f, e in zip(first, last)]
            r["post_min"] = [own[f:e].min() for f, e in zip(first, last)]  # NaN if any is
        recs.append(r)
        scales.append(np.array(sc))
        toff[t + 1] = toff[t] + len(first)
    recs = np.concatenate(recs) if recs else np.zeros(0, tract_dtype())
    scales = np.concatenate(scales) if scales else np.zeros((0, 3))
    return toff, recs, scales


def assert_tracts(got_off, got, want):
    """got against tract_oracle's (offsets, records, scale), field by field."""
    w_off, w, scale = want
    np.testing.assert_array_equal(got_off, w_off)
    assert len(got) == len(w)
    for f in ("first_bin", "n_bins", "state"):
        np.testing.assert_array_equal(got[f], w[f], err_msg=f)
    assert (got["reserved"] == 0).all()
    g, x = got["loglik"], w["loglik"]
    fin = np.isfinite(x)
    np.testing.assert_array_equal(g[~fin], x[~fin])
    assert (np.abs(g[fin] - x[fin]) <= 1e-12 * scale[fin]).all(), np.abs(g[fin] - x[fin]).max()
    np.testing.assert_array_equal(got["post_min"], w["post_min"])
    np.testing.assert_allclose(got["post_mean"], w["post_mean"], rtol=1e-13, atol=0, equal_nan=True)


def test_oracle_on_a_small_example():
    states = np.array([0, 0, 1, 1, 1, 2, 0, 0], np.uint8)
    lik = np.exp(np.arange(24, dtype=np.float64).reshape(8, 3) * -0.5)
    lik[4, 1] = 0.0
    post = np.full((8, 3), 0.25)
    post[3, 1] = 0.5
    post[4, 1] = 0.125
    toff, r, scale = tract_oracle(states, lik, [0, 0, 5, 8], False, post)
    np.testing.assert_array_equal(toff, [0, 0, 2, 4])
    np.testing.assert_array_equal(r["first_bin"], [0, 2, 0, 1])
    np.testing.assert_array_equal(r["n_bins"], [2, 3, 1, 2])
    np.testing.assert_array_equal(r["state"], [0, 1, 2, 0])
    np.testing.assert_allclose(r["loglik"][0], [-0.0 - 1.5, -0.5 - 2.0, -1.0 - 2.5])
    assert r["loglik"][1][1] == -np.inf  # a zero likelihood
    np.testing.assert_allclose(r["post_mean"], [0.25, (0.25 + 0.5 + 0.125) / 3, 0.25, 0.25])
    np.testing.assert_array_equal(r["post_min"], [0.25, 0.125, 0.25, 0.25])
    assert scale.shape == (4, 3)
    with np.errstate(divide="ignore"):
        _, r2, _ = tract_oracle(states, np.log(lik), [0, 5, 8], True)
    np.testing.assert_array_equal(r2["loglik"], np.concatenate([r["loglik"][:2], r["loglik"][2:]]))
    assert np.isnan(r2["post_mean"]).all() and np.isnan(r2["post_min"]).all()


def test_record_layout_matches_the_header():
    """hiddengem_tract is 64 bytes with the field offsets of include/ibdgem_b200.h; the ABI lists the new entries."""
    dt = tract_dtype()
    assert dt.itemsize == 64
    assert [dt.fields[f][1] for f in ("first_bin", "n_bins", "state", "reserved", "loglik", "post_mean", "post_min")] == \
        [0, 8, 16, 20, 24, 48, 56]
    hdr = open(os.path.join(ROOT, "include", "ibdgem_b200.h")).read()
    body = re.search(r"typedef struct \{(.*?)\} hiddengem_tract;", hdr, re.S).group(1)
    fields = re.findall(r"^\s*(int64_t|int32_t|double)\s+(\w+)(\[3\])?;", body, re.M)
    assert [(t, n) for t, n, _ in fields] == [("int64_t", "first_bin"), ("int64_t", "n_bins"), ("int32_t", "state"),
                                              ("int32_t", "reserved"), ("double", "loglik"), ("double", "post_mean"),
                                              ("double", "post_min")]
    from ibdgem_b200._lib import ABI_SYMBOLS
    for name in ("hiddengem_tracts_batch", "hiddengem_tracts_device", "hiddengem_last_tracts"):
        assert name in ABI_SYMBOLS and re.search(r"\bint %s\(" % name, hdr)


def test_ibdgem_tracts_without_hiddengem_is_rejected(fixture_dir, tmp_path):
    hostlib.build()
    inp = os.path.join(fixture_dir, "input")
    r = subprocess.run([os.path.join(hostlib.BIN, "ibdgem"), "-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"),
                        "-I", os.path.join(inp, "test.indv"), "-P", os.path.join(inp, "test1.pileup"), "-O", str(tmp_path),
                        "--tracts"], capture_output=True, text=True)
    assert r.returncode == 0  # option validation exits with status 0, as the reference's does
    assert r.stderr == "[::] ERROR: --tracts needs --hiddengem (the tracts are runs of the hiddengem states).\n"
    assert not list(tmp_path.iterdir())


def test_help_texts_name_the_option():
    hostlib.build()
    for binary in ("ibdgem", "hiddengem"):
        r = subprocess.run([os.path.join(hostlib.BIN, binary), "--help"], capture_output=True, text=True)
        assert r.returncode == 0 and "--tracts" in r.stderr and "LOD10" in r.stderr
