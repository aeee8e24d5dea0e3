"""hiddengem posterior: the log-space oracle (test_posterior_cpu.posterior_oracle) against exact enumeration of every
path in 60-digit arithmetic (mpmath), on the inputs the GPU edge tests (test_hiddengem_edges_gpu.py) judge with it:
rows whose states are 0 to 5,000 nats apart, -inf entries, NaN rows, text rows with subnormal and zero entries, and
penalties from 0 and the smallest subnormal up to 1.7e308.  The oracle must give NaN exactly where the total path
weight is 0 in real numbers."""
import itertools

import numpy as np
import pytest

from test_posterior_cpu import posterior_oracle

mp = pytest.importorskip("mpmath").mp

# Named tiny tables (natural-log rows, penalties (p01, p02, p12)).  With the penalties shown, the states that carry the
# weight are further apart than exp() of a double can reach, or the only paths between them are forbidden.
LOG_CASES = {
    "gap800_p02_zero": ([[0, -800, -900], [-900, -800, 0]], (1e-3, 0.0, 1e-3)),
    "gap700_p02_zero": ([[0, -700, -2000], [-2000, -699.7, 0]], (1e-3, 0.0, 1e-3)),
    "gap650_p02_zero": ([[0, -650, -2000], [-2000, -649.7, 0]], (1e-3, 0.0, 1e-3)),
    "gap650_tiny_penalties": ([[0, -650, -5000], [-5000, -650, 0]], (1e-100, 0.0, 1e-100)),
    "meet_below_range": ([[0, -710, -5000]] + [[-100, 0, -5000]] * 8, (0.0, 0.0, 0.0)),
    "huge_penalties": ([[0, -1, -2], [-2, -1, 0], [0, -1, -2]], (1e308, 1e308, 1e308)),
    "gap800_default": ([[0, -800, -900], [-900, -800, 0]], (1e-3, 1e-6, 1e-3)),
}

GAPS = (600, 690, 699, 700, 701, 745, 800, 5000)

PENALTY_SETS = {"default": (1e-3, 1e-6, 1e-3), "p02_zero": (1e-3, 0.0, 1e-3), "all_zero": (0.0, 0.0, 0.0),
                "p02_1e-300": (1e-3, 1e-300, 1e-3), "subnormal": (5e-324,) * 3, "1e300": (1e300,) * 3,
                "1.7e308": (1.7e308,) * 3}

PENALTY_VALUES = (0.0, 5e-324, 1e-300, 2.0 ** -400, 1e-6, 1.0, 1e300, 1.7e308)


def gap_rows(g):
    """IBD0 in bin 0, IBD2 in bin 1, IBD1 g nats behind in both: with p02 = 0 every path of weight comparable to
    exp(-g) passes through IBD1."""
    return np.array([[0.0, -g, -(g + 1300.0)], [-(g + 1300.0), -g + 0.3, 0.0]])


def to_text(rows):
    """Likelihoods with the same ratios where a double can hold them: each row scaled so its largest entry is e^700."""
    rows = np.asarray(rows, np.float64)
    with np.errstate(all="ignore"):
        m = np.max(np.where(np.isnan(rows), -np.inf, rows), axis=1, keepdims=True)
        m = np.where(np.isfinite(m), m, 0.0)
        return np.exp(rows - m + 700.0)


def _cpu_tables():
    """(name, rows, is_log) of 1-9 bins."""
    rng = np.random.default_rng(2)
    t = [(f"gap{g}", gap_rows(g), True) for g in (0, 1, 50, 650, 700, 745, 800, 5000)]
    t += [(name, np.array(rows, np.float64), True) for name, (rows, _) in LOG_CASES.items()]
    t += [("wide_random", rng.normal(0, 1500, (5, 3)), True),
          ("wide_random_long", rng.normal(0, 800, (7, 3)), True),
          ("neginf", np.array([[0, -np.inf, -3], [-np.inf, -np.inf, 0], [-1, -800, -np.inf], [-np.inf, 0, -np.inf]]), True),
          ("nan_row", np.array([[0, -1, -2], [np.nan, 0, 0], [-5, -1000, 0]]), True),
          ("all_neginf_row", np.array([[0, -760, -2], [-np.inf] * 3, [-900, 0, -1]]), True),
          ("one_bin", np.array([[-3, -800, -1]]), True),
          ("text_gaps", to_text(gap_rows(720)), False),
          ("text_subnormal", np.array([[1e-310, 5e-324, 0.0], [0.0, 1e-320, 1e-300], [1.0, 0.0, 0.0]]), False),
          ("text_subnormal_forced", np.array([[1e300, 5e-324, 0.0], [0.0, 5e-324, 1e300]]), False),
          ("text_zero_rows", np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [np.nan, 1.0, 1.0], [0.0, 1.0, 0.0], [np.inf, 0.0, 1.0]]), False),
          ("text_one_bin", np.array([[0.0, 3e-320, 1e-323]]), False)]
    return t


def mp_posterior(rows, is_log, pen, dps=60):
    """Every one of the 3^n paths of one table, in dps-digit arithmetic: (posterior [n, 3], expected [3]); NaN where
    the total weight Z is 0.  Emissions as the oracle defines them: text l_s / ((l0 + l1) + l2), log exp(L_s - max),
    and an undefined row uniform."""
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
        level = [((s,), nrm[0][s]) for s in range(3) if nrm[0][s] != 0]  # prefixes of positive weight
        for i in range(1, n):
            level = [(x + (s,), w * P[x[-1]][s] * nrm[i][s]) for x, w in level for s in range(3)]
            level = [(x, w) for x, w in level if w != 0]
        acc = [[mp.mpf(0)] * 3 for _ in range(n)]
        z = mp.mpf(0)
        for x, w in level:
            z += w
            for i, s in enumerate(x):
                acc[i][s] += w
        if z == 0:
            return np.full((n, 3), np.nan), np.full(3, np.nan)
        post = np.array([[float(acc[i][s] / z) for s in range(3)] for i in range(n)])
        expected = np.array([float(sum(acc[i][s] for i in range(n)) / z) for s in range(3)])
        return post, expected


def _penalty_sets():
    out = dict(PENALTY_SETS)
    for v in PENALTY_VALUES:
        out[f"all_{v:g}"] = (v, v, v)
        out[f"p02_{v:g}"] = (1e-3, v, 1e-3)
    return out


ALL_PENALTIES = _penalty_sets()


@pytest.mark.parametrize("pen", list(ALL_PENALTIES))
def test_oracle_equals_60_digit_enumeration(pen):
    p = ALL_PENALTIES[pen]
    tables = _cpu_tables()
    for is_log in (False, True):
        group = [(name, rows) for name, rows, lg in tables if lg == is_log]
        off = np.concatenate([[0], np.cumsum([len(r) for _, r in group])]).astype(np.int64)
        post, expected = posterior_oracle(np.concatenate([r for _, r in group]), off, is_log, *p)
        for t, (name, rows) in enumerate(group):
            want_p, want_e = mp_posterior(rows, is_log, p)
            got = post[off[t]: off[t + 1]]
            assert np.isnan(got).all() == np.isnan(want_p).all() and np.isnan(got).any() == np.isnan(want_p).any(), name
            np.testing.assert_allclose(got, want_p, rtol=0, atol=1e-12, equal_nan=True, err_msg=name)
            np.testing.assert_allclose(expected[t], want_e, rtol=0, atol=1e-12, equal_nan=True, err_msg=name)


@pytest.mark.parametrize("name", list(LOG_CASES))
def test_oracle_on_the_named_cases(name):
    """The named cases with their own penalties; the values the GPU tests expect of them."""
    rows, p = LOG_CASES[name]
    for is_log, lik in ((True, np.array(rows, np.float64)), (False, to_text(rows))):
        post, expected = posterior_oracle(lik, [0, len(lik)], is_log, *p)
        want_p, want_e = mp_posterior(lik, is_log, p)
        np.testing.assert_allclose(post, want_p, rtol=0, atol=1e-12, equal_nan=True)
        np.testing.assert_allclose(expected[0], want_e, rtol=0, atol=1e-12, equal_nan=True)
    post, _ = posterior_oracle(np.array(rows, np.float64), [0, len(rows)], True, *p)
    if name == "gap800_p02_zero":
        np.testing.assert_allclose(post[0], [0.5, 0.5, 0.0], rtol=0, atol=1e-12)
    if name == "gap700_p02_zero":
        np.testing.assert_allclose(post[0, :2], [0.574, 0.426], rtol=0, atol=1e-3)
    if name == "meet_below_range":
        np.testing.assert_allclose(post[0], [np.exp(-90.0), 1.0, 0.0], rtol=1e-9, atol=0)
    assert np.isfinite(post).all()


@pytest.mark.parametrize("pen", list(PENALTY_SETS))
def test_oracle_on_the_gap_sweep(pen):
    p = PENALTY_SETS[pen]
    tables = [gap_rows(g) for g in GAPS]
    off = np.concatenate([[0], np.cumsum([len(r) for r in tables])]).astype(np.int64)
    for is_log, conv in ((True, lambda r: r), (False, to_text)):
        lik = np.concatenate([conv(r) for r in tables])
        post, expected = posterior_oracle(lik, off, is_log, *p)
        for t, r in enumerate(tables):
            want_p, want_e = mp_posterior(conv(r), is_log, p)
            np.testing.assert_allclose(post[off[t]: off[t + 1]], want_p, rtol=0, atol=1e-12, equal_nan=True)
            np.testing.assert_allclose(expected[t], want_e, rtol=0, atol=1e-12, equal_nan=True)


def test_zero_weight_is_nan_only_where_real_weight_is_zero():
    # IBD0 then IBD2 with p02 = 0: weight 0; with p02 = 5e-324 the same table has a definite answer
    rows = np.array([[0.0, -np.inf, -np.inf], [-np.inf, -np.inf, 0.0]])
    post, expected = posterior_oracle(rows, [0, 2], True, 1.0, 0.0, 1.0)
    assert np.isnan(post).all() and np.isnan(expected).all()
    post, expected = posterior_oracle(rows, [0, 2], True, 1.0, 5e-324, 1.0)
    np.testing.assert_array_equal(post, [[1, 0, 0], [0, 0, 1]])
    # all-zero penalties: a path must stay in one state; no state has weight in both bins
    post, _ = posterior_oracle(np.array([[0.0, -np.inf, -5.0], [-np.inf, 0.0, -np.inf]]), [0, 2], True, 0.0, 0.0, 0.0)
    assert np.isnan(post).all()
    # a weight below every double (exp(-1e4) * 5e-324^2) is still not 0
    post, _ = posterior_oracle(np.array([[0.0, -1e4, -np.inf], [-np.inf, -1e4, 0.0]]), [0, 2], True, 5e-324, 0.0, 5e-324)
    want, _ = mp_posterior(np.array([[0.0, -1e4, -np.inf], [-np.inf, -1e4, 0.0]]), True, (5e-324, 0.0, 5e-324))
    assert np.isfinite(post).all()
    np.testing.assert_allclose(post, want, rtol=0, atol=1e-12)


def test_mp_reference_agrees_with_float_enumeration_on_ordinary_tables():
    """The 60-digit enumeration is the same model as brute_force of test_posterior_cpu.py where doubles suffice."""
    from test_posterior_cpu import brute_force
    rng = np.random.default_rng(9)
    for n in range(1, 7):
        l = np.exp(rng.normal(-10, 2, (n, 3)))
        for p in ((1e-3, 1e-6, 1e-3), (0.2, 0.0, 2.5)):
            want, _, _ = brute_force(l, False, *p)
            got, _ = mp_posterior(l, False, p)
            np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)
