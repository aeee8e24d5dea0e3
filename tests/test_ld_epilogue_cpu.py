"""The term calculator of ldterms.py against the long double oracle, and the case builder's planted structure.  Tests
of the tensor-path epilogues rely on both to state their preconditions: which tile a row's maximum sits in, how far it
climbs, and where LIBD0's own entry stands in the mass."""
import numpy as np
import pytest

import ldterms as lt
import refcases

CASES = {
    # duplicates, the pileup's own individual, a target inside the background and one outside it, twins
    "duplicates_pu_twins": dict(seed=1, S=900, N=30, window=60, targets=[3, 5, 9, 29], src=4, share=[3],
                                twins={9: 11}, bg=[1, 3, 3, 5, 9, 11, 12, 20, 4, 2, 2, 7], pu_idx=2),
    "variable_sites": dict(seed=2, S=900, N=24, window=40, targets=[0, 6, 23], src=6, share=[0], twins={23: 6},
                           bg=list(range(24)) + [6, 6], pu_idx=-1, opt_v=1),
    "target_is_source": dict(seed=3, S=700, N=20, window=50, targets=[4, 8], src=4, twins={8: 4}, bg=[4, 4, 8, 1, 2]),
}


@pytest.mark.parametrize("eps", [0.001, 0.02, 0.3, 0.45])
@pytest.mark.parametrize("name", list(CASES))
def test_column_terms_reproduce_the_oracle(name, eps):
    kw = dict(CASES[name])
    case = lt.ld_case(kw.pop("seed"), kw.pop("S"), kw.pop("N"), kw.pop("window"), kw.pop("targets"), eps=eps,
                      depth=3.0, **kw)
    for t, ora in zip(case.targets, refcases.oracle_run(case)):
        wins = lt.windows(case, t)
        assert len(wins) == ora["n_windows"] > 0
        np.testing.assert_array_equal([len(w) for w in wins], ora["w_nsites"])
        for w, sites in enumerate(wins):
            got = np.array(lt.column_terms(case, sites, t).libd())
            want = ora["w_log"][w, :2]
            np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
            ok = ~np.isnan(want)
            assert np.all(np.abs(got[ok] - want[ok]) <= 1e-9), (t, w, got, want)


def test_empty_background_gives_nan_terms():
    case = lt.ld_case(4, 300, 6, 50, [2], bg=[2, 2])
    ora = refcases.oracle_run(case)[0]
    for w, sites in enumerate(lt.windows(case, 2)):
        got = lt.column_terms(case, sites, 2).libd()
        assert np.isnan(got).all() and np.isnan(ora["w_log"][w, :2]).all()


def test_case_builder_plants_shared_haplotypes_and_twins():
    case = lt.ld_case(5, 2000, 50, 100, [10, 20], src=33, share=[10, 20], twins={40: 10, 41: 33})
    hap = case.pk.hap
    for t in (10, 20):
        np.testing.assert_array_equal(hap[:, 2 * t], hap[:, 2 * 33 + 1])
        assert (hap[:, 2 * t + 1] != hap[:, 2 * 33]).any()  # only one haplotype is shared
    np.testing.assert_array_equal(hap[:, 80:82], hap[:, 20:22])
    np.testing.assert_array_equal(hap[:, 82:84], hap[:, 66:68])
    # the reads follow the source's genotype: the alternate-base fraction separates its three genotypes
    g = hap[:, 66].astype(int) + hap[:, 67]
    d = case.pk.n_ref.astype(int) + case.pk.n_alt
    frac = [case.pk.n_alt[(g == k) & (d > 0)].sum() / d[(g == k) & (d > 0)].sum() for k in range(3)]
    assert frac[0] < 0.05 and 0.4 < frac[1] < 0.6 and frac[2] > 0.95
    # a shared haplotype makes the source's other haplotype the best column of the target's row 0 in every window
    for sites in lt.windows(case, 10):
        x = lt.column_terms(case, sites, 10).col_terms()
        assert int(np.argmax(x[0])) == 2 * 33
        # twins give the same LIBD0 term, bit for bit
        q = lt.column_terms(case, sites, 10).q
        assert q[40] == q[10] and q[41] == q[33]


def test_first_tile_climb_measures_the_late_maximum():
    case = lt.ld_case(6, 1200, 300, 1000, [5], src=200, share=[5], depth=6.0)
    sites = lt.windows(case, 5)[0]
    terms = lt.column_terms(case, sites, 5)
    climb = lt.first_tile_climb(terms, 256)
    x = terms.col_terms()
    assert climb[0] == x[0].max() - x[0, :256].max() and climb[0] > 600
    assert lt.first_tile_climb(terms, 2 * 300)[0] == 0.0


@pytest.mark.parametrize("opt_v", [0, 1])
def test_thinned_view_reproduces_the_oracle_under_downsampling(opt_v):
    """-D: each target's thinned counts, drawn in the reference's rand() order, give the oracle's windows site for site
    and its LIBD0 / LIBD1."""
    case = lt.ld_case(7, 900, 24, 40, [0, 5, 23], src=5, share=[0], depth=6.0, cull_p=0.5, opt_v=opt_v)
    for k, ora in enumerate(refcases.oracle_run(case)):
        view = lt.thinned(case, k)
        t = view.targets[0]
        wins = lt.windows(view, t)
        np.testing.assert_array_equal([len(w) for w in wins], ora["w_nsites"])
        np.testing.assert_array_equal([case.pk.pos[w[0]] for w in wins], ora["w_start"])
        np.testing.assert_array_equal([case.pk.pos[w[-1]] for w in wins[:-1]], ora["w_end"][:-1])
        for w, sites in enumerate(wins):
            got = np.array(lt.column_terms(view, sites, t).libd())
            assert np.all(np.abs(got - ora["w_log"][w, :2]) <= 1e-9), (k, w, got, ora["w_log"][w, :2])


@pytest.mark.parametrize("eps,nats", [(0.001, 596), (0.02, 598), (0.1, 262), (0.3, 45)])
def test_mma_mode_table_at_the_usual_error_rates(eps, nats):
    """Table mode, with the head-room dpos |kappa| a row's maximum may climb before its reference key moves."""
    table, delta, dpos = lt.mma_mode(eps, 600)
    assert table and delta + dpos + 1 <= 512
    assert round(dpos * -lt.kappa(eps)) == nats


def test_mma_mode_switches_to_the_exp_path():
    """At 600 columns the table holds the screen's reach up to eps = 0.353; from 0.354 on the exp path runs, and at
    0.45 the reach is thousands of keys."""
    assert lt.mma_mode(0.353, 600) == (True, 252, 256)
    assert lt.mma_mode(0.354, 600) == (False, 256, 256)
    assert not lt.mma_mode(0.45, 600)[0] and lt.mma_mode(0.45, 600)[1] > 2000
    # the screen's reach grows with ln(ncols) up to 32 nats
    assert lt.mma_mode(0.02, 2)[1] == 9 and lt.mma_mode(0.02, 40962)[1] == 13


@pytest.mark.parametrize("opt_v", [0, 1])
def test_screen_operands_complete_the_column_terms(opt_v):
    """C0 + R[a_i] + (Y + kappa M) is the LIBD1 term of every row and column, with alpha, beta, kappa read off the
    oracle's P(D|G); frequencies given to the builder reach the panel."""
    case = lt.ld_case(8, 1500, 30, 200, [4], src=17, share=[4], depth=9.0, max_cov=40, eps=0.01, opt_v=opt_v, af=0.9)
    assert abs(case.pk.hap.mean() - 0.9) < 0.01
    alpha, beta, kap = lt.depth_coefficients(0.01, 40)
    assert np.isclose(alpha, np.log(0.5 / 0.99)) and np.isclose(beta, np.log(50)) and np.isclose(kap, lt.kappa(0.01))
    L = lt.ln_pdg(0.01, 40)
    pk = case.pk
    for sites in lt.windows(case, 4):
        C0 = L[pk.n_ref[sites], pk.n_alt[sites], 0].sum()
        a = pk.hap[sites][:, [8, 9]].astype(np.float64)
        R = (alpha * pk.n_ref[sites] + beta * pk.n_alt[sites]) @ a
        got = C0 + R[:, None] + lt.screen_operands(case, sites, 4)
        want = lt.column_terms(case, sites, 4).l1
        assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()
