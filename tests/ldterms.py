"""Case builder and per-column term calculator for the --LD epilogue tests — TEST INFRASTRUCTURE ONLY.

`ld_case` builds synthetic --LD inputs (a refcases.Case, so enginecase.run_engine and refcases.oracle_run take it
unchanged) with control over where the reads come from, which targets share a haplotype with that individual, and
which individuals are exact copies of others.  `column_terms` evaluates, in float64 from the oracle's P(D|G) table,
the terms the tensor paths sum for one window of one target:

    LIBD1 terms  l1[i, k] = sum_s ln P_s[a_i,s + k_s]      (target haplotype i, background haplotype column k)
    LIBD0 terms  q[u]     = sum_s ln P_s[r0_s + r1_s]      (unique background individual u)

with the columns in the engine's order: unique background individuals in ascending index, the pileup's own
individual left out, two haplotype columns each.  The tests use it to check their own preconditions (which tile a
row's maximum sits in, how far it climbs, which branch of LIBD0 a target takes), never as the reference."""
from __future__ import annotations

import functools
from dataclasses import dataclass

import numpy as np

import oracle
import refcases
import refio


def ld_case(seed, S, N, window, targets, *, src=0, share=(), twins=None, bg=None, pu_idx=-1, opt_v=0, depth=2.0,
            eps=0.02, max_cov=20, cull_p=1.0, keep_frac=0.97, af=None):
    """Synthetic --LD case.  Reads are drawn from individual `src` (its genotype, error rate `eps`, Poisson(`depth`)
    bases per site).  Haplotype 0 of every individual in `share` is a copy of haplotype 1 of `src` (a relative sharing
    one haplotype).  `twins` maps an individual to another whose two haplotypes it copies; copies are made after the
    shared haplotypes are planted, and the reads are drawn last.  `bg` is the background list as given on the command
    line (order and repeats kept).  `af` gives the panel's alternate-allele frequency per site (a scalar or S values);
    by default they are drawn from Beta(0.5, 2)."""
    rng = np.random.default_rng(seed)
    drawn = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99)
    af = drawn if af is None else np.broadcast_to(np.asarray(af, np.float64), (S,))
    hap = (rng.random((S, 2 * N)) < af[:, None]).astype(np.uint8)
    for t in share:
        hap[:, 2 * t] = hap[:, 2 * src + 1]
    for x, y in (twins or {}).items():
        hap[:, 2 * x:2 * x + 2] = hap[:, 2 * y:2 * y + 2]
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = np.minimum(rng.poisson(depth, S), 255)
    g = hap[:, 2 * src] + hap[:, 2 * src + 1]
    n_alt = rng.binomial(d, np.where(g == 0, eps, np.where(g == 1, 0.5, 1 - eps)))
    n_ref = d - n_alt
    keep = (rng.random(S) < keep_frac).astype(np.uint8)
    pk = refio.Packed([f"i{i}" for i in range(N)], hap, pos, keep, n_ref.astype(np.uint8), n_alt.astype(np.uint8),
                      d.astype(np.uint32), ["1"] * S, ["."] * S, ["A"] * S, ["G"] * S, None)
    prm = oracle.Params(epsilon=eps, max_cov=max_cov, window=window, ld_mode=1, opt_v=opt_v, pu_idx=pu_idx,
                        cull_p=cull_p)
    case = refcases.Case(pk, prm, list(targets), np.asarray(bg if bg is not None else range(N), np.int32), None,
                         "UNKWN", "")
    case.src = src
    return case


@functools.lru_cache(maxsize=None)
def ln_pdg(eps, max_cov):
    """ln P(D|G) [n_ref, n_alt, g] from the oracle's own P(D|G)."""
    with np.errstate(divide="ignore"):
        return np.log(oracle.pDgG_table(eps, max_cov))


def thinned(case, k):
    """The -D case as target k sees it: a copy whose counts are the k-th target's thinned counts, drawn exactly as the
    reference and the oracle draw them (enginecase.draw_downsampled_counts), with no further thinning."""
    import copy

    import enginecase
    d = case.pk.n_ref.astype(np.int64) + case.pk.n_alt
    tc = enginecase.draw_downsampled_counts(case, None, (case.pk.host_keep != 0) & (d <= case.params.max_cov))
    view = copy.deepcopy(case)
    view.pk.n_ref, view.pk.n_alt = tc[k, :, 0].copy(), tc[k, :, 1].copy()
    view.params.cull_p = 1.0
    view.targets = [case.targets[k]]
    return view


def windows(case, target):
    """Site indices of each window of `target`, by the reference's rules for the counts as given (for -D, on the
    view `thinned` returns)."""
    pk, prm = case.pk, case.params
    assert prm.cull_p == 1.0, "thinned counts are drawn by the engine and the oracle, not here"
    d = pk.n_ref.astype(np.int64) + pk.n_alt
    ok = (pk.host_keep != 0) & (d <= prm.max_cov) & (d >= 1)
    if prm.opt_v:
        ok &= (pk.hap[:, 2 * target] | pk.hap[:, 2 * target + 1]) != 0
    idx = np.flatnonzero(ok)
    return [idx[a:a + prm.window] for a in range(0, len(idx), prm.window)]


@dataclass
class Terms:
    bgU: np.ndarray      # unique background individuals, ascending (the pileup's own individual left out)
    lnmult: np.ndarray   # ln of each one's multiplicity in the background list
    own: int             # index of the target in bgU, or -1
    l1: np.ndarray       # [2, 2 nU] LIBD1 terms
    q: np.ndarray        # [nU] LIBD0 terms

    def col_terms(self):
        """l1 with the multiplicity weights and the target's own columns at -inf: what the LIBD1 sum runs over."""
        x = self.l1 + np.repeat(self.lnmult, 2)[None, :]
        if self.own >= 0:
            x[:, 2 * self.own:2 * self.own + 2] = -np.inf
        return x

    def q_terms(self):
        x = self.q + self.lnmult
        if self.own >= 0:
            x[self.own] = -np.inf
        return x

    def n_b(self):
        m = np.exp(self.lnmult).round()
        return float(m.sum() - (m[self.own] if self.own >= 0 else 0.0))

    def libd(self):
        """(LIBD0, LIBD1) of the window in natural logs, NaN when the background has no one but the target."""
        nb = self.n_b()
        if nb == 0:
            return np.nan, np.nan
        return lse(self.q_terms()) - np.log(nb), lse(self.col_terms()) - np.log(4 * nb)


def lse(x):
    x = np.asarray(x, np.float64).ravel()
    m = x.max()
    if m == -np.inf:
        return -np.inf
    return m + np.log(np.exp(x - m).sum())


def column_terms(case, window_sites, target):
    pk, prm = case.pk, case.params
    lnP = ln_pdg(prm.epsilon, prm.max_cov)
    s = np.asarray(window_sites)
    L = lnP[pk.n_ref[s], pk.n_alt[s]]  # [W, 3]
    mult = np.bincount(np.asarray(case.bg)[np.asarray(case.bg) != prm.pu_idx], minlength=len(pk.names))
    bgU = np.flatnonzero(mult)
    own = int(np.searchsorted(bgU, target)) if mult[target] else -1
    h = pk.hap[s].astype(np.int64)
    cols = h[:, np.stack([2 * bgU, 2 * bgU + 1], axis=1).ravel()]  # [W, 2 nU]
    l1 = np.stack([np.take_along_axis(L, h[:, [2 * target + i]] + cols, axis=1).sum(axis=0) for i in (0, 1)])
    q = np.take_along_axis(L, h[:, 2 * bgU] + h[:, 2 * bgU + 1], axis=1).sum(axis=0)
    return Terms(bgU, np.log(mult[bgU].astype(np.float64)), own, l1, q)


def kappa(eps):
    return float(np.log(4 * eps * (1 - eps)))


def depth_coefficients(eps, max_cov):
    """(alpha, beta, kappa) of the depth-linear class table, read off the oracle's ln P(D|G): one REF base adds alpha
    to l1 - l0, one ALT base adds beta, and every base adds kappa to l2 - 2 l1 + l0."""
    L = ln_pdg(eps, max_cov)
    return L[1, 0, 1] - L[1, 0, 0], L[0, 1, 1] - L[0, 1, 0], L[1, 0, 2] - 2 * L[1, 0, 1] + L[1, 0, 0]


def mma_mode(eps, ncols):
    """(table, delta, dpos) of the ld_mma epilogue for `ncols` background haplotype columns: the screen's reach in key
    units, the head-room a row's maximum may climb above its reference key before the reference moves, and whether
    the exp table (delta + dpos + 1 entries of at most 512) is used.  Mirrors screen_nats (tc_common.cuh) and
    ld_mma.cu:1265-1276."""
    k = -kappa(eps)
    screen = min(32.0, np.log(max(ncols, 2)) + 16.2)
    delta = int(np.ceil(screen / k)) + 2
    dpos = int(min(256.0, np.floor(600.0 / k)))
    return dpos >= 8 and delta + dpos + 1 <= 512, delta, dpos


def screen_operands(case, sites, target):
    """Y[k] + kappa M[a_i, k] in float64 for each target haplotype row i and background column k (column_terms'
    order): the part of a term that the window's C0 + R[a_i] does not carry, and what ld_vmma screens in fp32."""
    pk = case.pk
    alpha, beta, kap = depth_coefficients(case.params.epsilon, case.params.max_cov)
    s = np.asarray(sites)
    nr, na = pk.n_ref[s].astype(np.float64), pk.n_alt[s].astype(np.float64)
    bgU = column_terms(case, sites, target).bgU
    cols = pk.hap[s][:, np.stack([2 * bgU, 2 * bgU + 1], axis=1).ravel()].astype(np.float64)  # [W, 2 nU]
    rows = pk.hap[s][:, [2 * target, 2 * target + 1]].astype(np.float64)                      # [W, 2]
    Y = (alpha * nr + beta * na) @ cols
    M = (rows * (nr + na)[:, None]).T @ cols
    return Y[None, :] + kap * M


def first_tile_climb(terms, tile_cols):
    """Per target haplotype row: how far (nats) the row's maximum over all columns lies above its maximum over the
    first `tile_cols` columns — the climb a row's running maximum makes after the first tile of its unit."""
    x = terms.col_terms()
    with np.errstate(invalid="ignore"):
        return x.max(axis=1) - x[:, :tile_cols].max(axis=1)
