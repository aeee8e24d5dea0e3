"""The --LD tensor-path epilogues where a row's maximum is not in the first column tile, where LIBD0's own entry is
not individual 0, and at the eligibility edges of both paths, against the long double oracle.

The parity tests draw every pileup from individual 0, the first background column: the running maximum of a row
never climbs after the first tile, so ld_mma's reference-key move never rescales a sum it holds, ld_vmma never screens
a later maximum in fp32, and ld_ibd0's own entry always sits at chunk 0, position 0, staged in shared memory.  Each
test here builds a case that reaches one of those branches (ldterms.ld_case), asserts in float64 that it does before
the engine runs, checks which path ran (ld_path 1 = ld_mma + ld_ibd0, 2 = ld_vmma, 0 = the general path) and compares
every target with the oracle at the parity bar: integers exact, window sums to 1e-6 absolute."""
import os
import subprocess
import sys

import numpy as np
import pytest

import ldterms as lt
import refcases

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MMA_TILE = 256        # background columns per ld_mma tile (CTA pairs); 128 with IBDGEM_MMA_VARIANT=1
VMMA_TILE = 2 * 80    # background columns per ld_vmma tile (80 individuals)


def check(case, path):
    """Runs the engine, checks the path and every target against the oracle; prints the largest |d| of LIBD0 and
    LIBD1 (shown with pytest -rP)."""
    import enginecase as ec
    res = ec.run_engine(case, expanded=False)
    assert res[0]["ld_path"] == path
    worst = np.zeros(2)
    for r, o in zip(res, refcases.oracle_run(case)):
        ec.assert_matches_oracle(r, o)
        d = np.abs(r["w_log"][:, :2] - o["w_log"][:, :2])
        worst = np.fmax(worst, np.nanmax(d, axis=0, initial=0.0))
    print(f"ld_path={path} max|dLIBD0|={worst[0]:.3g} max|dLIBD1|={worst[1]:.3g}")
    return res


def in_subprocess(env, body):
    """Runs `body` in a fresh interpreter with the environment knobs `env` (the engine reads each knob once per
    process) and this module imported as `g`."""
    code = "import sys; sys.path[:0] = ['tests', '.']\nimport test_ld_epilogue_gpu as g\n" + body + "\nprint('ok')\n"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, **env),
                       cwd=ROOT, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0 and r.stdout.rstrip().endswith("ok"), r.stdout[-2000:] + r.stderr[-3000:]


def climbs(case, targets, tile_cols, view=None):
    """first_tile_climb of row 0 (the haplotype shared with the source) of each target, in every window."""
    out = []
    for k, t in enumerate(case.targets):
        if t not in targets:
            continue
        c = lt.thinned(case, k) if view == "thinned" else case
        for sites in lt.windows(c, t):
            out.append(lt.first_tile_climb(lt.column_terms(c, sites, t), tile_cols)[0])
    assert out
    return np.array(out)


# ---- ld_mma: a row maximum after the first tile, table mode and the reference-key moves ----------------------------

DEPTH = {0.001: 6.0, 0.02: 8.0, 0.1: 8.0, 0.3: 12.0}
PLACES = {  # the source's individual; its column 2 src is the maximum of every shared row
    "middle_tile": 300,        # tile 2 of 6
    "last_partial_tile": 690,  # tile 5: columns 1280 .. 1399, then padding
    "set_end": 159,            # columns 62, 63 of epilogue set 0 of tile 1
    "next_set_start": 160,     # columns 0, 1 of set 1 of tile 1
}


def late_case(eps, src, seed=11, **kw):
    share = [src - 5, src + 3]
    kw.setdefault("depth", DEPTH.get(eps, 8.0))
    case = lt.ld_case(seed, kw.pop("S", 1950), kw.pop("N", 700), kw.pop("window", 1000), share + [src], src=src,
                      share=share, eps=eps, **kw)
    case.shared = share
    return case


def assert_late(case, tile_cols, above, below=np.inf):
    cl = climbs(case, case.shared, tile_cols)
    assert cl.min() > above and cl.max() < below, (cl, above, below)
    return cl


@pytest.mark.parametrize("place", list(PLACES))
@pytest.mark.parametrize("eps", [0.001, 0.02, 0.1, 0.3])
def test_mma_late_maximum_moves_a_reference_holding_a_sum(eps, place):
    src = PLACES[place]
    case = late_case(eps, src)
    col = 2 * src
    assert {"middle_tile": col // MMA_TILE == 2, "last_partial_tile": col // MMA_TILE == 1400 // MMA_TILE,
            "set_end": col % 64 == 62, "next_set_start": col % MMA_TILE == 64}[place]
    table, delta, dpos = lt.mma_mode(eps, 1400)
    reach = dpos * -lt.kappa(eps)
    assert table
    # the row's maximum lies more than dpos keys above everything the first tile holds: the reference moves while s > 0
    cl = assert_late(case, MMA_TILE, reach)
    if eps == 0.3:
        assert cl.min() > 2 * reach  # several moves in one row
    check(case, 1)


def test_mma_climb_within_the_head_room_moves_no_reference():
    """eps = 0.02, short window, low depth: the climb drops the first tile's columns out of the screen but stays
    below dpos keys, so the reference set by the first chunk stays."""
    case = late_case(0.02, 300, seed=12, S=640, window=200, depth=2.0)
    table, delta, dpos = lt.mma_mode(0.02, 1400)
    k = -lt.kappa(0.02)
    assert table
    assert_late(case, MMA_TILE, (delta + 1) * k, (dpos - 1) * k)
    check(case, 1)


def test_mma_deep_coverage_repeated_moves():
    """max_cov = 127 (the limit of the int8 operand), ~60 reads a site: the climb is thousands of nats, so a row moves
    its reference many times."""
    case = late_case(0.02, 200, seed=13, S=2000, N=300, depth=60.0, max_cov=127)
    table, delta, dpos = lt.mma_mode(0.02, 600)
    assert table
    assert_late(case, MMA_TILE, 10 * dpos * -lt.kappa(0.02))
    check(case, 1)


def test_mma_late_maximum_on_the_exp_path():
    in_subprocess({"IBDGEM_MMA_TABLE": "0"},
                  "case = g.late_case(0.02, 300)\n"
                  "g.assert_late(case, g.MMA_TILE, 600.0)\n"
                  "g.check(case, 1)")


def test_mma_late_maximum_single_cta_tiles():
    """128-column tiles: the maximum at column 600 is four tiles in."""
    in_subprocess({"IBDGEM_MMA_VARIANT": "1"},
                  "case = g.late_case(0.02, 300)\n"
                  "_, _, dpos = g.lt.mma_mode(0.02, 1400)\n"
                  "g.assert_late(case, 128, dpos * -g.lt.kappa(0.02))\n"
                  "g.check(case, 1)")


def test_mma_late_maximum_without_the_max_only_pass():
    """No warm tile: the first tile is screened against the running maximum as it comes, so with the source in the
    second 32-column chunk of set 0 the reference moves inside tile 0, over the sum of the first chunk."""
    in_subprocess({"IBDGEM_MMA_WARM_TILES": "0"},
                  "_, _, dpos = g.lt.mma_mode(0.02, 1400)\n"
                  "reach = dpos * -g.lt.kappa(0.02)\n"
                  "case = g.late_case(0.02, 300)\n"
                  "g.assert_late(case, g.MMA_TILE, reach)\n"
                  "g.check(case, 1)\n"
                  "case = g.late_case(0.02, 20, seed=14)\n"
                  "assert 32 <= 2 * 20 < 64\n"
                  "g.assert_late(case, 32, reach)\n"
                  "g.check(case, 1)")


@pytest.mark.parametrize("eps,table", [(0.353, True), (0.354, False)])
def test_mma_either_side_of_the_table_switch(eps, table):
    """At 600 columns delta + dpos + 1 passes the 512 table entries between eps = 0.353 and 0.354."""
    assert lt.mma_mode(eps, 600)[0] == table
    case = late_case(eps, 200, seed=15, S=1500, N=300, depth=12.0)
    assert_late(case, MMA_TILE, 0.0)
    check(case, 1)


@pytest.mark.parametrize("window,path", [(1024, 1), (1025, 0)])
def test_mma_eligibility_edge_of_the_window(window, path):
    """1,024 sites fill the resident target tile (8 k-blocks of 128); one more takes the general path."""
    case = late_case(0.02, 30, seed=16, S=2300, N=40, window=window, depth=3.0)
    check(case, path)


# ---- ld_ibd0: the target's own entry in LIBD0 -----------------------------------------------------------------------

def own_case(N, src, seed=21, twins=None, bg=None, pu_idx=-1, S=600, window=100):
    return lt.ld_case(seed, S, N, window, [src], src=src, twins=twins, bg=bg, pu_idx=pu_idx, depth=4.0)


def own_terms(case, t):
    return [lt.column_terms(case, sites, t) for sites in lt.windows(case, t)]


def assert_own_dominates(case, t, u, twin=None):
    """The target's own (multiplicity-weighted) entry is index u of the unique background and holds more than half of
    LIBD0's mass (the re-sum branch), or with an exact twin exactly half of it, up to e-30."""
    for te in own_terms(case, t):
        assert te.own == u
        q = te.q + te.lnmult
        if twin is None:
            assert q[u] > lt.lse(np.delete(q, u)) + 5.0
        else:
            assert te.q[twin] == te.q[u]
            assert lt.lse(np.delete(q, [u, twin])) < q[u] - 30.0


@pytest.mark.parametrize("N,src", [
    (50, 17), (50, 49),     # clen = 1: each chunk holds one entry; 49 is the last chunk with any
    (300, 35), (300, 39),   # clen = 5: first and last index of chunk 7
    (301, 300),             # clen = 5, nU not a multiple of 64: the own entry alone in the last chunk
])
def test_ibd0_dominating_own_entry_across_chunks(N, src):
    case = own_case(N, src)
    clen = -(-N // 64)
    assert (N, clen) in ((50, 1), (300, 5), (301, 5))
    assert_own_dominates(case, src, src)
    check(case, 1)


@pytest.mark.parametrize("N,src,twin", [(300, 35, 36), (300, 35, 200), (50, 20, 21)])
def test_ibd0_own_entry_with_an_exact_twin(N, src, twin):
    """The own term is exactly half of the mass: the boundary of x + x <= tot_s.  The twin in the own entry's chunk
    (36; and 21 with one entry a chunk) and in another (200)."""
    case = own_case(N, src, twins={twin: src})
    assert_own_dominates(case, src, src, twin=twin)
    check(case, 1)


def test_ibd0_own_entry_beyond_the_shared_memory_stage():
    """nU = 20,481: Q' no longer fits the 160 KB stage and is read from global memory; the own entry is the last one,
    in the partial last chunk."""
    N = 20481
    assert N * 8 > 160 * 1024 and 20481 // -(-N // 64) == 63
    case = own_case(N, N - 1, S=200, window=100)
    assert_own_dominates(case, N - 1, N - 1)
    check(case, 1)


def test_ibd0_target_that_is_the_pileup_individual_has_no_own_entry():
    case = own_case(300, 120, pu_idx=120)
    for te in own_terms(case, 120):
        assert te.own == -1 and 120 not in te.bgU and len(te.bgU) == 299
    check(case, 1)


def test_ibd0_target_listed_several_times_is_removed_as_a_whole():
    case = own_case(300, 37, bg=list(range(300)) + [37, 37])
    for te in own_terms(case, 37):
        assert te.lnmult[37] == np.log(3.0)
    assert_own_dominates(case, 37, 37)
    check(case, 1)


# ---- ld_vmma (-v, -D) -----------------------------------------------------------------------------------------------

def v_case(src, opt_v=1, cull_p=1.0, seed=31, targets=None, S=1500, window=300):
    """250 individuals: column tiles of 80 individuals 0, 1, 2 and a partial tile 3 (240 .. 249).  The source's
    twin is its neighbour, and the source is a target, so its own entry sits next to an exact copy."""
    share = [src - 7, src - 3]
    tg = share + [src, src + 1] if targets is None else targets
    case = lt.ld_case(seed, S, 250, window, tg, src=src, share=share, twins={src + 1: src}, opt_v=opt_v,
                      cull_p=cull_p, depth=6.0)
    case.shared = share
    return case


def v_reach(nU=250):
    return min(32.0, np.log(2 * nU) + 16.2) + 2.0  # ld_vmma's screen in nats (v_screen_nats + 2)


@pytest.mark.parametrize("opt_v,cull_p", [(1, 1.0), (1, 0.5), (0, 0.5)])
@pytest.mark.parametrize("src", [100, 245])  # column tile 1, and the last, partial tile
def test_vmma_late_maximum_and_own_entry_next_to_its_twin(src, opt_v, cull_p):
    case = v_case(src, opt_v=opt_v, cull_p=cull_p)
    cl = climbs(case, case.shared, VMMA_TILE, view="thinned" if cull_p < 1 else None)
    assert cl.min() > v_reach(), cl  # the first tile's survivors are rescaled by the fp64 climb
    k = case.targets.index(src)
    view = lt.thinned(case, k) if cull_p < 1 else case
    for te in own_terms(view, src):
        assert te.own == src and te.own // 80 == src // 80 >= 1 and te.q[src + 1] == te.q[src]
    check(case, 2)


@pytest.mark.parametrize("n_tw", [63, 64, 65, 129])
def test_vmma_row_tile_edges(n_tw):
    """One window a target, so the (target, window) pairs are the targets: row tiles of 64 pairs, full and not."""
    case = v_case(245, targets=[238, 242] + list(range(n_tw - 2)), S=400, window=400)
    assert sum(len(lt.windows(case, t)) for t in case.targets) == n_tw
    assert climbs(case, case.shared, VMMA_TILE).min() > v_reach()
    check(case, 2)


def v_magnitude(eps, max_cov, window):
    alpha, beta, kap = lt.depth_coefficients(eps, max_cov)
    return window * max_cov * (abs(alpha) + abs(beta) + abs(kap))


# eps = 0.001, max_cov = 100: the widest window the fp32 screen accepts
MAG_W = int(4.0e6 // v_magnitude(0.001, 100, 1))


@pytest.mark.parametrize("window,path", [(MAG_W, 2), (MAG_W + 1, 0)])
def test_vmma_fp32_screen_at_magnitude_and_its_eligibility_edge(window, path):
    """Deep reads at high allele frequencies over a window of ~3,200 sites: the screen operands Y + kappa M reach 2^20,
    where an fp32 ulp is 1/8 nat.  One site more and W max_cov (|alpha| + |beta| + |kappa|) passes 4e6: the general
    path takes over."""
    assert v_magnitude(0.001, 100, MAG_W) < 4.0e6 - 1.0 < 4.0e6 + 1.0 < v_magnitude(0.001, 100, MAG_W + 1)
    case = lt.ld_case(41, 7000, 40, window, [0, 1, 2], src=1, opt_v=1, eps=0.001, max_cov=100, depth=80.0, af=0.97)
    # target 0 is heterozygous at every site: its haplotype-0 row has M = 0, so Y alone (~500 nats a site of ALT
    # reads) is what the screen sees
    case.pk.hap[:, 0], case.pk.hap[:, 1] = 0, 1
    top = max(np.abs(lt.screen_operands(case, sites, 0)).max() for sites in lt.windows(case, 0))
    assert top >= 2.0**20, top
    check(case, path)
