"""hiddengem posterior tract counts on the GPU (hiddengem_tract_counts_batch / _device, hiddengem --posterior
--tract-counts, ibdgem --hiddengem --posterior --tract-counts) against the long double oracle of
test_tract_counts_cpu.py, and bit for bit against the posterior entries.

Tolerance, per table of n bins: means (expected, switches, tracts) within 1e-12 n, and
|dCov_st| <= 1e-9 sqrt(Var_s Var_t) + 1e-12 n for the covariance of the tract counts."""
import json
import os

import numpy as np
import pytest

import hostlib
from test_posterior_gpu import HG, _run, _summary_lik, _tables
from test_tract_counts_cpu import tract_counts_oracle

pytestmark = pytest.mark.gpu

PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "loose": (0.2, 0.05, 0.3), "one": (1.0, 1.0, 1.0), "zero_and_above_one": (0.0, 1e-3, 2.5)}
LOG_ARITHMETIC = {"zero_and_above_one"}


def _check(got, lik, off, is_log, pen):
    """got = (expected, switches, tracts, tract_cov) against the long double oracle; returns the oracle's."""
    want = [w.astype(np.float64) for w in tract_counts_oracle(lik, off, is_log, *pen, dtype=np.longdouble)]
    n = np.diff(off).astype(np.float64)
    for g, w in zip(got, want):
        assert (np.isnan(g) == np.isnan(w)).all()
    ok = ~np.isnan(want[0]).any(axis=1)
    for g, w in zip(got[:3], want[:3]):
        err = np.abs(g - w).reshape(len(n), -1)[ok]
        assert (err <= 1e-12 * n[ok, None]).all(), err.max()
    if got[3] is not None:
        v = np.abs(np.diagonal(want[3], axis1=1, axis2=2))
        bound = 1e-9 * np.sqrt(v[:, :, None] * v[:, None, :]) + 1e-12 * n[:, None, None]
        err = np.abs(got[3] - want[3])
        assert (err[ok] <= bound[ok]).all(), float((err[ok] / np.maximum(bound[ok], 1e-300)).max())
    return want


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 64, 300])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_host_entry_matches_oracle_and_the_posterior_entry(is_log, n_tables, pen):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(300 + n_tables + 7 * is_log)
    lik, off = _tables(rng, n_tables, is_log)
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        e.reset_stats()
        ex, sw, tr, tc = e.tract_counts_batch(lik, off, is_log, *p)
        stats = e.kernel_stats()
        ex2, sw2, tr2 = e.tract_counts_batch(lik, off, is_log, *p, cov=False)
        _, ex_p = e.posterior_batch(lik, off, is_log, *p)
    runs = int(off[-1] > 0)  # a batch of empty tables launches nothing
    assert stats["posterior_bwd_tracts"][1] == runs and stats["posterior_fwd"][1] == runs
    assert stats["posterior_bwd"][1] == 0 and stats["posterior_bwd_moments"][1] == 0
    lg = runs * int(pen in LOG_ARITHMETIC)
    assert stats["posterior_fwd_log"][1] == lg and stats["posterior_bwd_log"][1] == lg
    np.testing.assert_array_equal(ex, ex_p)
    np.testing.assert_array_equal(ex2, ex)
    np.testing.assert_array_equal(sw2, sw)
    np.testing.assert_array_equal(tr2, tr)
    _check((ex, sw, tr, tc), lik, off, is_log, p)
    np.testing.assert_array_equal(tc, tc.transpose(0, 2, 1))


@pytest.mark.parametrize("pen", ["default", "zero_and_above_one"])
def test_geometry_around_chunks_and_blocks(pen):
    """Table lengths around the 16-bin chunks, block counts around 32 tables, and the same table in any position of
    any batch gives the same bits."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(78)
    base = [0, 1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 49, 255, 256, 257, 1000]
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        for n_tables in (31, 32, 33, 65):
            lens = np.array([base[(k * 7) % len(base)] for k in range(n_tables)])
            off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            lik = rng.normal(-40, 4, (int(off[-1]), 3))
            got = e.tract_counts_batch(lik, off, True, *p)
            _check(got, lik, off, True, p)
            for t in (0, n_tables // 2, n_tables - 1):  # alone in a batch: the same bits
                one = lik[off[t]: off[t + 1]] if lens[t] else np.zeros((0, 3))
                got1 = e.tract_counts_batch(one, [0, lens[t]], True, *p)
                for a, b in zip(got1, got):
                    np.testing.assert_array_equal(a[0], b[t])
            for a in got:
                assert (a[lens == 0] == 0).all()


def test_edge_rules_and_rejections():
    import ibdgem_b200 as ib
    lik = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.2, 0.3, 0.5]])
    with ib.Engine(ib.Params()) as e:
        ex, sw, tr, tc = e.tract_counts_batch(lik, [0, 2, 3], False, 0.0, 1e-3, 1e-3)
        for a in (ex, sw, tr, tc):
            assert np.isnan(a[0]).all()  # the only path has weight p01 = 0
        g = np.array([0.2, 0.3, 0.5])
        np.testing.assert_array_equal(sw[1], 0.0)
        np.testing.assert_allclose(tr[1], g, rtol=0, atol=1e-15)
        np.testing.assert_allclose(tc[1], np.diag(g) - np.outer(g, g), rtol=0, atol=1e-15)
        for a in e.tract_counts_batch(np.zeros((0, 3)), [0, 0, 0], False):
            assert (a == 0).all()
        for bad in ((-1e-3, 1e-6, 1e-3), (1e-3, 1e-6, np.nan)):
            with pytest.raises(ib.EngineError, match=r"\[::\] ERROR in hiddengem_tract_counts_batch\(\): penalties must be finite"):
                e.tract_counts_batch(lik, [0, 2, 3], False, *bad)
        with pytest.raises(ib.EngineError, match=r"hiddengem_tract_counts_batch"):
            e.tract_counts_batch(lik, [0, 2, 1], False)


def test_long_and_clear_cut_tables():
    """A 120,000-bin table with planted segments against the oracle in x87 long double, and a clear-cut planted table
    whose expected tract counts are the planted runs with sd near 0."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(22)
    n = 120_000
    seg = np.repeat(rng.integers(0, 3, n // 300 + 1), 300)[:n]
    big = rng.normal(-150, 10, (n, 3))
    big[np.arange(n), seg] += 8.0
    runs = np.cumsum(rng.integers(1, 3, 40)) % 3  # neighbouring runs differ
    cut = np.repeat(runs, 250)
    clear = rng.normal(-150, 1, (len(cut), 3))
    clear[np.arange(len(cut)), cut] += 60.0
    with ib.Engine(ib.Params()) as e:
        got = e.tract_counts_batch(big, [0, n], True)
        assert all(np.isfinite(a).all() for a in got)
        want = _check(got, big, np.array([0, n]), True, PENALTIES["default"])
        print(f"n = {n}: E[T] = {want[2][0]}, sd of T = {np.sqrt(np.diag(want[3][0]))}")
        ex, sw, tr, tc = e.tract_counts_batch(clear, [0, len(cut)], True)
    np.testing.assert_allclose(tr[0], np.bincount(runs, minlength=3), rtol=0, atol=1e-9)
    assert (np.sqrt(np.maximum(np.diag(tc[0]), 0)) < 1e-4).all()


def test_device_entry_packed_and_strided_on_score_ld_window_scores():
    """The strided layout of a real score_ld call (ibdgem_scores.w_loglik_device), and the same tables packed: bit
    for bit the host entry, with and without the covariance."""
    import torch
    import ibdgem_b200 as ib
    rng = np.random.default_rng(9)
    S, N, W = 30000, 64, 60
    af = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99)
    hap = (rng.random((S, 2 * N)) < af[:, None]).astype(np.uint8)
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = rng.poisson(2.0, S)
    g = hap[:, 0] + hap[:, 1]
    n_alt = rng.binomial(d, np.where(g == 0, 0.02, np.where(g == 1, 0.5, 0.98))).astype(np.uint8)
    n_ref = (d - n_alt).astype(np.uint8)
    targets = np.arange(40, dtype=np.int32)
    T = len(targets)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, np.ones(S, np.uint8))
        e.upload_panel(ib.pack_bits(hap), N)
        mw = e.default_max_windows()
        d_wll = torch.full((T, mw, 3), np.nan, dtype=torch.float64, device="cuda")
        sc = e.score_ld(targets, np.arange(N, dtype=np.int32), -1, device_out=d_wll.data_ptr())
        nw = sc.n_windows.astype(np.int64)
        off = np.concatenate([[0], np.cumsum(nw)]).astype(np.int64)
        packed = np.concatenate([sc.w_loglik[t, : nw[t]] for t in range(T)])
        d_pk = torch.from_numpy(packed).cuda()
        for pen in ("default", "zero_and_above_one"):
            p = PENALTIES[pen]
            host = e.tract_counts_batch(packed, off, True, *p)
            for src, stride in ((d_wll, mw), (d_pk, 0)):
                for with_cov in (True, False):
                    d = [torch.zeros(s, dtype=torch.float64, device="cuda") for s in ((T, 3), (T, 3, 3), (T, 3), (T, 3, 3))]
                    e.tract_counts_device(src.data_ptr(), off, True, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(),
                                          d[3].data_ptr() if with_cov else 0, table_stride=stride, p01=p[0], p02=p[1], p12=p[2])
                    for k in range(4 if with_cov else 3):
                        np.testing.assert_array_equal(d[k].cpu().numpy(), host[k])
                    if not with_cov:
                        assert (d[3] == 0).all()
            _check(host, packed, off, True, p)


# ---- command lines ----------------------------------------------------------------------------------------------
def _parse_tc_block(lines):
    """(E[T] [3], sd of T [3], E[S] [3, 3] off the diagonal) of the nine --tract-counts lines."""
    mt, sd, sw = np.zeros(3), np.zeros(3), np.full((3, 3), np.nan)
    for k in range(3):
        head, val = lines[k].split(": ")
        assert head.startswith(f"#% posterior IBD{k} tracts (sd = ")
        sd[k] = float(head.split("= ")[1].rstrip(")"))
        mt[k] = float(val)
    j = 3
    for k in range(3):
        for l in range(3):
            if k != l:
                head, val = lines[j].split(": ")
                assert head == f"#% posterior switches IBD{k}>IBD{l}"
                sw[k, l] = float(val)
                j += 1
    return mt, sd, sw


def _check_tc_block(lines, want_sw, want_tr, want_tc, rel):
    assert len(lines) == 9
    mt, sd, sw = _parse_tc_block(lines)
    assert (np.abs(mt - want_tr) <= 0.005 + rel * want_tr).all(), (mt, want_tr)
    wsd = np.sqrt(np.maximum(np.diag(want_tc), 0))
    assert (np.abs(sd - wsd) <= 0.005 + rel * wsd).all(), (sd, wsd)
    off = ~np.eye(3, dtype=bool)
    assert (np.abs(sw[off] - want_sw[off]) <= 0.005 + rel * want_sw[off]).all(), (sw, want_sw)


@pytest.mark.parametrize("run,ind,tag,args", HG)
def test_hiddengem_tract_counts_command_line(golden_dir, run, ind, tag, args):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    summ = os.path.join(ca, run, f"UNKWN.{ind}.summary.txt")
    plain = _run("hiddengem", ["-s", summ, "--posterior"] + args).stdout
    got = _run("hiddengem", ["-s", summ, "--posterior", "--tract-counts"] + args).stdout.splitlines()
    assert "\n".join(got[:-9]) + "\n" == plain  # everything else byte for byte
    pen = [float(a) for a in args[1::2]] or [1e-3, 1e-6, 1e-3]
    lik = _summary_lik(summ)
    _, sw, tr, tc = tract_counts_oracle(lik, [0, len(lik)], False, *pen, dtype=np.longdouble)
    _check_tc_block(got[-9:], sw[0].astype(float), tr[0].astype(float), tc[0].astype(float), 1e-6)


def test_hiddengem_tract_counts_over_several_tables(golden_dir):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    files = [os.path.join(ca, "nonld_w10", f"UNKWN.{ind}.summary.txt") for ind in ("ind2", "ind3", "ind5")]
    args = sum((["-s", f] for f in files), [])
    plain = _run("hiddengem", args + ["--posterior"]).stdout
    got = _run("hiddengem", args + ["--posterior", "--tract-counts"]).stdout.splitlines()
    both = _run("hiddengem", args + ["--posterior", "--share-sd", "--tract-counts"]).stdout.splitlines()
    sd_only = _run("hiddengem", args + ["--posterior", "--share-sd"]).stdout.splitlines()
    liks = [_summary_lik(f) for f in files]
    off = np.concatenate([[0], np.cumsum([len(l) for l in liks])]).astype(np.int64)
    ex, sw, tr, tc = (a.astype(float) for a in tract_counts_oracle(np.concatenate(liks), off, False, dtype=np.longdouble))
    # each table: its plain lines followed by its nine --tract-counts lines; then the block over all tables
    rest, at = [], 0
    for t in range(len(files)):
        end = next(i for i in range(at, len(got)) if got[i].startswith("#% posterior IBD2 (n = "))
        rest += got[at: end + 1]
        _check_tc_block(got[end + 1: end + 10], sw[t], tr[t], tc[t], 1e-6)
        at = end + 10
    assert "\n".join(rest) + "\n" == plain
    block = got[at:]
    assert len(block) == 13 and block[0] == f"#% all 3 tables (n = {off[-1]})"
    e_sum = ex.sum(axis=0)
    for k in range(3):
        head, val = block[1 + k].split(": ")
        assert head.startswith(f"#% posterior IBD{k} (n = ")
        assert abs(float(head.split("= ")[1].rstrip(")")) - e_sum[k]) <= 0.005 + 1e-6 * off[-1]
    _check_tc_block(block[4:], sw.sum(axis=0), tr.sum(axis=0), tc.sum(axis=0), 1e-6)
    # with --share-sd too: its lines, then these, per table and over all tables
    assert [ln for ln in both if "tracts" not in ln and "switches" not in ln] == sd_only
    assert both[-9:] == got[-9:]


def test_ibdgem_hiddengem_tract_counts_files(golden_dir, tmp_path):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, "nonld_w10", "ARGS.json")))
    base = ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup"] + meta["args"] + ["--hiddengem", "--no-tab", "--posterior"]
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    _run("ibdgem", base + ["-O", str(tmp_path / "a")], cwd=ca)
    _run("ibdgem", base + ["-O", str(tmp_path / "b"), "--tract-counts"], cwd=ca)
    for ind in ("ind2", "ind3", "ind5"):
        plain = open(tmp_path / "a" / f"UNKWN.{ind}.hiddengem.txt").read()
        got = open(tmp_path / "b" / f"UNKWN.{ind}.hiddengem.txt").read().splitlines()
        assert "\n".join(got[:-9]) + "\n" == plain
        lik = _summary_lik(tmp_path / "b" / f"UNKWN.{ind}.summary.txt")  # the run's scores, to 7 significant digits
        with np.errstate(divide="ignore"):
            _, sw, tr, tc = tract_counts_oracle(np.log(lik), [0, len(lik)], True, dtype=np.longdouble)
        _check_tc_block(got[-9:], sw[0].astype(float), tr[0].astype(float), tc[0].astype(float), 1e-3)
