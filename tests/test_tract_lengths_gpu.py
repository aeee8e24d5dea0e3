"""hiddengem posterior tract-length spectrum on the GPU (hiddengem_tract_lengths_batch / _device, hiddengem --posterior
--tract-lengths, ibdgem --hiddengem --posterior --tract-lengths) against the long double oracle of
test_tract_lengths_cpu.py, against the tract-count entry at X = 1 bin, and bit for bit across batches and layouts.

Tolerance: |got - want| <= 1e-9 max(1, |want|) per table, threshold and state."""
import json
import os

import numpy as np
import pytest

import hostlib
from test_posterior_gpu import HG, _run, _summary_lik, _tables
from test_tract_lengths_cpu import conditioning_table, irregular_coords, tract_lengths_oracle

pytestmark = pytest.mark.gpu

PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "loose": (0.2, 0.05, 0.3), "zero_and_above_one": (0.0, 1e-3, 2.5)}
LOG_ARITHMETIC = {"zero_and_above_one"}


def _check(got, lik, off, th, is_log, pen, start=None, end=None):
    want = tract_lengths_oracle(lik, off, th, start, end, is_log, *pen, dtype=np.longdouble)
    assert got.shape == want.shape
    assert (np.isnan(got) == np.isnan(want)).all()
    ok = ~np.isnan(want)
    err = np.abs(got[ok] - want[ok])
    assert (err <= 1e-9 * np.maximum(1.0, np.abs(want[ok]))).all(), float(err.max())
    return want


def _coords(rng, off):
    parts = [irregular_coords(rng, int(off[t + 1] - off[t])) for t in range(len(off) - 1)]
    return np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])


@pytest.mark.parametrize("coords", [False, True])
@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 32, 33, 100])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_host_entry_matches_oracle(coords, is_log, n_tables, pen):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(500 + n_tables + 7 * is_log + 3 * coords)
    lik, off = _tables(rng, n_tables, is_log)
    start, end = _coords(rng, off) if coords else (None, None)
    th = [1, 50, 400, 2000, 9000] if coords else [1, 2, 30, 41, 200]
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        e.reset_stats()
        got = e.tract_lengths_batch(lik, off, th, start, end, is_log, *p)
        stats = e.kernel_stats()
        _, _, tr = e.tract_counts_batch(lik, off, is_log, *p, cov=False)
    runs = int(off[-1] > 0)
    assert stats["posterior_bwd_runs"][1] == runs and stats["posterior_fwd"][1] == runs and stats["tract_lengths"][1] == runs
    assert stats["posterior_bwd"][1] == 0 and stats["posterior_bwd_tracts"][1] == 0
    lg = runs * int(pen in LOG_ARITHMETIC)
    assert stats["posterior_fwd_log"][1] == lg and stats["posterior_bwd_log"][1] == lg
    _check(got, lik, off, th, is_log, p, start, end)
    assert (np.diff(got, axis=1)[~np.isnan(got[:, 1:])] <= 1e-12 * np.maximum(1, np.abs(got[:, :-1]))[~np.isnan(got[:, 1:])]).all()
    if not coords:  # X = 1 bin is the tract count
        live = ~np.isnan(tr).any(axis=1)
        np.testing.assert_allclose(got[live, 0], tr[live], rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("pen", ["default", "zero_and_above_one"])
def test_geometry_and_bit_identity(pen):
    """Tables around strides of 32 bins and blocks of 1,024, thresholds at 1, 2, 16, 17, n and n + 1 bins and inside a
    bin's own span, and the same table alone or anywhere in a batch: the same bits."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(91)
    base = [0, 1, 15, 16, 17, 31, 32, 33, 1000, 1023, 1024, 1025, 2100]
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        for n_tables in (13, 33):
            lens = np.array([base[(k * 5) % len(base)] for k in range(n_tables)])
            off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            lik = rng.normal(-40, 4, (int(off[-1]), 3))
            start, end = _coords(rng, off)
            for th, s, en in (([1, 2, 16, 17, 1000, 1001], None, None), ([1, 5, 20, 300, 30000, 10 ** 6], start, end)):
                got = e.tract_lengths_batch(lik, off, th, s, en, True, *p)
                _check(got, lik, off, th, True, p, s, en)
                for t in (0, n_tables // 2, n_tables - 1):
                    a, b = off[t], off[t + 1]
                    one = e.tract_lengths_batch(lik[a:b] if b > a else np.zeros((0, 3)), [0, lens[t]], th,
                                                None if s is None else s[a:b], None if en is None else en[a:b], True, *p)
                    np.testing.assert_array_equal(one[0], got[t])
                assert (got[lens == 0] == 0).all()
            for t in np.nonzero(lens > 0)[0][:3]:  # n and n + 1 bins of each table itself
                n = int(lens[t])
                got = e.tract_lengths_batch(lik[off[t]: off[t + 1]], [0, n], [n, n + 1], None, None, True, *p)
                _check(got, lik[off[t]: off[t + 1]], [0, n], [n, n + 1], True, p)
                assert (got[0, 1] == 0).all()


def test_edge_rules_and_rejections():
    import torch
    import ibdgem_b200 as ib
    lik = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.2, 0.3, 0.5]])
    s = np.array([10, 20, 30], np.uint64)
    en = np.array([14, 24, 34], np.uint64)
    with ib.Engine(ib.Params()) as e:
        got = e.tract_lengths_batch(lik, [0, 2, 3], [1, 5, 6], s, en, False, 0.0, 1e-3, 1e-3)
        assert np.isnan(got[0]).all()  # the only path has weight p01 = 0
        g = np.array([0.2, 0.3, 0.5])
        np.testing.assert_allclose(got[1, 1], g, rtol=0, atol=1e-15)  # one bin spanning 5 bp
        assert (got[1, 2] == 0).all()
        assert (e.tract_lengths_batch(np.zeros((0, 3)), [0, 0, 0], [1, 2]) == 0).all()
        for bad in ((-1e-3, 1e-6, 1e-3), (1e-3, 1e-6, np.nan)):
            with pytest.raises(ib.EngineError, match=r"\[::\] ERROR in hiddengem_tract_lengths_batch\(\): penalties must be finite"):
                e.tract_lengths_batch(lik, [0, 2, 3], [1], None, None, False, *bad)
        with pytest.raises(ib.EngineError, match=r"give both bin_start and bin_end"):
            e.tract_lengths_batch(lik, [0, 2, 3], [1], s, None)
        for th in ([], [0], [2, 2], [3, 2], list(range(1, 18))):
            with pytest.raises(ib.EngineError, match=r"thresholds must be 1 to 16 values >= 1, strictly increasing"):
                e.tract_lengths_batch(lik, [0, 2, 3], th)
        with pytest.raises(ib.EngineError, match=r"hiddengem_tract_lengths_batch"):
            e.tract_lengths_batch(lik, [0, 2, 1], [1])
        for bs, be in ((np.array([10, 9, 30], np.uint64), en), (s, np.array([14, 13, 34], np.uint64)),
                       (s, np.array([9, 24, 34], np.uint64))):
            with pytest.raises(ib.EngineError, match=r"bin coordinates are not sorted"):
                e.tract_lengths_batch(lik, [0, 3], [1], bs, be)
        assert e.tract_lengths_batch(lik, [0, 1, 3], [1], np.array([10, 5, 30], np.uint64), np.array([14, 24, 34], np.uint64)).shape == (2, 1, 3)
        d_lik = torch.from_numpy(lik).cuda()
        d_bs = torch.from_numpy(np.array([10, 30, 20], np.int64)).cuda()
        d_be = torch.from_numpy(np.array([14, 34, 24], np.int64)).cuda()
        d_sp = torch.zeros((1, 1, 3), dtype=torch.float64, device="cuda")
        with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_tract_lengths_device\(\): bin coordinates are not sorted"):
            e.tract_lengths_device(d_lik.data_ptr(), np.array([0, 3]), False, [1], d_sp.data_ptr(), d_bs.data_ptr(), d_be.data_ptr())
        with pytest.raises(ib.EngineError, match=r"hiddengem_tract_lengths_device\(\): give both"):
            e.tract_lengths_device(d_lik.data_ptr(), np.array([0, 3]), False, [1], d_sp.data_ptr(), d_bs.data_ptr(), 0)


def test_long_tables():
    """A 120,000-bin table with planted segments and the conditioning table, against the oracle in x87 long double."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(22)
    n = 120_000
    seg = np.repeat(rng.integers(0, 3, n // 300 + 1), 300)[:n]
    big = rng.normal(-150, 10, (n, 3))
    big[np.arange(n), seg] += 8.0
    cond = conditioning_table()
    with ib.Engine(ib.Params()) as e:
        th = [1, 100, 250, 300, 600, 5000]
        got = e.tract_lengths_batch(big, [0, n], th, None, None, True)
        _check(got, big, np.array([0, n]), th, True, PENALTIES["default"])
        th = [1, 100, 2000, 2999, 3000, 3001]
        got = e.tract_lengths_batch(cond, [0, len(cond)], th, None, None, True)
        _check(got, cond, np.array([0, len(cond)]), th, True, PENALTIES["default"])
    assert abs(got[0, 4, 2] - 1) < 1e-6


def test_device_entry_packed_and_strided_on_score_ld_window_scores():
    """The strided layout of a real score_ld call (w_loglik_device, w_start / w_end uploaded in the same layout), and
    the same tables packed: bit for bit the host entry."""
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
        ws = np.concatenate([sc.w_start[t, : nw[t]] for t in range(T)]).astype(np.uint64)
        we = np.concatenate([sc.w_end[t, : nw[t]] for t in range(T)]).astype(np.uint64)
        d_ws = torch.from_numpy(np.ascontiguousarray(sc.w_start[:, :mw]).astype(np.int64)).cuda()
        d_we = torch.from_numpy(np.ascontiguousarray(sc.w_end[:, :mw]).astype(np.int64)).cuda()
        d_pk = torch.from_numpy(packed).cuda()
        d_pws = torch.from_numpy(ws.astype(np.int64)).cuda()
        d_pwe = torch.from_numpy(we.astype(np.int64)).cuda()
        th = [60, 600, 3000, 12000]
        for pen in ("default", "zero_and_above_one"):
            p = PENALTIES[pen]
            host = e.tract_lengths_batch(packed, off, th, ws, we, True, *p)
            for src, bs, be, stride in ((d_wll, d_ws, d_we, mw), (d_pk, d_pws, d_pwe, 0)):
                d_sp = torch.zeros((T, len(th), 3), dtype=torch.float64, device="cuda")
                e.tract_lengths_device(src.data_ptr(), off, True, th, d_sp.data_ptr(), bs.data_ptr(), be.data_ptr(), table_stride=stride,
                                       p01=p[0], p02=p[1], p12=p[2])
                np.testing.assert_array_equal(d_sp.cpu().numpy(), host)
            _check(host, packed, off, th, True, p, ws, we)


# ---- command lines ----------------------------------------------------------------------------------------------
def _summary_coords(path):
    """START / END of a summary file's rows, as hiddengem keeps them."""
    s, en = [], []
    with open(path) as fh:
        for ln in fh:
            if ln.startswith("#") and not s:
                continue
            f = ln.split("\t")
            if len(f) >= 7:
                s.append(int(f[1]))
                en.append(int(f[2]))
    return np.array(s, np.uint64), np.array(en, np.uint64)


def _check_tl_block(lines, th, want, rel):
    assert len(lines) == 3 * len(th)
    j = 0
    for s in range(3):
        for k, x in enumerate(th):
            head, val = lines[j].split(": ")
            assert head == f"#% posterior IBD{s} tracts >= {x} bp"
            assert abs(float(val) - want[k, s]) <= 0.005 + rel * abs(want[k, s]), (lines[j], want[k, s])
            j += 1


@pytest.mark.parametrize("run,ind,tag,args", HG)
def test_hiddengem_tract_lengths_command_line(golden_dir, run, ind, tag, args):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    summ = os.path.join(ca, run, f"UNKWN.{ind}.summary.txt")
    th = [1, 50000, 200000, 1000000]
    plain = _run("hiddengem", ["-s", summ, "--posterior"] + args).stdout
    got = _run("hiddengem", ["-s", summ, "--posterior", "--tract-lengths", ",".join(map(str, th))] + args).stdout.splitlines()
    assert "\n".join(got[:-12]) + "\n" == plain
    pen = [float(a) for a in args[1::2]] or [1e-3, 1e-6, 1e-3]
    lik = _summary_lik(summ)
    s, en = _summary_coords(summ)
    want = tract_lengths_oracle(lik, [0, len(lik)], th, s, en, False, *pen, dtype=np.longdouble)
    _check_tl_block(got[-12:], th, want[0], 1e-6)


def test_hiddengem_tract_lengths_over_several_tables(golden_dir):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    files = [os.path.join(ca, "nonld_w10", f"UNKWN.{ind}.summary.txt") for ind in ("ind2", "ind3", "ind5")]
    args = sum((["-s", f] for f in files), [])
    th = [1, 100000]
    plain = _run("hiddengem", args + ["--posterior"]).stdout
    got = _run("hiddengem", args + ["--posterior", "--tract-lengths", "1,100000"]).stdout.splitlines()
    with_tc = _run("hiddengem", args + ["--posterior", "--tract-counts", "--tract-lengths", "1,100000"]).stdout.splitlines()
    tc_only = _run("hiddengem", args + ["--posterior", "--tract-counts"]).stdout.splitlines()
    liks = [_summary_lik(f) for f in files]
    co = [_summary_coords(f) for f in files]
    off = np.concatenate([[0], np.cumsum([len(l) for l in liks])]).astype(np.int64)
    want = tract_lengths_oracle(np.concatenate(liks), off, th, np.concatenate([c[0] for c in co]), np.concatenate([c[1] for c in co]),
                                False, dtype=np.longdouble)
    rest, at = [], 0
    for t in range(len(files)):
        end = next(i for i in range(at, len(got)) if got[i].startswith("#% posterior IBD2 (n = "))
        rest += got[at: end + 1]
        _check_tl_block(got[end + 1: end + 7], th, want[t], 1e-6)
        at = end + 7
    assert "\n".join(rest) + "\n" == plain
    block = got[at:]
    assert len(block) == 10 and block[0] == f"#% all 3 tables (n = {off[-1]})"
    _check_tl_block(block[4:], th, want.sum(axis=0), 1e-6)
    assert [ln for ln in with_tc if " tracts >= " not in ln] == tc_only  # after the tract-count lines, per table and overall
    assert with_tc[-6:] == got[-6:]


def test_ibdgem_hiddengem_tract_lengths_files(golden_dir, tmp_path):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, "nonld_w10", "ARGS.json")))
    base = ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup"] + meta["args"] + ["--hiddengem", "--no-tab", "--posterior"]
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    th = [1, 20000, 100000]
    _run("ibdgem", base + ["-O", str(tmp_path / "a")], cwd=ca)
    _run("ibdgem", base + ["-O", str(tmp_path / "b"), "--tract-lengths", "1,20000,100000"], cwd=ca)
    for ind in ("ind2", "ind3", "ind5"):
        plain = open(tmp_path / "a" / f"UNKWN.{ind}.hiddengem.txt").read()
        got = open(tmp_path / "b" / f"UNKWN.{ind}.hiddengem.txt").read().splitlines()
        assert "\n".join(got[:-9]) + "\n" == plain
        summ = tmp_path / "b" / f"UNKWN.{ind}.summary.txt"
        lik = _summary_lik(summ)  # the run's scores, to 7 significant digits
        s, en = _summary_coords(summ)
        with np.errstate(divide="ignore"):
            want = tract_lengths_oracle(np.log(lik), [0, len(lik)], th, s, en, True, dtype=np.longdouble)
        _check_tl_block(got[-9:], th, want[0], 1e-3)
