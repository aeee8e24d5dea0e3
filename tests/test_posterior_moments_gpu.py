"""hiddengem posterior moments on the GPU (hiddengem_posterior_moments_batch / _device, hiddengem --share-sd, ibdgem
--hiddengem --posterior --share-sd) against the long double oracle of test_posterior_moments_cpu.py, and bit for bit
against the posterior entries.

Tolerance, per table of n bins: |dCov_st| <= 1e-9 sqrt(Var_s Var_t) + 1e-12 n, and means within 1e-12 n."""
import json
import os

import numpy as np
import pytest

import hostlib
from test_posterior_gpu import HG, _run, _summary_lik, _tables
from test_posterior_moments_cpu import moments_oracle

pytestmark = pytest.mark.gpu

PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "loose": (0.2, 0.05, 0.3), "one": (1.0, 1.0, 1.0), "zero_and_above_one": (0.0, 1e-3, 2.5)}
LOG_ARITHMETIC = {"zero_and_above_one"}


def _check(expected, cov, lik, off, is_log, pen):
    want_e, want_c = moments_oracle(lik, off, is_log, *pen, dtype=np.longdouble)
    want_e, want_c = want_e.astype(np.float64), want_c.astype(np.float64)
    n = np.diff(off).astype(np.float64)
    assert (np.isnan(expected) == np.isnan(want_e)).all() and (np.isnan(cov) == np.isnan(want_c)).all()
    ok = ~np.isnan(want_e).any(axis=1)
    assert (np.abs(expected - want_e)[ok] <= 1e-12 * n[ok, None]).all(), np.abs(expected - want_e)[ok].max()
    v = np.abs(np.diagonal(want_c, axis1=1, axis2=2))
    bound = 1e-9 * np.sqrt(v[:, :, None] * v[:, None, :]) + 1e-12 * n[:, None, None]
    err = np.abs(cov - want_c)
    assert (err[ok] <= bound[ok]).all(), float((err[ok] / np.maximum(bound[ok], 1e-300)).max())
    return want_e, want_c


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 64, 300])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_host_entry_matches_oracle_and_the_posterior_entry(is_log, n_tables, pen):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(100 + n_tables + 7 * is_log)
    lik, off = _tables(rng, n_tables, is_log)
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        e.reset_stats()
        ex, cov, post = e.posterior_moments_batch(lik, off, is_log, *p, posterior=True)
        stats = e.kernel_stats()
        ex2, cov2 = e.posterior_moments_batch(lik, off, is_log, *p)
        post_p, ex_p = e.posterior_batch(lik, off, is_log, *p)
    runs = int(off[-1] > 0)  # a batch of empty tables launches nothing
    assert stats["posterior_bwd_moments"][1] == runs and stats["posterior_fwd"][1] == runs and stats["posterior_bwd"][1] == 0
    lg = runs * int(pen in LOG_ARITHMETIC)
    assert stats["posterior_fwd_log"][1] == lg and stats["posterior_bwd_log"][1] == lg
    np.testing.assert_array_equal(post, post_p)
    np.testing.assert_array_equal(ex, ex_p)
    np.testing.assert_array_equal(ex2, ex)
    np.testing.assert_array_equal(cov2, cov)
    _check(ex, cov, lik, off, is_log, p)
    ok = ~np.isnan(cov).any(axis=(1, 2))
    np.testing.assert_array_equal(cov, cov.transpose(0, 2, 1))
    scale = np.abs(cov[ok]).max(axis=(1, 2), initial=0.0) + np.diff(off)[ok]
    assert (np.abs(cov[ok].sum(axis=2)) <= 1e-12 * scale[:, None]).all()


@pytest.mark.parametrize("pen", ["default", "zero_and_above_one"])
def test_geometry_around_chunks_and_blocks(pen):
    """Table lengths around the 16-bin chunks, block counts around 32 tables, and the same table in any position of
    any batch gives the same bits."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(77)
    base = [0, 1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 49, 255, 256, 257, 1000]
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        for n_tables in (31, 32, 33, 65):
            lens = np.array([base[(k * 7) % len(base)] for k in range(n_tables)])
            off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            lik = rng.normal(-40, 4, (int(off[-1]), 3))
            ex, cov = e.posterior_moments_batch(lik, off, True, *p)
            _check(ex, cov, lik, off, True, p)
            for t in (0, n_tables // 2, n_tables - 1):  # alone in a batch: the same bits
                one = lik[off[t]: off[t + 1]] if lens[t] else np.zeros((0, 3))
                ex1, cov1 = e.posterior_moments_batch(one, [0, lens[t]], True, *p)
                np.testing.assert_array_equal(ex1[0], ex[t])
                np.testing.assert_array_equal(cov1[0], cov[t])
            assert (cov[lens == 0] == 0).all() and (ex[lens == 0] == 0).all()


def test_edge_rules_and_rejections():
    import ibdgem_b200 as ib
    lik = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.2, 0.3, 0.5]])
    with ib.Engine(ib.Params()) as e:
        ex, cov = e.posterior_moments_batch(lik, [0, 2, 3], False, 0.0, 1e-3, 1e-3)
        assert np.isnan(ex[0]).all() and np.isnan(cov[0]).all()  # the only path has weight p01 = 0
        g = np.array([0.2, 0.3, 0.5])
        np.testing.assert_allclose(cov[1], np.diag(g) - np.outer(g, g), rtol=0, atol=1e-15)
        ex, cov = e.posterior_moments_batch(np.zeros((0, 3)), [0, 0, 0], False)
        assert (ex == 0).all() and (cov == 0).all()
        for bad in ((-1e-3, 1e-6, 1e-3), (1e-3, 1e-6, np.nan)):
            with pytest.raises(ib.EngineError, match=r"\[::\] ERROR in hiddengem_posterior_moments_batch\(\): penalties must be finite"):
                e.posterior_moments_batch(lik, [0, 2, 3], False, *bad)
        with pytest.raises(ib.EngineError, match=r"hiddengem_posterior_moments_batch"):
            e.posterior_moments_batch(lik, [0, 2, 1], False)


def test_long_tables_against_long_double():
    """The 12,000-bin nearly flat table of the hiddengem long-table test, and a 120,000-bin table with planted
    segments, against the oracle in x87 long double."""
    import ibdgem_b200 as ib
    from test_cli_gpu import _long_table
    rng = np.random.default_rng(21)
    n = 120_000
    seg = np.repeat(rng.integers(0, 3, n // 300 + 1), 300)[:n]
    big = rng.normal(-150, 10, (n, 3))
    big[np.arange(n), seg] += 8.0
    with ib.Engine(ib.Params()) as e:
        for lik, is_log in ((_long_table(), False), (big, True)):
            off = np.array([0, len(lik)])
            ex, cov = e.posterior_moments_batch(lik, off, is_log)
            assert np.isfinite(ex).all() and np.isfinite(cov).all()
            _, want_c = _check(ex, cov, lik, off, is_log, PENALTIES["default"])
            print(f"n = {len(lik)}: sd of N = {np.sqrt(np.diag(want_c[0]))}")


def test_device_entry_packed_and_strided_on_score_ld_window_scores():
    """The strided layout of a real score_ld call (ibdgem_scores.w_loglik_device), and the same tables packed: bit
    for bit the host entry, with and without per-bin posteriors."""
    import torch
    import ibdgem_b200 as ib
    rng = np.random.default_rng(8)
    S, N, W = 30000, 64, 60
    af = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99)
    hap = (rng.random((S, 2 * N)) < af[:, None]).astype(np.uint8)
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = rng.poisson(2.0, S)
    g = hap[:, 0] + hap[:, 1]
    n_alt = rng.binomial(d, np.where(g == 0, 0.02, np.where(g == 1, 0.5, 0.98))).astype(np.uint8)
    n_ref = (d - n_alt).astype(np.uint8)
    targets = np.arange(40, dtype=np.int32)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, np.ones(S, np.uint8))
        e.upload_panel(ib.pack_bits(hap), N)
        mw = e.default_max_windows()
        d_wll = torch.full((len(targets), mw, 3), np.nan, dtype=torch.float64, device="cuda")
        sc = e.score_ld(targets, np.arange(N, dtype=np.int32), -1, device_out=d_wll.data_ptr())
        nw = sc.n_windows.astype(np.int64)
        off = np.concatenate([[0], np.cumsum(nw)]).astype(np.int64)
        packed = np.concatenate([sc.w_loglik[t, : nw[t]] for t in range(len(targets))])
        for pen in ("default", "zero_and_above_one"):
            p = PENALTIES[pen]
            eh, ch, ph = e.posterior_moments_batch(packed, off, True, *p, posterior=True)
            d_exp = torch.zeros((len(targets), 3), dtype=torch.float64, device="cuda")
            d_cov = torch.zeros((len(targets), 3, 3), dtype=torch.float64, device="cuda")
            d_post = torch.full((len(targets), mw, 3), 7.0, dtype=torch.float64, device="cuda")
            e.posterior_moments_device(d_wll.data_ptr(), off, True, d_exp.data_ptr(), d_cov.data_ptr(), d_post.data_ptr(),
                                       table_stride=mw, p01=p[0], p02=p[1], p12=p[2])
            np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
            np.testing.assert_array_equal(d_cov.cpu().numpy(), ch)
            p2 = d_post.cpu().numpy()
            for t in range(len(targets)):
                np.testing.assert_array_equal(p2[t, : nw[t]], ph[off[t]: off[t + 1]])
                assert (p2[t, nw[t]:] == 7.0).all()
            d_pk = torch.from_numpy(packed).cuda()
            d_exp.zero_()
            d_cov.zero_()
            e.posterior_moments_device(d_pk.data_ptr(), off, True, d_exp.data_ptr(), d_cov.data_ptr(), p01=p[0], p02=p[1], p12=p[2])
            np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
            np.testing.assert_array_equal(d_cov.cpu().numpy(), ch)
            _check(eh, ch, packed, off, True, p)


def test_c4_full_size():
    """10,000 tables x 10,000 bins with planted segments (as test_posterior_gpu.test_c4_full_size): means bit for bit
    the posterior entry's; every covariance finite, symmetric, rows summing to ~0, positive semi-definite within
    rounding; spot checks against the oracle.  How often the planted shares fall within 2 sd is printed, not asserted:
    the penalties are weights, not the process that planted the segments."""
    import torch
    import ibdgem_b200 as ib
    n_tables, n_bins = 10_000, 10_000
    nb = n_tables * n_bins
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=gen, device=dev).repeat_interleave(200)[:nb]
    ll = torch.randn((nb, 3), generator=gen, device=dev, dtype=torch.float64) * 10.0 - 150.0
    ll[torch.arange(nb, device=dev), seg] += 8.0
    planted = torch.stack([(seg.view(n_tables, n_bins) == s).sum(dim=1) for s in range(3)], dim=1).cpu().numpy()
    h_ll = ll.cpu().numpy()
    del ll, seg
    torch.cuda.empty_cache()
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    with ib.Engine(ib.Params()) as e:
        ex, cov = e.posterior_moments_batch(h_ll, off, True)
        _, ex_p = e.posterior_batch(h_ll, off, True)
    np.testing.assert_array_equal(ex, ex_p)
    assert np.isfinite(cov).all()
    np.testing.assert_array_equal(cov, cov.transpose(0, 2, 1))
    scale = np.abs(cov).max(axis=(1, 2)) + n_bins
    assert (np.abs(cov.sum(axis=2)) <= 1e-12 * scale[:, None]).all()
    assert (np.linalg.eigvalsh(cov).min(axis=1) >= -1e-12 * scale).all()
    for t in (0, n_tables // 2, n_tables - 1):
        sl = slice(t * n_bins, (t + 1) * n_bins)
        _check(ex[t: t + 1], cov[t: t + 1], h_ll[sl], [0, n_bins], True, PENALTIES["default"])
    sd = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
    within = (np.abs(planted - ex) <= 2 * sd).mean(axis=0)
    print(f"C4: planted IBD0/1/2 counts within 2 sd of the posterior mean in {within} of the tables; "
          f"median sd {np.median(sd, axis=0)} bins")


# ---- command lines ----------------------------------------------------------------------------------------------
def _parse_sd_block(lines):
    """(sd [3] of N, sd [3] of the share in %, kinship sd, kinship) of the four --share-sd lines."""
    sdn, sdp = [], []
    for k in range(3):
        head, val = lines[k].split(": ")
        assert head.startswith(f"#% posterior IBD{k} sd (n = ")
        sdn.append(float(head.split("= ")[1].rstrip(")")))
        sdp.append(float(val))
    head, val = lines[3].split(": ")
    assert head.startswith("#% posterior kinship (sd = ")
    return np.array(sdn), np.array(sdp), float(head.split("= ")[1].rstrip(")")), float(val)


def _check_sd_block(lines, want_e, want_c, n, rel):
    sdn, sdp, ksd, phi = _parse_sd_block(lines)
    sd = np.sqrt(np.maximum(np.diag(want_c), 0))
    assert (np.abs(sdn - sd) <= 0.005 + rel * sd).all(), (sdn, sd)
    assert (np.abs(sdp - sd / n * 100) <= 0.005 + rel * sd / n * 100).all()
    kv = (want_c[1, 1] / 16 + want_c[2, 2] / 4 + want_c[1, 2] / 4) / n ** 2
    assert abs(ksd - np.sqrt(max(kv, 0))) <= 0.00005 + rel * np.sqrt(max(kv, 0))
    assert abs(phi - (want_e[1] / 4 + want_e[2] / 2) / n) <= 0.00005 + rel


@pytest.mark.parametrize("run,ind,tag,args", HG)
def test_hiddengem_share_sd_command_line(golden_dir, run, ind, tag, args):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    summ = os.path.join(ca, run, f"UNKWN.{ind}.summary.txt")
    plain = _run("hiddengem", ["-s", summ, "--posterior"] + args).stdout
    got = _run("hiddengem", ["-s", summ, "--posterior", "--share-sd"] + args).stdout
    g = got.splitlines()
    assert "\n".join(g[:-4]) + "\n" == plain  # everything else byte for byte
    pen = [float(a) for a in args[1::2]] or [1e-3, 1e-6, 1e-3]
    lik = _summary_lik(summ)
    want_e, want_c = moments_oracle(lik, [0, len(lik)], False, *pen, dtype=np.longdouble)
    _check_sd_block(g[-4:], want_e[0].astype(float), want_c[0].astype(float), len(lik), 1e-6)


def test_hiddengem_share_sd_over_several_tables(golden_dir):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    files = [os.path.join(ca, "nonld_w10", f"UNKWN.{ind}.summary.txt") for ind in ("ind2", "ind3", "ind5")]
    args = sum((["-s", f] for f in files), [])
    plain = _run("hiddengem", args + ["--posterior"]).stdout
    got = _run("hiddengem", args + ["--posterior", "--share-sd"]).stdout.splitlines()
    liks = [_summary_lik(f) for f in files]
    off = np.concatenate([[0], np.cumsum([len(l) for l in liks])]).astype(np.int64)
    want_e, want_c = moments_oracle(np.concatenate(liks), off, False, dtype=np.longdouble)
    want_e, want_c = want_e.astype(float), want_c.astype(float)
    # each table: its plain lines followed by its four --share-sd lines; then the block over all tables
    rest, at = [], 0
    for t in range(len(files)):
        end = next(i for i in range(at, len(got)) if got[i].startswith("#% posterior IBD2 (n = "))
        rest += got[at: end + 1]
        _check_sd_block(got[end + 1: end + 5], want_e[t], want_c[t], len(liks[t]), 1e-6)
        at = end + 5
    assert "\n".join(rest) + "\n" == plain
    block = got[at:]
    assert len(block) == 8 and block[0] == f"#% all 3 tables (n = {off[-1]})"
    e_sum, c_sum = want_e.sum(axis=0), want_c.sum(axis=0)
    for k in range(3):
        head, val = block[1 + k].split(": ")
        assert head.startswith(f"#% posterior IBD{k} (n = ")
        assert abs(float(head.split("= ")[1].rstrip(")")) - e_sum[k]) <= 0.005 + 1e-6 * off[-1]
        assert abs(float(val) - e_sum[k] / off[-1] * 100) <= 0.005 + 1e-4
    _check_sd_block(block[4:], e_sum, c_sum, int(off[-1]), 1e-6)


def test_ibdgem_hiddengem_share_sd_files(golden_dir, tmp_path):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, "nonld_w10", "ARGS.json")))
    base = ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup"] + meta["args"] + ["--hiddengem", "--no-tab", "--posterior"]
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    _run("ibdgem", base + ["-O", str(tmp_path / "a")], cwd=ca)
    _run("ibdgem", base + ["-O", str(tmp_path / "b"), "--share-sd"], cwd=ca)
    for ind in ("ind2", "ind3", "ind5"):
        plain = open(tmp_path / "a" / f"UNKWN.{ind}.hiddengem.txt").read()
        got = open(tmp_path / "b" / f"UNKWN.{ind}.hiddengem.txt").read().splitlines()
        assert "\n".join(got[:-4]) + "\n" == plain
        lik = _summary_lik(tmp_path / "b" / f"UNKWN.{ind}.summary.txt")  # the run's scores, to 7 significant digits
        with np.errstate(divide="ignore"):
            want_e, want_c = moments_oracle(np.log(lik), [0, len(lik)], True, dtype=np.longdouble)
        _check_sd_block(got[-4:], want_e[0].astype(float), want_c[0].astype(float), len(lik), 1e-3)
