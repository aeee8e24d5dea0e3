"""hiddengem posterior on the GPU (hiddengem_posterior_batch[_device], hiddengem --posterior, ibdgem --hiddengem
--posterior) against the log-space oracle of test_posterior_cpu.py."""
import json
import os
import subprocess

import numpy as np
import pytest

import hostlib
from test_posterior_cpu import posterior_oracle

pytestmark = pytest.mark.gpu

PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "loose": (0.2, 0.05, 0.3), "one": (1.0, 1.0, 1.0), "zero_and_above_one": (0.0, 1e-3, 2.5)}


def _tables(rng, n_tables, is_log):
    """Ragged tables with planted segments, empty tables, and uninformative rows (text: all zero; log: NaN or -inf)."""
    lens = rng.integers(1, 600, n_tables)
    lens[rng.random(n_tables) < 0.1] = 0
    if n_tables > 1:
        lens[1] = 0
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nb = int(off[-1])
    seg = np.repeat(rng.integers(0, 3, nb // 40 + 1), 40)[:nb]
    if is_log:
        lik = rng.normal(-200, 30, (nb, 3))
        lik[np.arange(nb), seg] += 5.0
        lik[rng.random(nb) < 0.01] = np.nan
        lik[rng.random(nb) < 0.01] = -np.inf
        lik[rng.random(nb) < 0.01, 2] = -np.inf
    else:
        lik = np.exp(rng.normal(-20, 3, (nb, 3)))
        lik[np.arange(nb), seg] *= np.exp(5.0)
        lik[rng.random(nb) < 0.01] = 0.0
        lik[rng.random(nb) < 0.01, 1] = 0.0
    return lik, off


def _check(post, expected, lik, off, is_log, pen):
    want_p, want_e = posterior_oracle(lik, off, is_log, *pen)
    np.testing.assert_allclose(post, want_p, rtol=0, atol=1e-9, equal_nan=True)
    np.testing.assert_allclose(expected, want_e, rtol=0, atol=1e-6, equal_nan=True)
    ok = ~np.isnan(post).any(axis=1)
    np.testing.assert_allclose(post[ok].sum(axis=1), 1.0, rtol=0, atol=1e-12)
    lens = np.diff(off)
    for t in range(len(lens)):
        g = post[off[t]: off[t + 1]]
        if not np.isnan(g).any():
            np.testing.assert_allclose(expected[t], g.sum(axis=0), rtol=0, atol=1e-9 * max(int(lens[t]), 1))
        if lens[t] == 0:
            np.testing.assert_array_equal(expected[t], 0.0)


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 64, 300])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_host_entry_matches_oracle(is_log, n_tables, pen):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(100 + n_tables + 7 * is_log)
    lik, off = _tables(rng, n_tables, is_log)
    if int(off[-1]) == 0:
        off[-1] = 1
        lik = np.array([[0.1, 0.2, 0.3]])
    with ib.Engine(ib.Params()) as e:
        post, expected = e.posterior_batch(lik, off, is_log, *PENALTIES[pen])
        stats = e.kernel_stats()
    assert stats["posterior_fwd"][1] == 1 and stats["posterior_bwd"][1] == 1
    _check(post, expected, lik, off, is_log, PENALTIES[pen])


def test_zero_weight_table_and_rejected_penalties():
    import ibdgem_b200 as ib
    lik = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.2, 0.3, 0.5]])
    off = np.array([0, 2, 3])
    with ib.Engine(ib.Params()) as e:
        post, expected = e.posterior_batch(lik, off, False, 0.0, 1e-3, 1e-3)
        assert np.isnan(post[:2]).all() and np.isnan(expected[0]).all()  # the only path has weight p01 = 0
        np.testing.assert_allclose(post[2], [0.2, 0.3, 0.5], rtol=1e-14)  # one bin: the normalised row
        np.testing.assert_allclose(expected[1], [0.2, 0.3, 0.5], rtol=1e-14)
        for bad in ((-1e-3, 1e-6, 1e-3), (1e-3, -0.5, 1e-3), (1e-3, 1e-6, np.nan), (np.inf, 1e-6, 1e-3)):
            with pytest.raises(ib.EngineError, match=r"\[::\] ERROR in hiddengem_posterior_batch\(\): penalties must be finite"):
                e.posterior_batch(lik, off, False, *bad)
        # only empty tables: no rows, expected counts 0
        post, expected = e.posterior_batch(np.zeros((0, 3)), [0, 0, 0], False)
        assert post.shape == (0, 3) and (expected == 0).all()


@pytest.mark.parametrize("is_log", [False, True])
def test_uninformative_rows_are_exactly_uniform(is_log):
    """An all-zero text row, or a NaN / -inf log row, gives exactly the result of a row of three equal values (a
    text row of 0.5s is the uniform emission up to a power of two, which the kernels' scaling removes exactly)."""
    import ibdgem_b200 as ib
    rng = np.random.default_rng(3)
    lik, off = _tables(rng, 40, is_log)
    nb = int(off[-1])
    rows = rng.choice(nb, 60, replace=False)
    a, b = lik.copy(), lik.copy()
    if is_log:
        a[rows[:30]] = np.nan
        a[rows[30:]] = -np.inf
        b[rows] = -7.0
    else:
        a[rows] = 0.0
        b[rows] = 0.5
    with ib.Engine(ib.Params()) as e:
        pa, ea = e.posterior_batch(a, off, is_log)
        pb, eb = e.posterior_batch(b, off, is_log)
    np.testing.assert_array_equal(pa, pb)
    np.testing.assert_array_equal(ea, eb)
    _check(pa, ea, a, off, is_log, PENALTIES["default"])


def test_long_table_below_the_long_double_range():
    """The 12,000 nearly flat bins of the hiddengem long-table test (tests/golden/hiddengem_tables/long.*): the
    reference's running products leave the long double range; the scaled forward-backward does not."""
    import ibdgem_b200 as ib
    from test_cli_gpu import _long_table
    l = _long_table()
    off = np.array([0, len(l)])
    with ib.Engine(ib.Params()) as e:
        post, expected = e.posterior_batch(l, off, False)
    assert np.isfinite(post).all() and np.isfinite(expected).all()
    _check(post, expected, l, off, False, PENALTIES["default"])


@pytest.mark.parametrize("n_tables", [5, 96])
def test_device_entry_packed_and_strided_match_host_entry(n_tables):
    import torch
    import ibdgem_b200 as ib
    rng = np.random.default_rng(31)
    lens = rng.integers(300, 500, n_tables)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nb = int(off[-1])
    ll = rng.normal(-200, 30, (nb, 3))
    seg = np.repeat(rng.integers(0, 3, nb // 25 + 1), 25)[:nb]
    ll[np.arange(nb), seg] += 5.0
    stride = 512
    strided = np.full((n_tables, stride, 3), np.nan)
    for t in range(n_tables):
        strided[t, : lens[t]] = ll[off[t]: off[t + 1]]
    with ib.Engine(ib.Params()) as e:
        ph, eh = e.posterior_batch(ll, off, True)
        d_ll = torch.from_numpy(ll).cuda()
        d_post = torch.zeros((nb, 3), dtype=torch.float64, device="cuda")
        d_exp = torch.zeros((n_tables, 3), dtype=torch.float64, device="cuda")
        e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr())
        np.testing.assert_array_equal(d_post.cpu().numpy(), ph)
        np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
        d_str = torch.from_numpy(strided).cuda()
        d_post2 = torch.full((n_tables, stride, 3), 7.0, dtype=torch.float64, device="cuda")
        d_exp.zero_()
        e.posterior_batch_device(d_str.data_ptr(), off, True, d_post2.data_ptr(), d_exp.data_ptr(), table_stride=stride)
        p2 = d_post2.cpu().numpy()
        np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
        for t in range(n_tables):
            np.testing.assert_array_equal(p2[t, : lens[t]], ph[off[t]: off[t + 1]])
            assert (p2[t, lens[t]:] == 7.0).all()  # nothing is written past a table's bins
    _check(ph, eh, ll, off, True, PENALTIES["default"])


def test_device_entry_on_the_window_scores_of_score_ld():
    """The strided layout of a real score_ld call: ibdgem_scores.w_loglik_device ([T][max_windows][3] natural logs)."""
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
    keep = np.ones(S, np.uint8)
    targets = np.arange(40, dtype=np.int32)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, keep)
        e.upload_panel(ib.pack_bits(hap), N)
        mw = e.default_max_windows()
        d_wll = torch.full((len(targets), mw, 3), np.nan, dtype=torch.float64, device="cuda")
        sc = e.score_ld(targets, np.arange(N, dtype=np.int32), -1, device_out=d_wll.data_ptr())
        nw = sc.n_windows.astype(np.int64)
        off = np.concatenate([[0], np.cumsum(nw)]).astype(np.int64)
        packed = np.concatenate([sc.w_loglik[t, : nw[t]] for t in range(len(targets))])
        ph, eh = e.posterior_batch(packed, off, True)
        d_post = torch.full((len(targets), mw, 3), 7.0, dtype=torch.float64, device="cuda")
        d_exp = torch.zeros((len(targets), 3), dtype=torch.float64, device="cuda")
        e.posterior_batch_device(d_wll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), table_stride=mw)
    p2 = d_post.cpu().numpy()
    np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
    for t in range(len(targets)):
        np.testing.assert_array_equal(p2[t, : nw[t]], ph[off[t]: off[t + 1]])
        assert (p2[t, nw[t]:] == 7.0).all()
    _check(ph, eh, packed, off, True, PENALTIES["default"])


def test_c4_full_size():
    """10,000 tables x 10,000 bins of log-likelihoods with planted segments (as test_c4_full_size_spot_checks_against_oracle):
    first, middle and last table against the oracle; row sums and expected counts over the whole batch; the posterior
    arg-max recovers the planted segments about as often as the Viterbi states.  (The penalties are weights, not the
    process that planted the segments, so neither decoding is guaranteed to be the better one: on a B200 the posterior
    arg-max recovered 0.76124 of the bins, the Viterbi path 0.76152.)"""
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
    seg_h = seg.to(torch.uint8).cpu().numpy()
    h_ll = ll.cpu().numpy()
    del ll, seg
    torch.cuda.empty_cache()
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    with ib.Engine(ib.Params()) as e:
        post, expected = e.posterior_batch(h_ll, off, True)
        state, _, _ = e.viterbi_batch(h_ll, off, True)
    for t in (0, n_tables // 2, n_tables - 1):
        sl = slice(t * n_bins, (t + 1) * n_bins)
        want_p, want_e = posterior_oracle(h_ll[sl], [0, n_bins], True)
        np.testing.assert_allclose(post[sl], want_p, rtol=0, atol=1e-9)
        np.testing.assert_allclose(expected[t], want_e[0], rtol=0, atol=1e-6)
    p = torch.from_numpy(post)
    assert bool(torch.isfinite(p).all())
    assert float((p.sum(dim=1) - 1.0).abs().max()) <= 1e-12
    colsum = p.view(n_tables, n_bins, 3).sum(dim=1).numpy()
    np.testing.assert_allclose(expected, colsum, rtol=0, atol=1e-9 * n_bins)
    rec_post = float((p.argmax(dim=1).numpy().astype(np.uint8) == seg_h).mean())
    rec_vit = float((state == seg_h).mean())
    assert rec_post >= rec_vit - 1e-3 and rec_post > 0.75, (rec_post, rec_vit)


# ---- command lines ----------------------------------------------------------------------------------------------
def _run(binary, args, cwd=None):
    r = subprocess.run([os.path.join(hostlib.BIN, binary)] + args, capture_output=True, text=True, cwd=cwd, timeout=300)
    assert r.returncode == 0, r.stderr
    return r


def _summary_lik(path):
    """LIBD0/1/2 of a summary file, parsed as hiddengem parses it (leading '#' lines skipped)."""
    rows = []
    with open(path) as fh:
        for ln in fh:
            if ln.startswith("#") and not rows:
                continue
            f = ln.split("\t")
            if len(f) >= 7:
                rows.append([float(f[3]), float(f[4]), float(f[5])])
    return np.array(rows)


def _check_posterior_text(got, plain, want_p, want_e, tol):
    """got: output with --posterior; plain: the same run without it.  The first five columns and the "#% IBDk" lines
    are unchanged; the new columns and lines follow the oracle."""
    g, p = got.splitlines(), plain.splitlines()
    assert g[0] == p[0] + "\tP_IBD0\tP_IBD1\tP_IBD2"
    rows = [ln for ln in g[1:] if not ln.startswith("#")]
    prow = [ln for ln in p[1:] if not ln.startswith("#")]
    assert len(rows) == len(prow) == len(want_p)
    printed = np.array([[float(x) for x in r.split("\t")[5:8]] for r in rows])
    for a, b in zip(rows, prow):
        assert "\t".join(a.split("\t")[:5]) == b
    np.testing.assert_allclose(printed, want_p, rtol=0, atol=tol)
    gc = [ln for ln in g if ln.startswith("#")]
    assert gc[:3] == [ln for ln in p if ln.startswith("#")]
    n = len(want_p)
    for k in range(3):
        head, val = gc[3 + k].split(": ")
        assert head.startswith(f"#% posterior IBD{k} (n = ")
        assert abs(float(head.split("= ")[1].rstrip(")")) - want_e[k]) <= 0.005 + tol * n
        assert abs(float(val) - want_e[k] / n * 100) <= 0.005 + tol * 100


HG = [("nonld_w10", "ind2", "default", []), ("nonld_w10", "ind3", "default", []), ("nonld_w10", "ind5", "default", []),
      ("nonld_w10", "ind3", "loose", ["--p01", "0.2", "--p02", "0.05", "--p12", "0.3"]),
      ("ld_w100_underflow", "ind3", "ld_underflow", [])]


@pytest.mark.parametrize("run,ind,tag,args", HG)
def test_hiddengem_posterior_command_line(golden_dir, run, ind, tag, args):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    summ = os.path.join(ca, run, f"UNKWN.{ind}.summary.txt")
    plain = _run("hiddengem", ["-s", summ] + args).stdout
    got = _run("hiddengem", ["-s", summ, "--posterior"] + args).stdout
    # Inferred_State and the state counts are the reference's (golden stdout)
    want = open(os.path.join(ca, "hiddengem", f"{ind}.{tag}.txt")).read().splitlines()
    assert [r.split("\t")[4] for r in plain.splitlines()[1:] if not r.startswith("#")] == \
           [r.split("\t")[4] for r in want[1:] if not r.startswith("#")]
    assert [r for r in plain.splitlines() if r.startswith("#")] == [r for r in want if r.startswith("#")]
    pen = [float(a) for a in args[1::2]] or [1e-3, 1e-6, 1e-3]
    lik = _summary_lik(summ)
    want_p, want_e = posterior_oracle(lik, [0, len(lik)], False, *pen)
    _check_posterior_text(got, plain, want_p, want_e[0], 1e-6)


def test_ibdgem_hiddengem_posterior_files(golden_dir, tmp_path):
    hostlib.build()
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, "nonld_w10", "ARGS.json")))
    base = ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup"] + meta["args"] + ["--hiddengem", "--no-tab"]
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    _run("ibdgem", base + ["-O", str(tmp_path / "a")], cwd=ca)
    _run("ibdgem", base + ["-O", str(tmp_path / "b"), "--posterior"], cwd=ca)
    for ind in ("ind2", "ind3", "ind5"):
        plain = open(tmp_path / "a" / f"UNKWN.{ind}.hiddengem.txt").read()
        got = open(tmp_path / "b" / f"UNKWN.{ind}.hiddengem.txt").read()
        # the run's own window scores, as printed to its summary file (7 significant digits)
        lik = _summary_lik(tmp_path / "b" / f"UNKWN.{ind}.summary.txt")
        with np.errstate(divide="ignore"):
            want_p, want_e = posterior_oracle(np.log(lik), [0, len(lik)], True)
        _check_posterior_text(got, plain, want_p, want_e[0], 2e-5)
