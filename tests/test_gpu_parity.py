"""GPU parity tests proper: the CUDA engine, called through the C ABI, against (a) the
reference's golden text tables and (b) the pinned oracle on the same inputs.
Bar (BASELINE.json north_star): integer outputs bit-exact; per-site |dLL| <= 1e-9|LL|;
per-window sums |d| <= 1e-6 absolute."""
import os

import numpy as np
import pytest

import refcases
import refio

pytestmark = pytest.mark.gpu


def _engine():
    import enginecase
    return enginecase


@pytest.mark.parametrize("k", [1, 2, 3])
def test_fixture_replay_tables_byte_exact(fixture_dir, k):
    """The 18 golden files of supplementary/ibdgem-test/output, regenerated from engine output."""
    ec = _engine()
    inp = os.path.join(fixture_dir, "input")
    case = refcases.load_case(inp, "", hap="test.hap", legend="test.legend", indv="test.indv",
                              pileup=f"test{k}.pileup", args=[], pileup_name=f"sample{k}")
    case.out_dir = os.path.join(fixture_dir, "output")
    results = ec.run_engine(case)
    oracle_res = refcases.oracle_run(case)
    for t, res, ora in zip(case.targets, results, oracle_res):
        tab, summ = refcases.golden_texts(case, t)
        assert refio.format_tab(case.pk, res, t, 20) == tab
        assert refio.format_summary(res) == summ
        ec.assert_matches_oracle(res, ora)


@pytest.mark.parametrize("run", refcases.ALL_RUNS)
def test_reference_runs(golden_dir, run):
    """--LD, -v, -D, -B, -S/-s, -A, -p, -F/-f, -M, -e, -N-in-panel against reference outputs."""
    ec = _engine()
    case = refcases.load_case(os.path.join(golden_dir, "ref_runs", "caseA"), run)
    results = ec.run_engine(case)
    oracle_res = refcases.oracle_run(case)
    for t, res, ora in zip(case.targets, results, oracle_res):
        ec.assert_matches_oracle(res, ora)
        tab, summ = refcases.golden_texts(case, t)
        assert refio.format_tab(case.pk, res, t, case.params.max_cov, case.params.cull_p) == tab
        # summary text: identical wherever the printed 7 significant digits are stable; compare
        # the integer columns exactly and the likelihood columns numerically
        got = refio.format_summary(res).splitlines()
        want = summ.splitlines()
        assert len(got) == len(want)
        for g, w in zip(got[1:], want[1:]):
            gf, wf = g.split("\t"), w.split("\t")
            assert gf[:3] == wf[:3] and gf[6] == wf[6]
            for a, b in zip(gf[3:6], wf[3:6]):
                if "nan" in b:
                    assert "nan" in a
                else:
                    assert float(a) == pytest.approx(float(b), rel=2e-6, abs=1e-300)


@pytest.mark.parametrize("k", [1, 2])
def test_fixture_ld_against_reference(golden_dir, fixture_dir, k):
    ec = _engine()
    inp = os.path.join(fixture_dir, "input")
    case = refcases.load_case(inp, "", hap="test.hap", legend="test.legend", indv="test.indv",
                              pileup=f"test{k}.pileup", args=["--LD", "-w", "10"], pileup_name=f"sample{k}")
    for res, ora in zip(ec.run_engine(case), refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def _synth_case(seed, S, N, window, ld, targets, bg=None, pu_idx=-1, opt_v=0, depth=2.0, eps=0.02,
                max_cov=20, cull_p=1.0):
    import oracle
    rng = np.random.default_rng(seed)
    af = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99)
    hap = (rng.random((S, 2 * N)) < af[:, None]).astype(np.uint8)
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = rng.poisson(depth, S)
    g = hap[:, 0] + hap[:, 1]
    n_alt = rng.binomial(d, np.where(g == 0, eps, np.where(g == 1, 0.5, 1 - eps)))
    n_ref = d - n_alt
    keep = (rng.random(S) > 0.03).astype(np.uint8)
    pk = refio.Packed([f"i{i}" for i in range(N)], hap, pos, keep, n_ref.astype(np.uint8),
                      n_alt.astype(np.uint8), d.astype(np.uint32), ["1"] * S, ["."] * S, ["A"] * S,
                      ["G"] * S, None)
    prm = oracle.Params(epsilon=eps, max_cov=max_cov, window=window, ld_mode=int(ld), opt_v=opt_v, pu_idx=pu_idx,
                        cull_p=cull_p)
    return refcases.Case(pk, prm, list(targets), np.asarray(bg if bg is not None else range(N), np.int32),
                         None, "UNKWN", "")


@pytest.mark.parametrize("force_general", [True, False])
@pytest.mark.parametrize("window,S,N,T", [(100, 3000, 40, 5), (1000, 6100, 70, 9), (37, 1500, 33, 33)])
def test_ld_synthetic_vs_oracle(window, S, N, T, force_general):
    """Windows long enough that the reference's linear products underflow: log-space oracle."""
    ec = _engine()
    case = _synth_case(7 + window, S, N, window, True, range(T), pu_idx=2)
    results = ec.run_engine(case, force_general=force_general, expanded=False)
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)
    if not force_general:
        # the tensor path must be the one that ran for shared-window, depth-linear inputs
        assert results[0]["ld_path"] == 1


@pytest.mark.parametrize("eps", [0.001, 0.1, 0.3, 0.45])
def test_ld_other_error_rates_vs_oracle(eps):
    """The exp table of the ld_mma epilogue is sized from epsilon (kappa = ln 4 eps (1 - eps)): a dozen entries of
    reach at 0.001, ~400 at 0.3, and at 0.45 (kappa = -0.01) the screen's reach does not fit the table and the
    exp-based candidate path runs.  With the reads' source in the background (peaked rows) and without it (flat rows:
    many columns within the screen's reach of the row maximum)."""
    ec = _engine()
    N = 40
    for seed, bg, pu_idx in ((31, None, 2), (32, list(range(1, N)), -1)):
        case = _synth_case(seed, 3000, N, 100, True, range(7), bg=bg, pu_idx=pu_idx, eps=eps)
        results = ec.run_engine(case, expanded=False)
        assert results[0]["ld_path"] == 1
        for res, ora in zip(results, refcases.oracle_run(case)):
            ec.assert_matches_oracle(res, ora)


def test_ld_background_subsets_and_duplicates():
    ec = _engine()
    bg = [0, 3, 3, 5, 7, 8, 9, 11, 12, 20, 21, 22, 2]
    case = _synth_case(99, 2500, 24, 50, True, [2, 3, 20, 23], bg=bg, pu_idx=5)
    for fg in (True, False):
        for res, ora in zip(ec.run_engine(case, force_general=fg, expanded=False), refcases.oracle_run(case)):
            ec.assert_matches_oracle(res, ora)


def test_ld_empty_background_gives_nan():
    ec = _engine()
    case = _synth_case(5, 500, 6, 20, True, [1], bg=[1], pu_idx=-1)
    res = ec.run_engine(case, expanded=False)[0]
    assert np.isnan(res["w_log"][:, 0]).all() and np.isnan(res["w_log"][:, 1]).all()
    assert np.isfinite(res["w_log"][:, 2]).all()


def test_nonld_variable_sites_and_large_cov():
    ec = _engine()
    case = _synth_case(3, 4000, 20, 64, False, range(20), opt_v=1, depth=6.0, max_cov=30)
    for res, ora in zip(ec.run_engine(case), refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_nonld_window_properties_full_axis():
    """Size-independent properties on a 200k-site axis: window counts partition the informative
    sites, boundaries are sorted, and halving the window doubles-up exactly (sum of two
    half-windows == the full window)."""
    ec = _engine()
    S = 200_000
    case_a = _synth_case(11, S, 16, 100, False, range(4))
    case_b = _synth_case(11, S, 16, 50, False, range(4))
    ra = ec.run_engine(case_a, expanded=False)
    rb = ec.run_engine(case_b, expanded=False)
    for a, b in zip(ra, rb):
        inf = int((a["st_shared"] == 1).sum())
        assert int(a["w_nsites"].sum()) == inf == int(b["w_nsites"].sum())
        assert np.all(np.diff(a["w_start"].astype(np.int64)) > 0)
        assert np.all(a["w_end"] >= a["w_start"])
        assert a["n_windows"] == -(-inf // 100) and b["n_windows"] == -(-inf // 50)
        nb = b["n_windows"]
        pair = np.zeros((a["n_windows"], 3))
        for j in range(nb):
            pair[j // 2] += b["w_log"][j]
        np.testing.assert_allclose(pair, a["w_log"], rtol=0, atol=1e-8)
        assert a["processed"] + a["skipped"] == S


def test_hiddengem_vs_oracle_and_reference(golden_dir):
    import ibdgem_b200 as ib
    import oracle
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    tables, offs = [], [0]
    names = []
    for run, tg in (("nonld_w10", "ind2"), ("nonld_w10", "ind3"), ("nonld_w10", "ind5"),
                    ("ld_w100_underflow", "ind3"), ("nonld_v_w7", "ind1")):
        rows = refio.read_summary(os.path.join(ca, run, f"UNKWN.{tg}.summary.txt"))
        l = np.array([[r[2], r[3], r[4]] for r in rows])
        tables.append(l)
        offs.append(offs[-1] + len(l))
        names.append((run, tg))
    rng = np.random.default_rng(0)
    # long random tables with planted segments, zeros and an all-zero (NaN) row
    for n in (1000, 4097):
        seg = np.repeat(rng.integers(0, 3, n // 50 + 1), 50)[:n]
        l = np.exp(rng.normal(-20, 3, (n, 3)))
        l[np.arange(n), seg] *= np.exp(6.0)
        l[5, 1] = 0.0
        if n == 4097:
            l[100] = 0.0
        tables.append(l)
        offs.append(offs[-1] + n)
    lik = np.concatenate(tables)
    for pen in ((1e-3, 1e-6, 1e-3), (0.2, 0.05, 0.3), (2.0, 0.5, 4.0)):
        with ib.Engine(ib.Params()) as e:
            state, score, counts = e.viterbi_batch(lik, offs, False, *pen)
        for i, l in enumerate(tables):
            st, sc, _ = oracle.hiddengem(l, *pen)
            a, b = offs[i], offs[i + 1]
            np.testing.assert_array_equal(state[a:b], st)  # Inferred_State: bit-exact
            np.testing.assert_array_equal(counts[i], np.bincount(st, minlength=3))
            fin = np.isfinite(sc)
            np.testing.assert_array_equal(np.isnan(score[a:b]), np.isnan(sc))
            np.testing.assert_allclose(score[a:b][fin], sc[fin], rtol=0, atol=1e-7)


def test_hiddengem_log_front_end_matches_oracle():
    """is_log = 1 (the engine's own window scores, natural logs) against the ORACLE run on the same
    likelihoods in linear space — not against the CUDA text path."""
    import ibdgem_b200 as ib
    import oracle
    rng = np.random.default_rng(4)
    n = 2000
    ll = rng.normal(-300, 40, (n, 3))  # exp() stays a normal double (> -708), so the oracle can take it
    seg = np.repeat(rng.integers(0, 3, n // 50 + 1), 50)[:n]
    ll[np.arange(n), seg] += 6.0
    with ib.Engine(ib.Params()) as e:
        s_log, sc_log, cnt = e.viterbi_batch(ll, [0, n], True)
    st, sc, _ = oracle.hiddengem(np.exp(ll))
    np.testing.assert_array_equal(s_log, st)
    np.testing.assert_array_equal(cnt[0], np.bincount(st, minlength=3))
    np.testing.assert_allclose(sc_log, sc, rtol=0, atol=1e-7)


def test_c3_full_size_spot_checks_against_oracle():
    """BASELINE.json configs[2] at full size (1,000,000 sites x 2,504 samples x 1,000 targets, window
    1,000): windows are independent, so any window of any target can be re-scored by the CPU oracle
    from that window's slice of the inputs.  Nine (target, window) cells, all three likelihoods, plus
    size-independent integer properties of the whole table."""
    import torch
    import ibdgem_b200 as ib
    import oracle
    from ibdgem_b200.synth import synth_panel_torch, unpack_rows
    S, N, T, W = 1_000_000, 2504, 1000, 1000
    d = synth_panel_torch(S, N, seed=1, device="cuda")
    bits = d["bits"].numpy().view(np.uint32)
    pos = d["pos"].numpy().view(np.uint64)
    n_ref, n_alt, keep = d["n_ref"].numpy(), d["n_alt"].numpy(), d["keep"].numpy()
    targets = np.arange(T, dtype=np.int32)
    bg = np.arange(N, dtype=np.int32)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, keep)
        e.upload_panel(bits, N)
        sc = e.score_ld(targets, bg, -1)  # panel chunks still in flight: ranges of windows, streamed results
        assert e.last_ld_path() == 1  # the tensor-core path is the one that ran
        sc2 = e.score_ld(targets, bg, -1)  # panel resident: one range, one result copy
    for a, b in ((sc.w_start, sc2.w_start), (sc.w_end, sc2.w_end), (sc.w_nsites, sc2.w_nsites),
                 (sc.n_windows, sc2.n_windows)):
        np.testing.assert_array_equal(a, b)
    # the order in which a row's tiles reach the fp64 log-sum-exp follows the dynamic unit schedule:
    # the two runs may differ in the last bits (NaN == NaN here: the unused trailing columns)
    np.testing.assert_allclose(sc.w_loglik, sc2.w_loglik, rtol=0, atol=1e-9, equal_nan=True)
    nW = S // W
    assert (sc.n_windows == nW).all()
    assert (sc.w_nsites[:, :nW] == W).all() and int(sc.processed[0]) == S and int(sc.skipped[0]) == 0
    np.testing.assert_array_equal(sc.w_start[0, :nW], pos[0::W])
    np.testing.assert_array_equal(sc.w_end[0, :nW], pos[W - 1::W])
    assert np.isfinite(sc.w_loglik[:, :nW]).all()
    # LIBD0 of a window is a mean over the background minus the target.  The reads were drawn from
    # individual 0, whose term dominates every window: all targets but 0 see (nearly) the same LIBD0,
    # and target 0 — whose own entry is omitted — sees a far smaller one.
    l0 = sc.w_loglik[:, :nW, 0]
    assert np.ptp(l0[1:], axis=0).max() < 1e-3
    assert (l0[0] < l0[1] - 100.0).all()
    prm = oracle.Params(window=W, ld_mode=1)
    for w in (0, 417, nW - 1):
        sl = slice(w * W, (w + 1) * W)
        hap = unpack_rows(bits, 2 * N, np.arange(w * W, (w + 1) * W))
        for t in (0, 333, T - 1):
            o = oracle.compare_target(prm, pos[sl], keep[sl], n_ref[sl], n_alt[sl], hap, int(t), bg)
            assert o["n_windows"] == 1
            np.testing.assert_allclose(sc.w_loglik[t, w], o["w_log"][0], rtol=0, atol=1e-6)


@pytest.mark.parametrize("ragged", [False, True])
def test_hiddengem_batched_pipeline_vs_oracle(ragged):
    """>= 64 tables of similar lengths take the batched path (viterbi_fused_kernel, back-trace, state transpose);
    states must be bit-exact and scores within 1e-7 of the per-table oracle, for equal-length and ragged batches,
    with zero and all-zero (NaN) rows, at penalties below 1 and at penalties above 1 that reward a switch."""
    import ibdgem_b200 as ib
    import oracle
    rng = np.random.default_rng(12)
    n_tables = 96
    lens = rng.integers(700, 1000, n_tables) if ragged else np.full(n_tables, 777)
    tables, offs = [], [0]
    for k, n in enumerate(lens):
        seg = np.repeat(rng.integers(0, 3, n // 40 + 1), 40)[:n]
        l = np.exp(rng.normal(-20, 3, (n, 3)))
        l[np.arange(n), seg] *= np.exp(5.0)
        if k % 7 == 0:
            l[3, 2] = 0.0
        if k % 11 == 0:
            l[n // 2] = 0.0
        tables.append(l)
        offs.append(offs[-1] + int(n))
    lik = np.concatenate(tables)
    for pen in ((1e-3, 1e-6, 1e-3), (0.2, 0.05, 0.3), (2.0, 0.5, 4.0)):
        with ib.Engine(ib.Params()) as e:
            state, score, counts = e.viterbi_batch(lik, offs, False, *pen)
            stats = e.kernel_stats()
        assert stats["viterbi_back"][1] > 0  # the batched kernels are the ones that ran
        for i, l in enumerate(tables):
            st, sc, _ = oracle.hiddengem(l, *pen)
            a, b = offs[i], offs[i + 1]
            np.testing.assert_array_equal(state[a:b], st)
            np.testing.assert_array_equal(counts[i], np.bincount(st, minlength=3))
            fin = np.isfinite(sc)
            np.testing.assert_array_equal(np.isnan(score[a:b]), np.isnan(sc))
            np.testing.assert_allclose(score[a:b][fin], sc[fin], rtol=0, atol=1e-7)


def test_ld_disjoint_background_many_targets_c5_shape():
    """BASELINE.json configs[4] in miniature: targets and background are disjoint sets (-S / -B), more
    target rows than one row block pair holds, several column tiles."""
    ec = _engine()
    N = 700
    case = _synth_case(21, 6000, N, 500, True, range(0, 300), bg=list(range(300, N)))
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 1
    import oracle
    for k in (0, 1, 149, 299):  # the oracle is slow: four of the 300 targets
        o = oracle.compare_target(case.params, case.pk.pos, case.pk.host_keep, case.pk.n_ref, case.pk.n_alt, case.pk.hap,
                                  case.targets[k], case.bg, af_user=case.af_user, reseed=True)
        ec.assert_matches_oracle(results[k], o)


def test_ld_window_batching_under_a_small_operand_budget():
    """The int8 operands of all windows do not fit the budget: windows go through in batches."""
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, 'tests'); sys.path.insert(0, '.')\n"
        "import numpy as np, enginecase as ec, refcases\n"
        "from test_gpu_parity import _synth_case\n"
        "case = _synth_case(33, 12000, 80, 400, True, range(12), pu_idx=3)\n"
        "res = ec.run_engine(case, expanded=False)\n"
        "assert res[0]['ld_path'] == 1 and res[0]['kernel_stats']['ld_mma'][1] >= 3, res[0]['kernel_stats']['ld_mma']\n"
        "for r, o in zip(res, refcases.oracle_run(case)): ec.assert_matches_oracle(r, o)\n"
        "print('ok')\n")
    env = dict(os.environ, IBDGEM_LD_BUDGET_MB="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))), timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_ld_deep_pileup_large_max_cov():
    """Depths well above the default: the int8 target operand carries n_s up to max_cov (unsigned),
    the dp4a marginals sum count bytes above 31, and kappa * M spans thousands of nats."""
    ec = _engine()
    case = _synth_case(71, 5000, 48, 300, True, range(10), pu_idx=4, depth=14.0, max_cov=60)
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 1
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_ld_window_larger_than_tensor_tile_uses_general_path():
    """Windows above 1,024 sites do not fit the resident target tile: the general path takes over."""
    ec = _engine()
    case = _synth_case(72, 5000, 24, 1500, True, range(4))
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 0
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


@pytest.mark.parametrize("ld", [True, False])
def test_panel_rows_not_16_byte_aligned(ld):
    """words_per_site is the caller's choice (include/ibdgem_b200.h): 3 words per row here, so no
    kernel may assume 16-byte-aligned panel rows."""
    ec = _engine()
    case = _synth_case(73, 3000, 40, 100, ld, range(6), pu_idx=1)
    for fg in ((True, False) if ld else (False,)):
        results = ec.run_engine(case, force_general=fg, expanded=False, align_words=1)
        for res, ora in zip(results, refcases.oracle_run(case)):
            ec.assert_matches_oracle(res, ora)


def test_panel_in_caller_device_memory_declared_in_pieces():
    """ibdgem_engine_set_panel_device / _panel_rows_ready (the NVLink replication path of
    shard.replicate_panel, here on one GPU): same scores as ibdgem_engine_upload_panel; rows that were
    never declared ready are an error, not a read of unwritten memory."""
    import torch
    import ibdgem_b200 as ib
    from ibdgem_b200.shard import panel_pieces, replicate_panel
    ec = _engine()
    case = _synth_case(74, 6000, 40, 100, True, range(7), pu_idx=3)
    pk = case.pk
    want = ec.run_engine(case, expanded=False)
    bits = ib.pack_bits(pk.hap)
    h_bits = torch.from_numpy(bits.view(np.int32)).pin_memory()
    S, Wh = bits.shape
    with ib.Engine(ib.Params(window_size=100)) as e:
        e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
        for pieces in (1, 3):
            per, padded = panel_pieces(S, 1, pieces)
            d_panel = torch.empty((padded, Wh), dtype=torch.int32, device="cuda")
            side = torch.cuda.Stream()
            replicate_panel(e, h_bits, d_panel, len(pk.names), pieces=pieces, stream=side)
            sc = e.score_ld(case.targets, case.bg, 3)
            for k, w in enumerate(want):
                nw = w["n_windows"]
                assert int(sc.n_windows[k]) == nw
                np.testing.assert_allclose(sc.w_loglik[k, :nw], w["w_log"], rtol=0, atol=1e-9)
                np.testing.assert_array_equal(sc.w_nsites[k, :nw], w["w_nsites"])
        d_panel = torch.from_numpy(bits.view(np.int32)).cuda()
        e.set_panel_device(d_panel.data_ptr(), S, len(pk.names), Wh)
        e.panel_rows_ready(S // 2)
        with pytest.raises(RuntimeError, match="declared ready"):
            e.score_ld(case.targets, case.bg, 3)


def test_ld_more_windows_than_a_grid_dimension():
    """70,000 windows of ten sites: the window index rides on gridDim.y (limit 65,535) in the
    transposition and expansion kernels, so such calls are sliced."""
    ec = _engine()
    case = _synth_case(75, 760_000, 6, 10, True, range(2), pu_idx=-1, depth=3.0)
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 1 and results[0]["n_windows"] > 65535
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_variable_sites_scored_while_the_pinned_panel_is_still_arriving():
    """-v ranks sites by the target's genotype, so the per-target window map reads panel rows.  With a
    page-locked panel the upload is asynchronous and chunked (>= 2 chunks of 16 MB here); the first
    score call right after it must wait for the rows before it builds the map (ADVICE r01)."""
    import torch
    import ibdgem_b200 as ib
    import oracle
    rng = np.random.default_rng(5)
    S, N, W = 60_000, 2504, 100
    af = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99).astype(np.float32)
    hap = (rng.random((S, 2 * N), dtype=np.float32) < af[:, None]).astype(np.uint8)
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = rng.poisson(2.0, S)
    n_alt = rng.binomial(d, 0.3).astype(np.uint8)
    n_ref = (d - n_alt).astype(np.uint8)
    keep = np.ones(S, np.uint8)
    bits = torch.from_numpy(ib.pack_bits(hap).view(np.int32)).pin_memory()
    assert bits.numel() * 4 >= 2 * (16 << 20)
    targets = np.array([0, 7, 2503], np.int32)
    prm = oracle.Params(window=W, opt_v=1)
    for _ in range(2):  # a fresh engine each time: nothing is resident when the score call is issued
        with ib.Engine(ib.Params(window_size=W, variable_sites_only=1)) as e:
            e.upload_sites(pos, n_ref, n_alt, keep)
            e.upload_panel(bits.numpy().view(np.uint32), N)
            sc = e.score_nonld(targets)
        for k, t in enumerate(targets):
            o = oracle.compare_target(prm, pos, keep, n_ref, n_alt, hap, int(t), np.arange(N, dtype=np.int32))
            nw = o["n_windows"]
            assert int(sc.n_windows[k]) == nw
            np.testing.assert_array_equal(sc.w_start[k, :nw], o["w_start"])
            np.testing.assert_array_equal(sc.w_end[k, :nw], o["w_end"])
            np.testing.assert_array_equal(sc.w_nsites[k, :nw], o["w_nsites"])
            assert int(sc.processed[k]) == o["processed"] and int(sc.skipped[k]) == o["skipped"]
            np.testing.assert_allclose(sc.w_loglik[k, :nw], o["w_log"], rtol=0, atol=1e-6)


def test_window_shards_reassemble_the_unsharded_table():
    """Multi-GPU partition by windows, emulated on one GPU: each of 3 shards scores its own windows of every
    target, reads only its own panel rows (the others hold garbage in the device buffer), and writes its
    columns of a shared device table (ibdgem_scores.w_loglik_device).  The union is the unsharded result."""
    import torch
    import ibdgem_b200 as ib
    from ibdgem_b200.shard import upload_window_shard_rows
    ec = _engine()
    case = _synth_case(81, 9000, 40, 100, True, range(7), pu_idx=3)
    pk = case.pk
    want = ec.run_engine(case, expanded=False)
    bits = ib.pack_bits(pk.hap)
    h_bits = torch.from_numpy(bits.view(np.int32)).pin_memory()
    S, Wh = bits.shape
    T = len(case.targets)
    count = 3
    maxW = S // 100 + 2
    d_table = torch.full((T, maxW, 3), float("nan"), dtype=torch.float64, device="cuda")
    merged = np.full((T, maxW, 3), np.nan)
    covered = []
    with ib.Engine(ib.Params(window_size=100)) as e:
        for idx in range(count):
            e.set_window_shard(idx, count)
            e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
            d_panel = torch.full((S, Wh), -1, dtype=torch.int32, device="cuda")  # rows outside the shard: all ones
            nbytes = upload_window_shard_rows(e, h_bits, d_panel, len(pk.names))
            wb, we, sb, se = e.window_shard()
            assert nbytes == (se - sb) * Wh * 4 and 0 <= sb < se <= S
            covered.append((wb, we, sb, se))
            sc = e.score_ld(case.targets, case.bg, 3, max_windows=maxW, device_out=d_table.data_ptr())
            assert e.last_ld_path() == 1
            got = sc.w_loglik
            assert np.isnan(got[:, :wb]).all() and np.isnan(got[:, we:]).all()  # only the shard's columns are written
            merged[:, wb:we] = got[:, wb:we]
            for k, w in enumerate(want):
                assert int(sc.n_windows[k]) == w["n_windows"]
                np.testing.assert_array_equal(sc.w_nsites[k, :w["n_windows"]], w["w_nsites"])
                np.testing.assert_array_equal(sc.w_start[k, :w["n_windows"]], w["w_start"])
        # compact, window-major host table of a shard: [we - wb][T][3], the same numbers
        e.set_shard_compact_output(True)
        wb, we, _, _ = e.window_shard()
        scc = e.score_ld(case.targets, case.bg, 3, max_windows=maxW)
        compact = scc.w_loglik.reshape(-1)[: T * (we - wb) * 3].reshape(we - wb, T, 3).transpose(1, 0, 2)
        np.testing.assert_array_equal(compact, merged[:, wb:we])
        e.set_shard_compact_output(False)
        # non-tensor paths refuse a window shard instead of silently scoring everything
        with pytest.raises(RuntimeError, match="window shard"):
            e.score_nonld(case.targets)
    # shards tile the windows and the panel rows exactly
    assert covered[0][0] == 0 and covered[0][2] == 0 and covered[-1][3] == S
    for a, b in zip(covered, covered[1:]):
        assert a[1] == b[0] and a[3] == b[2]
    table = d_table.cpu().numpy()
    for k, w in enumerate(want):
        nw = w["n_windows"]
        assert covered[-1][1] == nw
        np.testing.assert_allclose(merged[k, :nw], w["w_log"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(table[k, :nw], w["w_log"], rtol=0, atol=1e-9)


def test_window_shard_without_windows_still_reports_the_bookkeeping():
    """More shards than windows: a rank whose shard is empty scores nothing, writes no score column, and still reports
    the window bookkeeping (the same on every rank)."""
    import ibdgem_b200 as ib
    ec = _engine()
    case = _synth_case(85, 250, 20, 100, True, range(5), pu_idx=3)
    pk = case.pk
    want = ec.run_engine(case, expanded=False)
    nW = want[0]["n_windows"]
    count = nW + 3
    seen = np.zeros(nW, bool)
    with ib.Engine(ib.Params(window_size=100)) as e:
        for idx in range(count):
            e.set_window_shard(idx, count)
            e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
            e.upload_panel(ib.pack_bits(pk.hap), len(pk.names))
            wb, we, _, _ = e.window_shard()
            sc = e.score_ld(case.targets, case.bg, 3, max_windows=nW + 2)
            for k, w in enumerate(want):
                assert int(sc.n_windows[k]) == nW
                np.testing.assert_array_equal(sc.w_nsites[k, :nW], w["w_nsites"])
                np.testing.assert_array_equal(sc.w_start[k, :nW], w["w_start"])
                np.testing.assert_array_equal(sc.w_end[k, :nW], w["w_end"])
                assert np.isnan(sc.w_loglik[k, :wb]).all() and np.isnan(sc.w_loglik[k, we:]).all()
                np.testing.assert_allclose(sc.w_loglik[k, wb:we], w["w_log"][wb:we], rtol=0, atol=1e-9)
            assert not seen[wb:we].any()
            seen[wb:we] = True
    assert seen.all()


# ---- per-target windows on the tensor cores (-v, -D): ld_vmma.cu, ld_path == 2 ------------------
@pytest.mark.parametrize("window,S,N,T", [(10, 2500, 30, 7), (100, 9000, 40, 33), (1000, 30000, 100, 70), (37, 4000, 170, 90)])
def test_ld_variable_sites_tensor_path_vs_oracle(window, S, N, T):
    """-v --LD: every target has its own windows; rows of the GEMM are (target, window) pairs.  Shapes cover
    one and several row tiles (64 pairs each), one to three column tiles (80 individuals each), hulls of one
    and of many k-blocks, and windows shorter than a 32-slot word."""
    ec = _engine()
    case = _synth_case(100 + window, S, N, window, True, range(T), pu_idx=2, opt_v=1)
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 2
    assert results[0]["kernel_stats"]["ld_vmma"][1] >= 1
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_ld_variable_sites_general_path_still_matches():
    ec = _engine()
    case = _synth_case(141, 3000, 30, 50, True, range(6), pu_idx=2, opt_v=1)
    results = ec.run_engine(case, force_general=True, expanded=False)
    assert results[0]["ld_path"] == 0
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


@pytest.mark.parametrize("opt_v", [0, 1])
def test_ld_downsampled_counts_tensor_path_vs_oracle(opt_v):
    """-D (with and without -v): per-target thinned counts, drawn with glibc rand() in the reference's order;
    windows, row operands and the class sums all follow the target's own counts."""
    ec = _engine()
    case = _synth_case(150 + opt_v, 2500, 90, 40, True, range(9), pu_idx=1, opt_v=opt_v, depth=5.0, cull_p=0.5)
    results = ec.run_engine(case, expanded=True)
    assert results[0]["ld_path"] == 2
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_ld_variable_sites_background_subsets_duplicates_and_disjoint_targets():
    ec = _engine()
    bg = [0, 3, 3, 5, 7, 8, 9, 11, 12, 20, 21, 22, 2] + list(range(30, 130))
    case = _synth_case(160, 6000, 140, 120, True, [2, 3, 20, 23, 135, 139], bg=bg, pu_idx=5, opt_v=1)
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 2
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)


def test_ld_variable_sites_row_tiles_in_batches_under_a_small_budget():
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, 'tests'); sys.path.insert(0, '.')\n"
        "import numpy as np, enginecase as ec, refcases\n"
        "from test_gpu_parity import _synth_case\n"
        "case = _synth_case(170, 20000, 60, 100, True, range(40), pu_idx=3, opt_v=1)\n"
        "res = ec.run_engine(case, expanded=False)\n"
        "assert res[0]['ld_path'] == 2 and res[0]['kernel_stats']['ld_vmma'][1] >= 3, res[0]['kernel_stats']['ld_vmma']\n"
        "for r, o in zip(res, refcases.oracle_run(case)): ec.assert_matches_oracle(r, o)\n"
        "print('ok')\n")
    env = dict(os.environ, IBDGEM_V_BUDGET_MB="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))), timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_c3_variable_sites_full_size_spot_checks_against_oracle():
    """C3 with -v at full size (1,000,000 sites x 2,504 samples x 1,000 targets, window 1,000 VARIABLE sites):
    a window of a target depends only on the sites between its first and last member, so any (target, window)
    cell can be re-scored by the CPU oracle from that slice of the inputs."""
    import torch
    import ibdgem_b200 as ib
    import oracle
    from ibdgem_b200.synth import synth_panel_torch, unpack_rows
    S, N, T, W = 1_000_000, 2504, 1000, 1000
    d = synth_panel_torch(S, N, seed=1, device="cuda")
    bits = d["bits"].numpy().view(np.uint32)
    pos = d["pos"].numpy().view(np.uint64)
    n_ref, n_alt, keep = d["n_ref"].numpy(), d["n_alt"].numpy(), d["keep"].numpy()
    targets = np.arange(T, dtype=np.int32)
    bg = np.arange(N, dtype=np.int32)
    with ib.Engine(ib.Params(window_size=W, variable_sites_only=1)) as e:
        e.upload_sites(pos, n_ref, n_alt, keep)
        e.upload_panel(bits, N)
        sc = e.score_ld(targets, bg, -1)
        assert e.last_ld_path() == 2
    prm = oracle.Params(window=W, ld_mode=1, opt_v=1)
    for t in (0, 333, T - 1):
        nw = int(sc.n_windows[t])
        assert 250 < nw < 400
        assert int(sc.w_nsites[t, :nw - 1].min()) == W and np.all(np.diff(sc.w_start[t, :nw].astype(np.int64)) > 0)
        assert np.isfinite(sc.w_loglik[t, :nw]).all()
        for w in (0, nw // 2, nw - 1):
            s0 = int((int(sc.w_start[t, w]) - 1000) // 60)
            s1 = int((int(sc.w_end[t, w]) - 1000) // 60) + 1
            sl = slice(s0, s1)
            hap = unpack_rows(bits, 2 * N, np.arange(s0, s1))
            o = oracle.compare_target(prm, pos[sl], keep[sl], n_ref[sl], n_alt[sl], hap, int(t), bg)
            assert o["n_windows"] == 1 and int(o["w_nsites"][0]) == int(sc.w_nsites[t, w])
            np.testing.assert_allclose(sc.w_loglik[t, w], o["w_log"][0], rtol=0, atol=1e-6)


@pytest.mark.parametrize("n_tables", [5, 96])
def test_hiddengem_device_entry_matches_host_entry(n_tables):
    """hiddengem_viterbi_batch_device: packed tables, and tables at a fixed stride exactly as score_ld leaves them in
    ibdgem_scores.w_loglik_device ([T][max_windows][3] natural logs, rows past n_windows NaN)."""
    import torch
    import ibdgem_b200 as ib
    import oracle
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
        st_h, sc_h, cnt_h = e.viterbi_batch(ll, off, True)
        d_ll = torch.from_numpy(ll).cuda()
        d_state = torch.zeros(nb, dtype=torch.uint8, device="cuda")
        d_score = torch.zeros((nb, 3), dtype=torch.float64, device="cuda")
        d_cnt = torch.zeros((n_tables, 3), dtype=torch.int64, device="cuda")
        e.viterbi_batch_device(d_ll.data_ptr(), off, True, d_state.data_ptr(), d_score.data_ptr(), d_cnt.data_ptr())
        np.testing.assert_array_equal(d_state.cpu().numpy(), st_h)
        np.testing.assert_array_equal(d_cnt.cpu().numpy(), cnt_h)
        np.testing.assert_allclose(d_score.cpu().numpy(), sc_h, rtol=0, atol=1e-9)
        d_str = torch.from_numpy(strided).cuda()
        d_state2 = torch.full((n_tables, stride), 9, dtype=torch.uint8, device="cuda")
        d_score2 = torch.zeros((n_tables, stride, 3), dtype=torch.float64, device="cuda")
        d_cnt.zero_()
        e.viterbi_batch_device(d_str.data_ptr(), off, True, d_state2.data_ptr(), d_score2.data_ptr(), d_cnt.data_ptr(), table_stride=stride)
        s2 = d_state2.cpu().numpy()
        np.testing.assert_array_equal(d_cnt.cpu().numpy(), cnt_h)
        for t in range(n_tables):
            np.testing.assert_array_equal(s2[t, : lens[t]], st_h[off[t]: off[t + 1]])
            assert (s2[t, lens[t]:] == 9).all()  # nothing is written past a table's bins
    for t in (0, n_tables - 1):
        st, sc, _ = oracle.hiddengem(np.exp(ll[off[t]: off[t + 1]]))
        np.testing.assert_array_equal(st_h[off[t]: off[t + 1]], st)


def test_hiddengem_near_tie_guard_flags_and_matches_long_double():
    """Dyadic likelihoods and power-of-two penalties make exact ties in the reference's long double products; the
    device flags those tables and the host long double recurrence decides them (oracle: long double restatement)."""
    import ibdgem_b200 as ib
    import oracle
    rng = np.random.default_rng(41)
    vals = np.array([2.0 ** -k for k in range(4, 12)])
    tables, offs = [], [0]
    for n in [50] * 70 + [700]:
        tables.append(vals[rng.integers(0, len(vals), (n, 3))])
        offs.append(offs[-1] + n)
    lik = np.concatenate(tables)
    pen = (0.5, 0.25, 0.5)
    with ib.Engine(ib.Params()) as e:
        state, score, counts = e.viterbi_batch(lik, offs, False, *pen)
        assert e.viterbi_last_flagged() > 0
    for i, l in enumerate(tables):
        st, sc, _ = oracle.hiddengem(l, *pen)
        a, b = offs[i], offs[i + 1]
        np.testing.assert_array_equal(state[a:b], st)
        np.testing.assert_array_equal(counts[i], np.bincount(st, minlength=3))
        np.testing.assert_allclose(score[a:b], sc, rtol=0, atol=1e-7)


def test_panel_cloned_from_another_engine():
    """ibdgem_engine_clone_panel (what `ibdgem --gpus N` does for devices 1 .. N-1, here between two engines on one
    GPU): the clone follows the source's upload chunk by chunk and scores exactly like an engine that uploaded."""
    import torch
    import ibdgem_b200 as ib
    ec = _engine()
    case = _synth_case(91, 50_000, 300, 100, True, range(5), pu_idx=2)
    pk = case.pk
    want = ec.run_engine(case, expanded=False)
    bits = torch.from_numpy(ib.pack_bits(pk.hap).view(np.int32)).pin_memory()  # page-locked: the source's upload is asynchronous
    with ib.Engine(ib.Params(window_size=100)) as src, ib.Engine(ib.Params(window_size=100)) as dst:
        src.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
        src.upload_panel(bits.numpy().view(np.uint32), len(pk.names))
        dst.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
        dst.clone_panel(src)
        sc = dst.score_ld(case.targets, case.bg, 2)
        for k, w in enumerate(want):
            nw = w["n_windows"]
            assert int(sc.n_windows[k]) == nw
            np.testing.assert_allclose(sc.w_loglik[k, :nw], w["w_log"], rtol=0, atol=1e-9)
            np.testing.assert_array_equal(sc.w_nsites[k, :nw], w["w_nsites"])
    with ib.Engine(ib.Params(window_size=100)) as a, ib.Engine(ib.Params(window_size=100)) as b:
        with pytest.raises(RuntimeError, match="no panel"):
            b.clone_panel(a)


def test_ld_results_stored_straight_into_page_locked_host_memory():
    """With a page-locked w_loglik buffer the GEMM's merge warps store finished (LIBD0, LIBD1, LIBD2) triples into the
    caller's table themselves (no result copy after the kernel); the table must equal the one a pageable buffer
    receives by cudaMemcpy, NaN padding columns included."""
    import torch
    import ibdgem_b200 as ib
    from ibdgem_b200.engine import _CScores
    ec = _engine()
    case = _synth_case(95, 20_000, 320, 100, True, range(300), pu_idx=7)
    pk = case.pk
    T = len(case.targets)
    targets = np.asarray(case.targets, np.int32)
    with ib.Engine(ib.Params(window_size=100)) as e:
        e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)
        e.upload_panel(ib.pack_bits(pk.hap), len(pk.names))
        want = e.score_ld(targets, case.bg, 7)  # pageable numpy outputs
        assert e.last_ld_path() == 1
        maxW = want.w_loglik.shape[1]
        o_nw = torch.zeros(T, dtype=torch.int32).pin_memory()
        o_ll = torch.full((T, maxW, 3), -7.0, dtype=torch.float64).pin_memory()
        cs = _CScores(maxW, o_nw.data_ptr(), None, None, None, o_ll.data_ptr(), None, None, None, None, None, None, None, None)
        for _ in range(2):
            e.invalidate()
            e.score_ld_raw(targets, np.asarray(case.bg, np.int32), 7, cs)
    np.testing.assert_array_equal(o_nw.numpy(), want.n_windows)
    got = o_ll.numpy()
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want.w_loglik))
    np.testing.assert_allclose(np.nan_to_num(got), np.nan_to_num(want.w_loglik), rtol=0, atol=1e-9)


def test_ld_variable_sites_degenerate_targets():
    """-v edge cases on the tensor path: a target with no variable site at all (zero windows), one with fewer than a
    window's worth (a single partial window), a single-target call, and a call in which NO target has a variable site."""
    ec = _engine()
    case = _synth_case(181, 3000, 40, 50, True, [3, 5, 9, 11], pu_idx=1, opt_v=1)
    case.pk.hap[:, 6:8] = 0            # individual 3: hom-ref everywhere
    case.pk.hap[:, 10:12] = 0          # individual 5: variable at 7 sites only
    case.pk.hap[100:2000:300, 10] = 1
    results = ec.run_engine(case, expanded=False)
    assert results[0]["ld_path"] == 2
    assert results[0]["n_windows"] == 0 and results[1]["n_windows"] == 1
    for res, ora in zip(results, refcases.oracle_run(case)):
        ec.assert_matches_oracle(res, ora)
    one = _synth_case(182, 3000, 40, 50, True, [7], pu_idx=-1, opt_v=1)
    for res, ora in zip(ec.run_engine(one, expanded=False), refcases.oracle_run(one)):
        ec.assert_matches_oracle(res, ora)
    none = _synth_case(183, 800, 12, 20, True, [2, 4], pu_idx=-1, opt_v=1)
    none.pk.hap[:, 4:6] = 0
    none.pk.hap[:, 8:10] = 0
    for res, ora in zip(ec.run_engine(none, expanded=False), refcases.oracle_run(none)):
        assert res["n_windows"] == 0
        ec.assert_matches_oracle(res, ora)


def test_window_shard_in_sub_ranges_with_compact_output():
    """A window shard scored in three sub-ranges (as large shards are: the copy of one sub-range's columns runs under the
    next one's GEMM), compact window-major host table: same numbers as the unsharded run."""
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, 'tests'); sys.path.insert(0, '.')\n"
        "import numpy as np, ibdgem_b200 as ib, enginecase as ec\n"
        "from test_gpu_parity import _synth_case\n"
        "case = _synth_case(83, 9000, 40, 100, True, range(7), pu_idx=3)\n"
        "want = ec.run_engine(case, expanded=False)\n"
        "pk = case.pk; T = 7; maxW = 9000 // 100 + 2\n"
        "with ib.Engine(ib.Params(window_size=100)) as e:\n"
        "    e.set_window_shard(1, 2); e.set_shard_compact_output(True)\n"
        "    e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep, None)\n"
        "    e.upload_panel(ib.pack_bits(pk.hap), len(pk.names))\n"
        "    wb, we, _, _ = e.window_shard()\n"
        "    sc = e.score_ld(case.targets, case.bg, 3, max_windows=maxW)\n"
        "    assert e.kernel_stats()['ld_mma'][1] == 3, e.kernel_stats()['ld_mma']\n"
        "got = sc.w_loglik.reshape(-1)[: T * (we - wb) * 3].reshape(we - wb, T, 3).transpose(1, 0, 2)\n"
        "for k, w in enumerate(want):\n"
        "    np.testing.assert_allclose(got[k, : w['n_windows'] - wb], w['w_log'][wb:we], rtol=0, atol=1e-9)\n"
        "print('ok')\n")
    env = dict(os.environ, IBDGEM_SHARD_PARTS="-3")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))), timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_c2_full_size_spot_checks_against_oracle():
    """BASELINE.json configs[1] at full size (1,000,000 sites x 2,504 samples x 100 targets, window 100, depth
    Poisson(2): 13.5 % of the sites carry no read and belong to no window).  Windows are independent, so any window
    of any target can be re-scored by the CPU oracle from the window's own panel lines; plus the size-independent
    integer properties of the whole table."""
    import ibdgem_b200 as ib
    import oracle
    from ibdgem_b200.synth import synth_panel_torch, unpack_rows
    S, N, T, W = 1_000_000, 2504, 100, 100
    d = synth_panel_torch(S, N, seed=1, device="cuda")
    bits = d["bits"].numpy().view(np.uint32)
    pos = d["pos"].numpy().view(np.uint64)
    rng = np.random.default_rng(2)
    g = (bits[:, 0] & 1) + ((bits[:, 0] >> 1) & 1)  # genotype of individual 0, the source of the reads
    depth = np.minimum(rng.poisson(2.0, S), 20)
    n_alt = rng.binomial(depth, np.where(g == 0, 0.02, np.where(g == 1, 0.5, 0.98))).astype(np.uint8)
    n_ref = (depth - n_alt).astype(np.uint8)
    keep = np.ones(S, np.uint8)
    targets = np.arange(T, dtype=np.int32)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, keep)
        e.upload_panel(bits, N)
        sc = e.score_nonld(targets)
        assert e.kernel_stats()["window_nonld"][1] >= 1
    idx = np.flatnonzero(depth >= 1)
    nW = -(-len(idx) // W)
    assert (sc.n_windows == nW).all()
    assert (sc.w_nsites[:, :nW - 1] == W).all() and (sc.w_nsites[:, :nW].sum(axis=1) == len(idx)).all()
    np.testing.assert_array_equal(sc.w_start[0, :nW], pos[idx[0::W]])
    np.testing.assert_array_equal(sc.w_end[T - 1, :nW - 1], pos[idx[W - 1::W]][:nW - 1])
    assert np.isfinite(sc.w_loglik[:, :nW]).all()
    assert int(sc.processed[0]) + int(sc.skipped[0]) == S
    # LIBD0 does not depend on the target's genotype
    assert np.ptp(sc.w_loglik[:, :nW, 0], axis=0).max() == 0.0
    prm = oracle.Params(window=W, ld_mode=0)
    bg = np.arange(N, dtype=np.int32)
    for w in (0, 4321, nW - 2):
        rows = np.arange(idx[w * W], idx[(w + 1) * W - 1] + 1)
        hap = unpack_rows(bits, 2 * N, rows)
        for t in (0, 57, T - 1):
            o = oracle.compare_target(prm, pos[rows], keep[rows], n_ref[rows], n_alt[rows], hap, int(t), bg)
            assert o["n_windows"] == 1 and int(o["w_nsites"][0]) == W
            np.testing.assert_allclose(sc.w_loglik[t, w], o["w_log"][0], rtol=0, atol=1e-8)


def test_c4_full_size_spot_checks_against_oracle():
    """BASELINE.json configs[3] at full size (10,000 tables x 10,000 bins of log-likelihoods, planted segments):
    tables are independent, so any table can be decoded by the CPU oracle on its own (as far as the reference's
    long double range reaches); plus size-independent properties of the whole batch (state counts of every table)."""
    import torch
    import ibdgem_b200 as ib
    import oracle
    n_tables, n_bins = 10_000, 10_000
    nb = n_tables * n_bins
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=gen, device=dev).repeat_interleave(200)[:nb]
    ll = torch.randn((nb, 3), generator=gen, device=dev, dtype=torch.float64) * 10.0 - 150.0
    ll[torch.arange(nb, device=dev), seg] += 8.0
    h_ll = ll.cpu().numpy()
    del ll, seg
    torch.cuda.empty_cache()
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    with ib.Engine(ib.Params()) as e:
        state, score, counts = e.viterbi_batch(h_ll, off, True)
        assert e.kernel_stats()["viterbi_back"][1] > 0  # the batched kernels are the ones that ran
    st2 = state.reshape(n_tables, n_bins)
    assert int(st2.max()) <= 2 and (counts.sum(axis=1) == n_bins).all()
    for k in range(3):
        np.testing.assert_array_equal((st2 == k).sum(axis=1), counts[:, k])
    # The reference's running long double products leave the normal range after ~5,700 of these bins (about -2 nats
    # per bin) and every later state reads 0 there (SURVEY.md Appendix A; INTEGRATION.md 4): the log-space front-end
    # keeps going, so the oracle is the judge up to that bin — forward scores exactly up to it, states up to one
    # segment before it (the back-trace enters the valid part from whatever the tail decided and coalesces within bins).
    tiny = np.finfo(np.longdouble).tiny
    for t in (0, 4999, n_tables - 1):
        sl = slice(t * n_bins, (t + 1) * n_bins)
        st, sc, sc_ld = oracle.hiddengem(np.exp(h_ll[sl]))
        bad = np.flatnonzero((sc_ld < tiny).any(axis=1))
        n_ok = int(bad[0]) if len(bad) else n_bins
        assert n_ok > 2000, n_ok
        np.testing.assert_allclose(score[sl][:n_ok], sc[:n_ok], rtol=0, atol=1e-6)
        np.testing.assert_array_equal(st2[t][: n_ok - 400], st[: n_ok - 400])
