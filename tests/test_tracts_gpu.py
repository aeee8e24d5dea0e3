"""hiddengem IBD tracts on the GPU (hiddengem_tracts_device / _batch, hiddengem --tracts, ibdgem --hiddengem --tracts)
against the run-length oracle of test_tracts_cpu.py over the Viterbi states and posteriors."""
import json
import os
import subprocess

import numpy as np
import pytest

import hostlib
from test_cli_gpu import TIE_PENALTIES, _golden_states, _long_table, _tie_tables
from test_posterior_gpu import PENALTIES, _tables
from test_tracts_cpu import assert_tracts, tract_oracle

pytestmark = pytest.mark.gpu

CA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_runs", "caseA")


def _geometry(rng, n_tables, is_log):
    """Ragged tables around the 32-bin strides (0, 1, 31, 32, 33, 63, 64, 65 and up to 4,000 bins), planted runs."""
    edge = np.array([0, 1, 31, 32, 33, 63, 64, 65, 4000])
    lens = np.where(rng.random(n_tables) < 0.5, edge[rng.integers(0, len(edge), n_tables)], rng.integers(0, 4001, n_tables))
    lens[rng.random(n_tables) < 0.1] = 0
    lens[0] = edge[n_tables % len(edge)]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nb = int(off[-1])
    seg = np.repeat(rng.integers(0, 3, nb // 37 + 1), 37)[:nb]
    if is_log:
        lik = rng.normal(-200, 30, (nb, 3))
        lik[np.arange(nb), seg] += 6.0
        lik[rng.random(nb) < 0.005, 1] = -np.inf
    else:
        lik = np.exp(rng.normal(-20, 3, (nb, 3)))
        lik[np.arange(nb), seg] *= np.exp(6.0)
        lik[rng.random(nb) < 0.005, 2] = 0.0
    return lik, off


def _device_states(e, lik, off, is_log, stride, pen=(1e-3, 1e-6, 1e-3)):
    """Viterbi states and posteriors through the two device entries, in the packed (stride 0) or strided layout: the
    device buffers (lik, state, posterior) and host copies laid out the same way, plus each table's start."""
    import torch
    nt = len(off) - 1
    lens = np.diff(off)
    if stride:
        lay = np.full((nt * stride, 3), np.nan)
        starts = np.arange(nt, dtype=np.int64) * stride
        for t in range(nt):
            lay[starts[t]: starts[t] + lens[t]] = lik[off[t]: off[t + 1]]
    else:
        lay, starts = lik, off[:-1]
    n = max(len(lay), 1)
    d_lik = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    d_lik[: len(lay)] = torch.from_numpy(np.ascontiguousarray(lay)).cuda()
    d_state = torch.zeros(n, dtype=torch.uint8, device="cuda")
    d_score = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    d_counts = torch.zeros((nt, 3), dtype=torch.int64, device="cuda")
    d_post = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
    d_exp = torch.zeros((nt, 3), dtype=torch.float64, device="cuda")
    p01, p02, p12 = pen
    e.viterbi_batch_device(d_lik.data_ptr(), off, is_log, d_state.data_ptr(), d_score.data_ptr(), d_counts.data_ptr(),
                           table_stride=stride, p01=p01, p02=p02, p12=p12)
    e.posterior_batch_device(d_lik.data_ptr(), off, is_log, d_post.data_ptr(), d_exp.data_ptr(), table_stride=stride,
                             p01=p01, p02=p02, p12=p12)
    return d_lik, d_state, d_post, lay, starts, d_counts


@pytest.mark.parametrize("with_post", [False, True])
@pytest.mark.parametrize("stride", [0, 4096])
@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 64, 97, 300])
def test_device_entry_geometry(n_tables, is_log, stride, with_post):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(1000 + n_tables + 10 * is_log)
    lik, off = _geometry(rng, n_tables, is_log)
    if int(off[-1]) == 0:
        off[1:] += 1
        lik = np.full((1, 3), 0.5 if not is_log else -1.0)
    with ib.Engine(ib.Params()) as e:
        d_lik, d_state, d_post, lay, starts, _ = _device_states(e, lik, off, is_log, stride)
        e.enable_timing(True)
        e.reset_stats()
        toff, got = e.tracts_device(d_lik.data_ptr(), off, is_log, d_state.data_ptr(), d_post.data_ptr() if with_post else 0,
                                    table_stride=stride)
        stats = e.kernel_stats()
        states, post = d_state.cpu().numpy(), d_post.cpu().numpy()
    assert stats["tract_count"][1] == 1 and stats["tract_emit"][1] == 1
    assert_tracts(toff, got, tract_oracle(states, lay, off, is_log, post if with_post else None, starts))


def _crafted(n_tables, n, kind, rng):
    lens = np.full(n_tables, n)
    if kind == "every_bin":
        x = [np.arange(k, k + n) % 3 for k in range(n_tables)]
    elif kind == "stride_edges":  # changes at 32k - 1, 32k, 32k + 1
        x = []
        for t in range(n_tables):
            s = np.zeros(n, np.int64)
            for k in range(1, n // 32 + 1):
                for j, b in enumerate((32 * k - 1, 32 * k, 32 * k + 1)):
                    if b < n and (k + t + j) % 2:
                        s[b:] = (s[b] + 1 + (k + j) % 2) % 3
            x.append(s)
    elif kind == "one_state":
        x = [np.full(n, t % 3) for t in range(n_tables)]
    else:
        raise ValueError(kind)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    states = np.concatenate(x).astype(np.uint8)
    nb = int(off[-1])
    lik = rng.normal(-50, 10, (nb, 3))
    post = rng.random((nb, 3))
    post /= post.sum(axis=1, keepdims=True)
    post[rng.random(nb) < 0.001] = np.nan
    return states, lik, post, off


@pytest.mark.parametrize("kind,n_tables,n", [("every_bin", 5, 4000), ("every_bin", 70, 97), ("stride_edges", 9, 3000),
                                             ("stride_edges", 40, 161), ("one_state", 33, 2000), ("one_state", 1, 1_000_000)])
def test_device_entry_crafted_states(kind, n_tables, n):
    import torch
    import ibdgem_b200 as ib
    rng = np.random.default_rng(7)
    states, lik, post, off = _crafted(n_tables, n, kind, rng)
    with ib.Engine(ib.Params()) as e:
        d_lik, d_post = torch.from_numpy(lik).cuda(), torch.from_numpy(post).cuda()
        d_state = torch.from_numpy(states).cuda()
        for with_post in (True, False):
            toff, got = e.tracts_device(d_lik.data_ptr(), off, True, d_state.data_ptr(), d_post.data_ptr() if with_post else 0)
            assert_tracts(toff, got, tract_oracle(states, lik, off, True, post if with_post else None))
    if kind == "every_bin":
        assert toff[-1] == off[-1]
    if kind == "one_state":
        assert toff[-1] == n_tables and (got["n_bins"] == n).all()


def test_state_byte_above_two_fails_the_call():
    import torch
    import ibdgem_b200 as ib
    states = np.zeros(100, np.uint8)
    states[77] = 3
    lik = np.zeros((100, 3))
    with ib.Engine(ib.Params()) as e:
        d_lik, d_state = torch.from_numpy(lik).cuda(), torch.from_numpy(states).cuda()
        with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_tracts_device\(\): a state byte is above 2"):
            e.tracts_device(d_lik.data_ptr(), [0, 40, 100], True, d_state.data_ptr())
        d_state[77] = 1  # the engine is still usable
        toff, got = e.tracts_device(d_lik.data_ptr(), [0, 40, 100], True, d_state.data_ptr())
        np.testing.assert_array_equal(toff, [0, 1, 4])


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("n_tables", [1, 31, 64, 300])
@pytest.mark.parametrize("pen", list(PENALTIES))
def test_host_entry_matches_viterbi_and_posterior(is_log, n_tables, pen):
    import ibdgem_b200 as ib
    rng = np.random.default_rng(200 + n_tables + 7 * is_log)
    lik, off = _tables(rng, n_tables, is_log)
    if int(off[-1]) == 0:
        off[-1] = 1
        lik = np.array([[0.1, 0.2, 0.3]])
    p = PENALTIES[pen]
    with ib.Engine(ib.Params()) as e:
        states, _, _ = e.viterbi_batch(lik, off, is_log, *p)
        post, _ = e.posterior_batch(lik, off, is_log, *p)
        toff, got = e.tracts_batch(lik, off, is_log, *p)
        assert_tracts(toff, got, tract_oracle(states, lik, off, is_log, post))
        toff, got = e.tracts_batch(lik, off, is_log, *p, posterior=False)
        assert_tracts(toff, got, tract_oracle(states, lik, off, is_log))


def test_host_entry_zero_weight_table_and_zero_penalties():
    import ibdgem_b200 as ib
    lik = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.2, 0.3, 0.5], [0.0, 0.0, 0.0], [0.5, 0.2, 0.3]])
    off = np.array([0, 2, 5])
    with ib.Engine(ib.Params()) as e:
        toff, got = e.tracts_batch(lik, off, False, 0.0, 1e-3, 1e-3)
        states, _, _ = e.viterbi_batch(lik, off, False, 0.0, 1e-3, 1e-3)
        post, _ = e.posterior_batch(lik, off, False, 0.0, 1e-3, 1e-3)
        assert np.isnan(post[:2]).all()
        assert_tracts(toff, got, tract_oracle(states, lik, off, False, post))
        t0 = got[: toff[1]]
        assert np.isnan(t0["post_mean"]).all() and np.isnan(t0["post_min"]).all()  # the zero-weight table
        assert np.isfinite(got[toff[1]:]["post_mean"]).all()
        for pen in ((0.0, 0.0, 0.0), (0.0, 1e-3, 0.0)):  # without posteriors, zero penalties are accepted
            toff, got = e.tracts_batch(lik, off, False, *pen, posterior=False)
            states, _, _ = e.viterbi_batch(lik, off, False, *pen)
            assert_tracts(toff, got, tract_oracle(states, lik, off, False))


def _as_text(l):
    """The values hiddengem reads back from a summary file written with "%e" (test_cli_gpu._write_summary)."""
    return np.array([[float("%e" % v) for v in row] for row in l])


@pytest.mark.parametrize("tag", list(TIE_PENALTIES))
def test_near_tie_guard_states(tag):
    import ibdgem_b200 as ib
    pen = TIE_PENALTIES[tag]
    p = dict(zip(pen[0::2], map(float, pen[1::2])))
    p = (p.get("--p01", 1e-3), p.get("--p02", 1e-6), p.get("--p12", 1e-3))
    tables = [_as_text(l) for l in _tie_tables()]
    names = [f"tie{k}.{tag}" for k in range(len(tables))]
    if tag == "default":
        tables.append(_as_text(_long_table()))
        names.append("long")
    lik = np.concatenate(tables)
    off = np.concatenate([[0], np.cumsum([len(l) for l in tables])]).astype(np.int64)
    want = np.concatenate([np.array(_golden_states(nm)[0], dtype=np.int64) for nm in names]).astype(np.uint8)
    with ib.Engine(ib.Params()) as e:
        toff, got = e.tracts_batch(lik, off, False, *p)
        flagged = e.viterbi_last_flagged()
        post, _ = e.posterior_batch(lik, off, False, *p)
        states, _, _ = e.viterbi_batch(lik, off, False, *p)
        assert e.viterbi_last_flagged() == flagged
    assert flagged > 0
    np.testing.assert_array_equal(states, want)
    assert_tracts(toff, got, tract_oracle(want, lik, off, False, post))


def test_chained_device_path_from_score_ld():
    """score_ld's w_loglik_device ([T][max_windows][3]) through both device entries into the tract entry, strided,
    equals the host tract entry on the packed host copy.  Penalties 1: the unrelated targets' states then follow the
    windows' likelihoods, so tables hold many tracts."""
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
        d_state = torch.zeros((len(targets), mw), dtype=torch.uint8, device="cuda")
        d_score = torch.zeros((len(targets), mw, 3), dtype=torch.float64, device="cuda")
        d_counts = torch.zeros((len(targets), 3), dtype=torch.int64, device="cuda")
        d_post = torch.zeros((len(targets), mw, 3), dtype=torch.float64, device="cuda")
        d_exp = torch.zeros((len(targets), 3), dtype=torch.float64, device="cuda")
        pen = dict(p01=1.0, p02=1.0, p12=1.0)
        e.viterbi_batch_device(d_wll.data_ptr(), off, True, d_state.data_ptr(), d_score.data_ptr(), d_counts.data_ptr(), table_stride=mw,
                               **pen)
        e.posterior_batch_device(d_wll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), table_stride=mw, **pen)
        toff_d, got_d = e.tracts_device(d_wll.data_ptr(), off, True, d_state.data_ptr(), d_post.data_ptr(), table_stride=mw)
        toff_h, got_h = e.tracts_batch(packed, off, True, **pen)
        states, _, _ = e.viterbi_batch(packed, off, True, **pen)
        post, _ = e.posterior_batch(packed, off, True, **pen)
    assert toff_h[-1] > len(targets)  # some tables have more than one tract
    np.testing.assert_array_equal(toff_d, toff_h)
    assert got_d.tobytes() == got_h.tobytes()
    assert_tracts(toff_h, got_h, tract_oracle(states, packed, off, True, post))


def test_c4_full_size():
    """C4: 10,000 tables x 10,000 bins (tools/bench_posterior.py's tables), device-resident."""
    import torch
    import ibdgem_b200 as ib
    n_tables, n_bins = 10_000, 10_000
    nb = n_tables * n_bins
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=g, device=dev).repeat_interleave(200)[:nb]
    d_ll = torch.randn((nb, 3), generator=g, device=dev, dtype=torch.float64) * 10.0 - 150.0
    d_ll[torch.arange(nb, device=dev), seg] += 8.0
    del seg
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    d_state = torch.empty((nb,), dtype=torch.uint8, device=dev)
    d_post = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_counts = torch.empty((n_tables, 3), dtype=torch.int64, device=dev)
    with ib.Engine(ib.Params()) as e:
        d_score = torch.empty((nb, 3), dtype=torch.float64, device=dev)
        e.viterbi_batch_device(d_ll.data_ptr(), off, True, d_state.data_ptr(), d_score.data_ptr(), d_counts.data_ptr())
        del d_score
        d_exp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
        e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr())
        e.enable_timing(True)
        e.reset_stats()
        toff, got = e.tracts_device(d_ll.data_ptr(), off, True, d_state.data_ptr(), d_post.data_ptr())
        stats = e.kernel_stats()
    assert stats["tract_count"][1] == 1 and stats["tract_emit"][1] == 1
    st = d_state.view(n_tables, n_bins)
    changes = int((st[:, 1:] != st[:, :-1]).sum())
    assert toff[-1] == changes + n_tables
    table = np.repeat(np.arange(n_tables), np.diff(toff))
    per_state = np.zeros((n_tables, 3), np.int64)
    np.add.at(per_state, (table, got["state"]), got["n_bins"])
    np.testing.assert_array_equal(per_state, d_counts.cpu().numpy())
    rng = np.random.default_rng(4)
    for t in rng.choice(n_tables, 12, replace=False):
        a, b = int(off[t]), int(off[t + 1])
        want = tract_oracle(st[t].cpu().numpy(), d_ll[a:b].cpu().numpy(), [0, n_bins], True, d_post[a:b].cpu().numpy())
        assert_tracts(toff[t: t + 2] - toff[t], got[toff[t]: toff[t + 1]], want)


def test_errors():
    import torch
    import ibdgem_b200 as ib
    lik = np.full((10, 3), 0.3)
    with ib.Engine(ib.Params()) as e:
        with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_last_tracts\(\): no tract call has succeeded"):
            e.last_tracts(1)
        with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_tracts_batch\(\): table 1 has -3 bins"):
            e.tracts_batch(lik, [0, 7, 4, 10])
        d_lik, d_state = torch.from_numpy(lik).cuda(), torch.zeros(10, dtype=torch.uint8, device="cuda")
        with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_tracts_device\(\): table 1 has -3 bins"):
            e.tracts_device(d_lik.data_ptr(), [0, 7, 4, 10], False, d_state.data_ptr())
        for bad in ((-1e-3, 1e-6, 1e-3), (1e-3, np.nan, 1e-3)):
            with pytest.raises(ib.EngineError, match=r"ERROR in hiddengem_tracts_batch\(\): penalties must be finite"):
                e.tracts_batch(lik, [0, 10], False, *bad)
        with pytest.raises(ib.EngineError, match=r"no tract call has succeeded"):
            e.last_tracts(1)
        toff, got = e.tracts_batch(lik, [0, 4, 10], False)
        np.testing.assert_array_equal(toff, [0, 1, 2])
        with pytest.raises(ib.EngineError, match=r"penalties must be finite"):  # rejected before the records are touched
            e.tracts_batch(lik, [0, 10], False, -1.0, 1e-6, 1e-3)
        assert e.last_tracts(2).tobytes() == got.tobytes()


# --- command lines ---------------------------------------------------------------------------------------------------
def _run(binary, args, cwd=None):
    r = subprocess.run([os.path.join(hostlib.BIN, binary)] + args, capture_output=True, text=True, cwd=cwd, timeout=300)
    assert r.returncode == 0, r.stderr
    return r


def _rows(path):
    with open(path) as fh:
        lines = fh.read().splitlines()
    return lines[0].split("\t"), [ln.split("\t") for ln in lines[1:]]


def _summary_bins(path):
    rows = [ln.split("\t") for ln in open(path).read().splitlines() if ln and not ln.startswith("#")]
    return [(int(r[1]), int(r[2]), int(r[6])) for r in rows]


def _stdout_bins(text):
    rows = [ln.split("\t") for ln in text.splitlines()[1:] if not ln.startswith("#")]
    return [r[4] for r in rows], [[r[5], r[6], r[7]] for r in rows if len(r) > 5]


_LOOSE = ["--p01", "0.2", "--p02", "0.05", "--p12", "0.3"]
HG = [("nonld_w10", "ind2", "default", []), ("nonld_w10", "ind3", "default", []), ("nonld_w10", "ind5", "default", []),
      ("nonld_w10", "ind2", "loose", _LOOSE), ("nonld_w10", "ind3", "loose", _LOOSE), ("nonld_w10", "ind5", "loose", _LOOSE),
      ("ld_w100_underflow", "ind3", "ld_underflow", [])]


@pytest.fixture(scope="module")
def _built():
    hostlib.build()


@pytest.mark.parametrize("run,ind,tag,args", HG)
@pytest.mark.parametrize("posterior", [False, True])
def test_hiddengem_tracts_file(_built, tmp_path, run, ind, tag, args, posterior):
    sfile = os.path.join(CA, run, f"UNKWN.{ind}.summary.txt")
    extra = args + (["--posterior"] if posterior else [])
    plain = _run("hiddengem", ["-s", sfile] + extra).stdout
    tf = str(tmp_path / "tracts.txt")
    r = _run("hiddengem", ["-s", sfile, "--tracts", tf] + extra)
    assert r.stdout == plain  # stdout is unchanged
    head, rows = _rows(tf)
    assert head == ["Summary", "Tract", "Inferred_State", "First_Segment", "Last_Segment", "START", "END", "N_Segments",
                    "NUM_SITES", "LOD10"] + (["P_Mean", "P_Min"] if posterior else [])
    ref_states, _ = _stdout_bins(open(os.path.join(CA, "hiddengem", f"{ind}.{tag}.txt")).read())
    bins = _summary_bins(sfile)
    decoded = []
    for k, row in enumerate(rows):
        assert row[0] == sfile and int(row[1]) == k + 1
        a, b, n = int(row[3]), int(row[4]), int(row[7])
        assert b - a + 1 == n and a == len(decoded) + 1
        decoded += [row[2]] * n
        assert int(row[5]) == bins[a - 1][0] and int(row[6]) == bins[b - 1][1]
        assert int(row[8]) == sum(x[2] for x in bins[a - 1: b])
        float(row[9])
    assert decoded == ref_states  # run-length decodes to the reference's Inferred_State column
    if posterior:
        states, p = _stdout_bins(plain)
        for row in rows:
            a, b, s = int(row[3]), int(row[4]), int(row[2])
            own = [p[i][s] for i in range(a - 1, b)]
            assert row[11] == min(own, key=float)  # rounding is monotone: the printed minimum is exact
            assert float(row[10]) == pytest.approx(np.mean([float(v) for v in own]), abs=1e-6)


def test_hiddengem_tracts_several_files_in_order(_built, tmp_path):
    files = [os.path.join(CA, "nonld_w10", f"UNKWN.{ind}.summary.txt") for ind in ("ind3", "ind2", "ind5", "ind2")]
    args = []
    for f in files:
        args += ["-s", f]
    tf = str(tmp_path / "all.txt")
    _run("hiddengem", args + ["--tracts", tf])
    _, rows = _rows(tf)
    singles = []
    for k, f in enumerate(files[:3]):
        one = str(tmp_path / f"one{k}.txt")
        _run("hiddengem", ["-s", f, "--tracts", one])
        singles.append(_rows(one)[1])
    assert rows == singles[0] + singles[1] + singles[2] + singles[1]  # each file's tracts under its name, in -s order


def test_ibdgem_hiddengem_tracts_files(_built, tmp_path):
    """ibdgem --hiddengem --tracts writes <pileup>.<target>.tracts.txt; apart from the Summary column they equal hiddengem
    --tracts on the run's own summary files (LOD10 up to the 7 printed digits of those files' likelihoods)."""
    meta = json.load(open(os.path.join(CA, "nonld_w10", "ARGS.json")))
    base = ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup"] + meta["args"] + ["--hiddengem", "--no-tab"]
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    _run("ibdgem", base + ["-O", str(tmp_path / "a"), "--posterior"], cwd=CA)
    _run("ibdgem", base + ["-O", str(tmp_path / "b"), "--posterior", "--tracts"], cwd=CA)
    for ind in ("ind2", "ind3", "ind5"):
        for f in ("hiddengem", "summary"):  # the other outputs do not change
            assert open(tmp_path / "b" / f"UNKWN.{ind}.{f}.txt").read() == open(tmp_path / "a" / f"UNKWN.{ind}.{f}.txt").read()
        head, rows = _rows(tmp_path / "b" / f"UNKWN.{ind}.tracts.txt")
        tf = str(tmp_path / f"{ind}.txt")
        _run("hiddengem", ["-s", str(tmp_path / "b" / f"UNKWN.{ind}.summary.txt"), "--tracts", tf, "--posterior"])
        whead, wrows = _rows(tf)
        assert head == whead[1:]
        assert len(rows) == len(wrows)
        for g, w in zip(rows, wrows):
            assert g[:8] == w[1:9]
            assert float(g[8]) == pytest.approx(float(w[9]), abs=2e-4 + 1e-5 * int(g[6]))  # LOD10
            assert float(g[9]) == pytest.approx(float(w[10]), abs=2e-6) and float(g[10]) == pytest.approx(float(w[11]), abs=2e-6)
    assert not list((tmp_path / "a").glob("*.tracts.txt"))
