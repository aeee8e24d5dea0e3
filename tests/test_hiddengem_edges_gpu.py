"""hiddengem on the GPU at the edges of its range and of its batch geometry.

Posterior (hiddengem_posterior_batch and _device) against the log-space oracle of test_posterior_cpu.py, which
test_hiddengem_edges_cpu.py checks against 60-digit enumeration on exactly these rows: states thousands of nats apart,
zero, subnormal and near-DBL_MAX penalties, with each awkward table a lane beside healthy ones in the same block.
Viterbi (hiddengem_viterbi_batch and _device) against the C oracle's states and counts on the tables whose lengths and
numbers sit at the kernels' 16-bin chunks, 32-table blocks and the 64-table threshold of the batched path."""
import numpy as np
import pytest

from test_cli_gpu import TIE_PENALTIES, _long_table, _tie_tables
from test_hiddengem_edges_cpu import GAPS, LOG_CASES, PENALTY_SETS, gap_rows, to_text
from test_posterior_cpu import posterior_oracle
from test_posterior_gpu import _check
from test_tracts_gpu import _as_text

pytestmark = pytest.mark.gpu

LENGTHS = (0, 1, 2, 15, 16, 17, 31, 32, 33, 255, 256, 257, 4000)
N_TABLES = (1, 31, 32, 33, 63, 64, 65, 97)


def linear_path(p):
    """The posterior's fp64 linear-space kernels serve the call (posterior.cu): every penalty positive and
    max(1, p) / min(1, p) <= 2^400."""
    lo, hi = min(1.0, *p), max(1.0, *p)
    return lo > 0 and hi / lo <= 2.0 ** 400


def _healthy(rng, n, is_log):
    seg = np.repeat(rng.integers(0, 3, n // 40 + 1), 40)[:n]
    if is_log:
        lik = rng.normal(-200, 30, (n, 3))
        lik[np.arange(n), seg] += 5.0
    else:
        lik = np.exp(rng.normal(-20, 3, (n, 3)))
        lik[np.arange(n), seg] *= np.exp(5.0)
    return lik


def _embed(special, rng, is_log):
    """The special tables among healthy ragged ones (1-300 bins), each with healthy neighbours in its block."""
    tables, where = [], []
    for t in special:
        for _ in range(int(rng.integers(1, 4))):
            tables.append(_healthy(rng, int(rng.integers(1, 300)), is_log))
        where.append(len(tables))
        tables.append(np.asarray(t, np.float64))
    tables.append(_healthy(rng, 100, is_log))
    return tables, where


def _offsets(tables):
    return np.concatenate([[0], np.cumsum([len(t) for t in tables])]).astype(np.int64)


def _posterior_both_entries(tables, is_log, pen):
    """Host entry, then the device entry on a [T][longest][3] layout (table_stride = the longest table, so it has no
    padding); the two must agree bit for bit and the device entry writes nothing past a table's bins.
    Returns (lik, off, post, expected, kernel_stats)."""
    import torch
    import ibdgem_b200 as ib
    off = _offsets(tables)
    lens = np.diff(off)
    lik = np.concatenate(tables) if off[-1] else np.zeros((0, 3))
    with ib.Engine(ib.Params()) as e:
        post, expected = e.posterior_batch(lik, off, is_log, *pen)
        stats = e.kernel_stats()
        stride = int(lens.max())
        if stride:
            strided = np.full((len(tables), stride, 3), np.nan)
            for t, l in enumerate(tables):
                strided[t, : len(l)] = l
            d_lik = torch.from_numpy(strided).cuda()
            d_post = torch.full((len(tables), stride, 3), 7.0, dtype=torch.float64, device="cuda")
            d_exp = torch.zeros((len(tables), 3), dtype=torch.float64, device="cuda")
            e.posterior_batch_device(d_lik.data_ptr(), off, is_log, d_post.data_ptr(), d_exp.data_ptr(), table_stride=stride,
                                     p01=pen[0], p02=pen[1], p12=pen[2])
            p2 = d_post.cpu().numpy()
            np.testing.assert_array_equal(d_exp.cpu().numpy(), expected)
            for t in range(len(tables)):
                np.testing.assert_array_equal(p2[t, : lens[t]], post[off[t]: off[t + 1]])
                assert (p2[t, lens[t]:] == 7.0).all()
    return lik, off, post, expected, stats


def _judge(lik, off, is_log, pen, post, expected, stats=None):
    """Posteriors within 1e-9 and expected counts within 1e-6 of the oracle; NaN exactly in the tables whose oracle
    total weight is 0, and every other table finite."""
    _check(post, expected, lik, off, is_log, pen)
    want, _ = posterior_oracle(lik, off, is_log, *pen)
    for t in range(len(off) - 1):
        g, w = post[off[t]: off[t + 1]], want[off[t]: off[t + 1]]
        if np.isnan(w).any():
            assert np.isnan(g).all() and np.isnan(expected[t]).all(), t
        else:
            assert np.isfinite(g).all() and np.isfinite(expected[t]).all(), t
    if stats is not None:  # both passes ran once, in linear or in natural-log arithmetic as the penalties require
        lin = linear_path(pen)
        assert stats["posterior_fwd"][1] == 1 and stats["posterior_bwd"][1] == 1, ("path", stats)
        assert stats.get("posterior_fwd_log", (0, 0))[1] == int(not lin), ("path", stats)
        assert stats.get("posterior_bwd_log", (0, 0))[1] == int(not lin), ("path", stats)


# ---- range x penalties ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("name", list(LOG_CASES))
def test_posterior_named_range_cases(is_log, name):
    rows, pen = LOG_CASES[name]
    rng = np.random.default_rng(sorted(LOG_CASES).index(name))
    special = np.array(rows, np.float64) if is_log else to_text(rows)
    tables, where = _embed([special, special], rng, is_log)
    lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, pen)
    _judge(lik, off, is_log, pen, post, expected, stats)


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("pen", list(PENALTY_SETS))
def test_posterior_gap_sweep(is_log, pen):
    """Gaps of 600 to 5,000 nats between IBD1 and the best state of each bin, every penalty set."""
    p = PENALTY_SETS[pen]
    rng = np.random.default_rng(40 + list(PENALTY_SETS).index(pen))
    special = [gap_rows(g) if is_log else to_text(gap_rows(g)) for g in GAPS]
    tables, _ = _embed(special, rng, is_log)
    lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, p)
    _judge(lik, off, is_log, p, post, expected, stats)


def _adversarial(rng, is_log):
    """Rows that stress a linear-space forward-backward: IBD1 745+ nats behind, states forced to alternate through
    the weakest transition, and 300-bin tables whose entries spread over thousands of nats."""
    t = [gap_rows(g) for g in (745, 800, 1500, 5000)]
    alt = np.full((20, 3), -np.inf)
    alt[0::2, 0] = 0.0
    alt[1::2, 2] = 0.0
    t.append(alt)  # IBD0 / IBD2 alternate: every path pays p02 19 times
    via1 = np.full((21, 3), -np.inf)
    via1[0::4, 0] = 0.0
    via1[1::4, 1] = -760.0
    via1[1::4, 0] = 0.0
    via1[2::4, 2] = 0.0
    via1[3::4, 1] = -760.0
    via1[3::4, 2] = 0.0
    t.append(via1)
    t += [rng.normal(0, 1000, (300, 3)), rng.normal(-500, 400, (300, 3))]
    return t if is_log else [to_text(x) for x in t]


BOUNDARY = {  # penalties, and whether the linear kernels serve them
    "all_2^-400": ((2.0 ** -400,) * 3, True),
    "all_2^400": ((2.0 ** 400,) * 3, True),
    "spread_2^400": ((2.0 ** -200, 2.0 ** 200, 2.0 ** -200), True),
    "p02_2^-400": ((1e-3, 2.0 ** -400, 1e-3), True),
    "below_2^-400": ((np.nextafter(2.0 ** -400, 0),) * 3, False),
    "above_2^400": ((np.nextafter(2.0 ** 400, np.inf),) * 3, False),
    "spread_above_2^400": ((2.0 ** -200, np.nextafter(2.0 ** 200, np.inf), 2.0 ** -200), False),
    "mixed_2^-400_2^400": ((2.0 ** -400, 2.0 ** 400, 2.0 ** -400), False),
}


@pytest.mark.parametrize("is_log", [False, True])
@pytest.mark.parametrize("name", list(BOUNDARY))
def test_posterior_at_the_linear_path_bound(is_log, name):
    pen, lin = BOUNDARY[name]
    assert linear_path(pen) == lin
    rng = np.random.default_rng(70 + list(BOUNDARY).index(name))
    tables, _ = _embed(_adversarial(rng, is_log), rng, is_log)
    lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, pen)
    _judge(lik, off, is_log, pen, post, expected, stats)


def test_posterior_chained_from_score_ld_with_p02_zero():
    """score_ld window scores of long windows over a pileup whose source changes from target 0 to target 1 halfway
    along the sites, straight from w_loglik_device into posterior_batch_device with p02 = 0 and
    table_stride = max_windows: at the change, a state that led one window is over 700 nats behind in the next."""
    import torch
    import ibdgem_b200 as ib
    rng = np.random.default_rng(21)
    N, W, n_win = 32, 8000, 16
    S = W * n_win
    af = np.clip(rng.beta(0.5, 2.0, S), 0.01, 0.99)
    hap = (rng.random((S, 2 * N)) < af[:, None]).astype(np.uint8)
    pos = (1000 + 60 * np.arange(S)).astype(np.uint64)
    d = rng.poisson(4.0, S)
    src = np.where(np.arange(S) < S // 2, 0, 1)
    g = hap[np.arange(S), 2 * src] + hap[np.arange(S), 2 * src + 1]
    n_alt = rng.binomial(d, np.where(g == 0, 0.02, np.where(g == 1, 0.5, 0.98))).astype(np.uint8)
    n_ref = (d - n_alt).astype(np.uint8)
    keep = np.ones(S, np.uint8)
    targets = np.arange(8, dtype=np.int32)
    pen = (1e-3, 0.0, 1e-3)
    with ib.Engine(ib.Params(window_size=W)) as e:
        e.upload_sites(pos, n_ref, n_alt, keep)
        e.upload_panel(ib.pack_bits(hap), N)
        mw = e.default_max_windows()
        d_wll = torch.full((len(targets), mw, 3), np.nan, dtype=torch.float64, device="cuda")
        sc = e.score_ld(targets, np.arange(N, dtype=np.int32), -1, device_out=d_wll.data_ptr())
        nw = sc.n_windows.astype(np.int64)
        off = np.concatenate([[0], np.cumsum(nw)]).astype(np.int64)
        packed = np.concatenate([sc.w_loglik[t, : nw[t]] for t in range(len(targets))])
        d_post = torch.full((len(targets), mw, 3), 7.0, dtype=torch.float64, device="cuda")
        d_exp = torch.zeros((len(targets), 3), dtype=torch.float64, device="cuda")
        e.posterior_batch_device(d_wll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), table_stride=mw,
                                 p01=pen[0], p02=pen[1], p12=pen[2])
        ph, eh = e.posterior_batch(packed, off, True, *pen)
    np.testing.assert_array_equal(np.asarray(packed), np.concatenate([d_wll.cpu().numpy()[t, : nw[t]] for t in range(len(targets))]))
    rel = packed - packed.max(axis=1, keepdims=True)
    jump = max(float(np.abs(np.diff(rel[off[t]: off[t + 1]], axis=0)).max()) for t in range(2))
    assert jump > 700.0, jump
    p2 = d_post.cpu().numpy()
    np.testing.assert_array_equal(d_exp.cpu().numpy(), eh)
    for t in range(len(targets)):
        np.testing.assert_array_equal(p2[t, : nw[t]], ph[off[t]: off[t + 1]])
        assert (p2[t, nw[t]:] == 7.0).all()
    _judge(packed, off, True, pen, ph, eh)


# ---- geometry: posterior --------------------------------------------------------------------------------------
def _cycled(n_tables):
    return [LENGTHS[(5 * k + n_tables) % len(LENGTHS)] for k in range(n_tables)]


@pytest.mark.parametrize("n_tables", N_TABLES)
@pytest.mark.parametrize("pen", ["default", "p02_zero"])
def test_posterior_geometry_n_tables(n_tables, pen):
    p = PENALTY_SETS[pen]
    is_log = bool(n_tables % 2)
    rng = np.random.default_rng(n_tables)
    tables = [_healthy(rng, n, is_log) for n in _cycled(n_tables)]
    lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, p)
    _judge(lik, off, is_log, p, post, expected, stats)


@pytest.mark.parametrize("length", LENGTHS)
def test_posterior_geometry_lengths(length):
    """One table alone, then 33 of the same length with a 1-bin table at lane 31 and 32 (block edges)."""
    rng = np.random.default_rng(1000 + length)
    for is_log in (False, True):
        for tables in ([_healthy(rng, length, is_log)],
                       [_healthy(rng, 1 if k in (31, 32) else length, is_log) for k in range(33)]):
            if sum(len(t) for t in tables) == 0:
                continue
            lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, PENALTY_SETS["default"])
            _judge(lik, off, is_log, PENALTY_SETS["default"], post, expected, stats)


def _special_layouts(rng, is_log):
    long_block = [_healthy(rng, 4000, is_log)] + [_healthy(rng, 1, is_log) for _ in range(31)] + \
                 [_healthy(rng, int(n), is_log) for n in rng.integers(1, 200, 32)]
    empty_block = [_healthy(rng, int(n), is_log) for n in rng.integers(1, 200, 32)] + [np.zeros((0, 3))] * 32 + \
                  [_healthy(rng, int(n), is_log) for n in rng.integers(1, 200, 33)]
    return {"long_and_31_one_bin": long_block, "empty_block": empty_block}


@pytest.mark.parametrize("layout", ["long_and_31_one_bin", "empty_block"])
@pytest.mark.parametrize("pen", ["default", "p02_zero", "all_zero"])
def test_posterior_special_layouts(layout, pen):
    p = PENALTY_SETS[pen]
    for is_log in (False, True):
        tables = _special_layouts(np.random.default_rng(5), is_log)[layout]
        lik, off, post, expected, stats = _posterior_both_entries(tables, is_log, p)
        _judge(lik, off, is_log, p, post, expected, stats)


# ---- geometry: Viterbi ----------------------------------------------------------------------------------------
VITERBI_PENALTIES = {"default": (1e-3, 1e-6, 1e-3), "p02_zero": (1e-3, 0.0, 1e-3), "all_zero": (0.0, 0.0, 0.0),
                     "loose": (0.2, 0.05, 0.3), "reward": (2.0, 0.5, 4.0)}


def _text_tables(rng, lens):
    out = []
    for k, n in enumerate(lens):
        seg = np.repeat(rng.integers(0, 3, n // 40 + 1), 40)[:n]
        l = np.exp(rng.normal(-20, 3, (n, 3)))
        l[np.arange(n), seg] *= np.exp(5.0)
        if n > 3 and k % 5 == 0:
            l[n // 2] = 0.0  # all-zero row
        if n > 3 and k % 7 == 0:
            l[1, 2] = 0.0
        out.append(l)
    return out


def _viterbi_batched(lens):
    n, total, maxbins = len(lens), int(sum(lens)), int(max(lens))
    return n >= 64 and maxbins * n <= 2 * total  # hidden.cu: viterbi_on_device


def _viterbi_check(tables, pen, want_batched, is_log=False):
    """Host entry and strided device entry (table_stride = the longest table) against oracle.hiddengem (on exp() of
    log rows); which path ran, from kernel_stats."""
    import torch
    import ibdgem_b200 as ib
    import oracle
    lens = [len(t) for t in tables]
    assert _viterbi_batched(lens) == want_batched
    off = _offsets(tables)
    lik = np.concatenate(tables)
    with ib.Engine(ib.Params()) as e:
        state, score, counts = e.viterbi_batch(lik, off, is_log, *pen)
        stats = e.kernel_stats()
        stride = max(lens)
        strided = np.full((len(tables), stride, 3), np.nan)
        for t, l in enumerate(tables):
            strided[t, : len(l)] = l
        d_lik = torch.from_numpy(strided).cuda()
        d_state = torch.full((len(tables), stride), 9, dtype=torch.uint8, device="cuda")
        d_score = torch.zeros((len(tables), stride, 3), dtype=torch.float64, device="cuda")
        d_cnt = torch.full((len(tables), 3), -1, dtype=torch.int64, device="cuda")
        e.viterbi_batch_device(d_lik.data_ptr(), off, is_log, d_state.data_ptr(), d_score.data_ptr(), d_cnt.data_ptr(),
                               table_stride=stride, p01=pen[0], p02=pen[1], p12=pen[2])
        s2, c2 = d_state.cpu().numpy(), d_cnt.cpu().numpy()
    assert (stats["viterbi_back"][1] > 0) == want_batched, stats
    assert stats["viterbi"][1] > 0
    np.testing.assert_array_equal(c2, counts)
    for t, l in enumerate(tables):
        a, b = off[t], off[t + 1]
        np.testing.assert_array_equal(s2[t, : len(l)], state[a:b])
        assert (s2[t, len(l):] == 9).all()
        if len(l) == 0:
            np.testing.assert_array_equal(counts[t], 0)
            continue
        with np.errstate(under="ignore"):
            st, _, _ = oracle.hiddengem(np.exp(l) if is_log else l, *pen)
        np.testing.assert_array_equal(state[a:b], st, err_msg=f"table {t} ({len(l)} bins)")
        np.testing.assert_array_equal(counts[t], np.bincount(st, minlength=3))


@pytest.mark.parametrize("n_tables", N_TABLES)
@pytest.mark.parametrize("pen", list(VITERBI_PENALTIES))
def test_viterbi_geometry_mixed_lengths(n_tables, pen):
    """Every length of LENGTHS, cycled: the per-table kernel (the 4,000-bin tables make the batch too ragged)."""
    lens = _cycled(n_tables)
    if max(lens) == 0:
        lens[0] = 17
    _viterbi_check(_text_tables(np.random.default_rng(n_tables), lens), VITERBI_PENALTIES[pen], False)


@pytest.mark.parametrize("n_tables", N_TABLES)
@pytest.mark.parametrize("around", [16, 32, 256])
@pytest.mark.parametrize("pen", list(VITERBI_PENALTIES))
def test_viterbi_geometry_even_lengths(n_tables, around, pen):
    """Lengths around - 1, around, around + 1 with two empty tables: the batched fused kernel from 64 tables on."""
    lens = [around - 1 + k % 3 for k in range(n_tables)]
    if n_tables > 2:
        lens[1] = lens[n_tables // 2] = 0
    _viterbi_check(_text_tables(np.random.default_rng(n_tables + around), lens), VITERBI_PENALTIES[pen], n_tables >= 64)


@pytest.mark.parametrize("pen", list(VITERBI_PENALTIES))
def test_viterbi_special_layouts(pen):
    rng = np.random.default_rng(6)
    p = VITERBI_PENALTIES[pen]
    # one 4,000-bin table and 31 one-bin tables in a block, then 64 tables of 3,500-4,000 bins: batched
    lens = [4000] + [1] * 31 + [int(n) for n in rng.integers(3500, 4001, 64)]
    _viterbi_check(_text_tables(rng, lens), p, True)
    # a block of empty tables between non-empty ones, per-table (fewer than 64 tables) and batched
    lens = [int(n) for n in rng.integers(200, 260, 16)] + [0] * 32 + [int(n) for n in rng.integers(200, 260, 15)]
    _viterbi_check(_text_tables(rng, lens), p, False)
    lens = [int(n) for n in rng.integers(200, 260, 32)] + [0] * 32 + [int(n) for n in rng.integers(200, 260, 96)]
    _viterbi_check(_text_tables(rng, lens), p, True)
    # natural-log rows within exp() range
    ll = [np.log(t) for t in _text_tables(rng, [int(n) for n in rng.integers(100, 140, 70)])]
    with np.errstate(divide="ignore"):
        _viterbi_check(ll, p, True, is_log=True)


@pytest.mark.parametrize("layout", ["packed", "strided"])
@pytest.mark.parametrize("tag", list(TIE_PENALTIES))
def test_viterbi_device_entry_near_ties(tag, layout):
    """The tie tables (and, at the default penalties, the long table) of test_tracts_gpu.test_near_tie_guard_states
    through hiddengem_viterbi_batch_device: the tables the near-tie guard flags are re-evaluated in long double and
    written back to the device buffers.  States, counts and the number of flagged tables equal the host entry's,
    scores of the flagged tables bit for bit (both from the long double recurrence), and nothing outside a table's bins
    is written."""
    import torch
    import ibdgem_b200 as ib
    opt = dict(zip(TIE_PENALTIES[tag][0::2], map(float, TIE_PENALTIES[tag][1::2])))
    pen = (opt.get("--p01", 1e-3), opt.get("--p02", 1e-6), opt.get("--p12", 1e-3))
    tables = [_as_text(l) for l in _tie_tables()]
    if tag == "default":
        tables.append(_as_text(_long_table()))
    off = _offsets(tables)
    lens = np.diff(off)
    lik = np.concatenate(tables)
    stride = int(lens.max()) + 37 if layout == "strided" else 0
    starts = np.arange(len(tables)) * stride if stride else off[:-1]
    rows = len(tables) * stride if stride else int(off[-1]) + 64
    inside = np.zeros(rows, bool)
    lay = np.full((rows, 3), np.nan)
    for t, l in enumerate(tables):
        inside[starts[t]: starts[t] + lens[t]] = True
        lay[starts[t]: starts[t] + lens[t]] = l
    with ib.Engine(ib.Params()) as e:
        flagged = []
        for l in tables:  # which tables the guard hands to the host: fewer than 64 tables run the per-table kernel
            e.viterbi_batch(l, [0, len(l)], False, *pen)
            flagged.append(e.viterbi_last_flagged() == 1)
        state, score, counts = e.viterbi_batch(lik, off, False, *pen)
        n_flagged = e.viterbi_last_flagged()
        d_lik = torch.from_numpy(lay).cuda()
        d_state = torch.full((rows,), 9, dtype=torch.uint8, device="cuda")
        d_score = torch.full((rows, 3), 7.0, dtype=torch.float64, device="cuda")
        d_cnt = torch.full((len(tables), 3), -1, dtype=torch.int64, device="cuda")
        e.viterbi_batch_device(d_lik.data_ptr(), off, False, d_state.data_ptr(), d_score.data_ptr(), d_cnt.data_ptr(),
                               table_stride=stride, p01=pen[0], p02=pen[1], p12=pen[2])
        assert e.viterbi_last_flagged() == n_flagged
        s2, sc2 = d_state.cpu().numpy(), d_score.cpu().numpy()
        np.testing.assert_array_equal(d_cnt.cpu().numpy(), counts)
    assert n_flagged > 0 and n_flagged == sum(flagged)
    for t in range(len(tables)):
        a, b, s = off[t], off[t + 1], starts[t]
        np.testing.assert_array_equal(s2[s: s + lens[t]], state[a:b])
        if flagged[t]:
            np.testing.assert_array_equal(sc2[s: s + lens[t]], score[a:b])
        else:
            np.testing.assert_allclose(sc2[s: s + lens[t]], score[a:b], rtol=0, atol=1e-9)
    assert (s2[~inside] == 9).all() and (sc2[~inside] == 7.0).all()


def test_non_monotone_offsets_rejected():
    """A table of negative length (bin_offsets going backwards) is an error in every entry that takes a layout."""
    import torch
    import ibdgem_b200 as ib
    off = np.array([0, 10, 5, 20], np.int64)
    lik = np.full((20, 3), 0.3)
    d_lik = torch.from_numpy(lik).cuda()
    d_out = torch.zeros((20, 3), dtype=torch.float64, device="cuda")
    d_state = torch.zeros(20, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros((3, 3), dtype=torch.int64, device="cuda")
    with ib.Engine(ib.Params()) as e:
        calls = {
            "hiddengem_viterbi_batch": lambda: e.viterbi_batch(lik, off),
            "hiddengem_viterbi_batch_device": lambda: e.viterbi_batch_device(d_lik.data_ptr(), off, False, d_state.data_ptr(),
                                                                             d_out.data_ptr(), d_cnt.data_ptr()),
            "hiddengem_posterior_batch": lambda: e.posterior_batch(lik, off),
            "hiddengem_posterior_batch_device": lambda: e.posterior_batch_device(d_lik.data_ptr(), off, False, d_out.data_ptr(),
                                                                                 d_cnt.data_ptr()),
        }
        for fn, call in calls.items():
            with pytest.raises(ib.EngineError, match=rf"{fn}\(\): table 1 has -5 bins"):
                call()
        # the engine is still usable
        state, _, counts = e.viterbi_batch(lik, [0, 10, 20])
        assert counts.sum() == 20
