"""score_ld / score_nonld where the path is chosen and where a call ends: a background that is nothing but the pileup's
own individual (no background member left, nU = 0) on both --LD path families, and a call that fails on too small a
max_windows, followed by a call on the same engine, on every scoring path (ld_path 0 = the general --LD kernels,
1 = ld_mma, 2 = ld_vmma), with the host score table in pageable and in page-locked memory."""
import numpy as np
import pytest

import ldterms as lt
import refcases

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("opt_v,path", [(0, 1), (1, 0)])
def test_background_of_only_the_pileup_individual(opt_v, path):
    """Every background entry is the reads' source, which never contributes: LIBD0 = LIBD1 = 0/0 in every window.
    Shared windows stay on ld_mma, which scores nU = 0 itself; per-target windows (-v) take the general path."""
    import enginecase as ec
    case = lt.ld_case(41, 1500, 12, 50, range(6), src=3, bg=[3, 3, 3], pu_idx=3, opt_v=opt_v)
    res = ec.run_engine(case, expanded=False)
    assert res[0]["ld_path"] == path
    for r, o in zip(res, refcases.oracle_run(case)):
        ec.assert_matches_oracle(r, o)
        assert r["n_windows"] > 0
        assert np.isnan(r["w_log"][:, :2]).all() and np.isfinite(r["w_log"][:, 2]).all()


PATHS = {  # entry, -v, force_general, ld_path
    "nonld_shared": ("nonld", 0, False, None),
    "nonld_v": ("nonld", 1, False, None),
    "ld_general": ("ld", 0, True, 0),
    "ld_mma": ("ld", 0, False, 1),
    "ld_vmma": ("ld", 1, False, 2),
}


def _engine(case, force_general):
    import ibdgem_b200 as ib
    pk, prm = case.pk, case.params
    e = ib.Engine(ib.Params(epsilon=prm.epsilon, max_cov=prm.max_cov, window_size=prm.window,
                            variable_sites_only=prm.opt_v))
    e.upload_sites(pk.pos, pk.n_ref, pk.n_alt, pk.host_keep)
    e.upload_panel(ib.pack_bits(pk.hap), len(pk.names))
    e.force_general_ld(force_general)
    return e


def _score(e, entry, case, max_windows, pinned):
    """One call through the C ABI with the score table w_loglik in pageable or page-locked host memory."""
    import torch
    from ibdgem_b200.engine import _CScores
    T = len(case.targets)
    out = dict(n_windows=np.zeros(T, np.int32), w_start=np.zeros((T, max_windows), np.uint64),
               w_end=np.zeros((T, max_windows), np.uint64), w_nsites=np.zeros((T, max_windows), np.int32))
    ll = torch.empty((T, max_windows, 3), dtype=torch.float64, pin_memory=pinned)
    cs = _CScores(max_windows, out["n_windows"].ctypes.data, out["w_start"].ctypes.data, out["w_end"].ctypes.data,
                  out["w_nsites"].ctypes.data, ll.data_ptr(), None, None, None, None, None, None, None, None)
    targets = np.asarray(case.targets, np.int32)
    if entry == "nonld":
        e.score_nonld_raw(targets, cs)
    else:
        e.score_ld_raw(targets, np.asarray(case.bg, np.int32), case.params.pu_idx, cs)
        out["ld_path"] = e.last_ld_path()
    out["w_loglik"] = ll.numpy().copy()
    return out


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("name", list(PATHS))
def test_failed_call_leaves_the_engine_reusable(name, pinned):
    """A call that returns an error has finished with the caller's buffers and leaves no state behind: the next call on
    the same engine gives what a fresh engine gives (integers exact, window sums to the parity bar of 1e-6)."""
    from ibdgem_b200 import EngineError
    entry, opt_v, force_general, path = PATHS[name]
    case = lt.ld_case(51, 3000, 40, 100, range(7), pu_idx=2, opt_v=opt_v)
    max_windows = 3000 // 100 + 2
    with _engine(case, force_general) as e:
        want = _score(e, entry, case, max_windows, pinned)
    with _engine(case, force_general) as e:
        with pytest.raises(EngineError, match="max_windows"):
            _score(e, entry, case, 2, pinned)
        assert e.last_ld_path() == -1  # set by a call that succeeded only
        got = _score(e, entry, case, max_windows, pinned)
    assert got.get("ld_path") == want.get("ld_path") == path
    assert (got["n_windows"] > 2).all()
    for k in ("n_windows", "w_start", "w_end", "w_nsites"):
        np.testing.assert_array_equal(got[k], want[k])
    a, b = got["w_loglik"], want["w_loglik"]
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_allclose(a[~np.isnan(a)], b[~np.isnan(b)], rtol=0, atol=1e-6)
