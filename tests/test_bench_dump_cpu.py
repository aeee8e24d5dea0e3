"""bench.py --dump-outputs: what is written (only the windows each target has, all finite) and the 64 MB bound."""
import os

import numpy as np

import bench


def _results(T, maxW, seed=0):
    """Result buffers as the score call leaves them: slots past a target's n_windows hold whatever was there."""
    rng = np.random.default_rng(seed)
    nw = rng.integers(maxW - 3, maxW + 1, T).astype(np.int32)
    ws = rng.integers(0, 10 ** 8, (T, maxW)).astype(np.int64)
    ll = rng.random((T, maxW, 3))
    past = np.arange(maxW)[None, :] >= nw[:, None]
    ll[past] = np.nan
    return np.arange(T, dtype=np.int32), nw, ws, ws + 59, np.full((T, maxW), 1000, np.int32), ll


def _load(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}


def _size(path):
    return sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def test_dump_writes_the_windows_of_every_target_in_order(tmp_path):
    targets, nw, ws, we, wn, ll = _results(50, 40)
    bench.dump_outputs(str(tmp_path), targets, nw, ws, we, wn, ll)
    assert sorted(os.listdir(tmp_path)) == [f"{n}.npy" for n in ("n_windows", "targets", "w_end", "w_loglik", "w_nsites", "w_start")]
    got = _load(tmp_path)
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in got.values())
    np.testing.assert_array_equal(got["targets"], targets)
    np.testing.assert_array_equal(got["n_windows"], nw)
    assert got["w_start"].shape == (nw.sum(),) and got["w_loglik"].shape == (nw.sum(), 3)
    off = np.concatenate([[0], np.cumsum(nw)])
    for k in range(len(targets)):
        n, sl = nw[k], slice(off[k], off[k + 1])
        np.testing.assert_array_equal(got["w_start"][sl], ws[k, :n])
        np.testing.assert_array_equal(got["w_end"][sl], we[k, :n])
        np.testing.assert_array_equal(got["w_nsites"][sl], wn[k, :n])
        np.testing.assert_array_equal(got["w_loglik"][sl], ll[k, :n])


def test_dump_of_a_large_result_is_a_fixed_sample_under_64_mb(tmp_path):
    targets, nw, ws, we, wn, ll = _results(3000, 1002)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), targets, nw, ws, we, wn, ll)
        assert _size(tmp_path / d) < 64_000_000
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    rows = a["targets"].astype(int)
    assert 1000 < len(rows) < 3000 and (np.diff(rows) > 0).all()
    assert all(np.array_equal(a[k], b[k]) and np.isfinite(a[k]).all() for k in a)
    np.testing.assert_array_equal(a["n_windows"], nw[rows])
    np.testing.assert_array_equal(a["w_loglik"][: nw[rows[0]]], ll[rows[0], : nw[rows[0]]])
