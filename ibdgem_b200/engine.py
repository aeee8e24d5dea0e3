"""Python mirror of the C ABI in include/ibdgem_b200.h (same names, argument meaning and error
behaviour).  Every method is one ABI call; arrays are numpy host buffers unless stated."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from ._lib import load_library


class EngineError(RuntimeError):
    pass


class _CParams(C.Structure):
    _fields_ = [("epsilon", C.c_double), ("max_cov", C.c_uint32), ("window_size", C.c_int32),
                ("min_af", C.c_double), ("max_af", C.c_double), ("variable_sites_only", C.c_int32),
                ("device", C.c_int32)]


class _CScores(C.Structure):
    _fields_ = [("max_windows", C.c_int32), ("n_windows", C.c_void_p), ("w_start", C.c_void_p),
                ("w_end", C.c_void_p), ("w_nsites", C.c_void_p), ("w_loglik", C.c_void_p),
                ("processed", C.c_void_p), ("skipped", C.c_void_p), ("final_total_cov", C.c_void_p),
                ("final_dist", C.c_void_p), ("site_status", C.c_void_p), ("site_lik", C.c_void_p),
                ("w_lik_linear", C.c_void_p), ("w_loglik_device", C.c_void_p)]


@dataclass
class Params:
    """ibdgem_params: the option statics of src/ibdgem.c:21-38 the arithmetic reads."""
    epsilon: float = 0.02
    max_cov: int = 20
    window_size: int = 100
    min_af: float = 0.0
    max_af: float = 1.0
    variable_sites_only: int = 0
    device: int = 0


@dataclass
class Scores:
    """Host copies of an ibdgem_scores result for T targets."""
    n_windows: np.ndarray
    w_start: np.ndarray
    w_end: np.ndarray
    w_nsites: np.ndarray
    w_loglik: np.ndarray
    processed: np.ndarray
    skipped: np.ndarray
    final_total_cov: np.ndarray
    final_dist: np.ndarray
    site_status: np.ndarray | None = None
    site_lik: np.ndarray | None = None
    w_lik_linear: np.ndarray | None = None
    extra: dict = field(default_factory=dict)


# hiddengem_tract (include/ibdgem_b200.h): one IBD tract, a maximal run of one Viterbi state within a table
TRACT_DTYPE = np.dtype([("first_bin", "<i8"), ("n_bins", "<i8"), ("state", "<i4"), ("reserved", "<i4"),
                        ("loglik", "<f8", (3,)), ("post_mean", "<f8"), ("post_min", "<f8")])
assert TRACT_DTYPE.itemsize == 64


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Engine:
    def __init__(self, params: Params):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.params = params
        cp = _CParams(params.epsilon, params.max_cov, params.window_size, params.min_af, params.max_af,
                      params.variable_sites_only, params.device)
        self._check(self._lib.ibdgem_engine_create(C.byref(cp), C.byref(self._h)))
        self.S = 0
        self.N = 0

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise EngineError(self._lib.ibdgem_last_error().decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.ibdgem_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.ibdgem_engine_set_stream(self._h, C.c_void_p(cuda_stream)))

    # -- inputs -----------------------------------------------------------------------------
    def upload_sites(self, pos, n_ref, n_alt, host_keep, af_user=None):
        self._sites = (np.ascontiguousarray(pos, np.uint64), np.ascontiguousarray(n_ref, np.uint8),
                       np.ascontiguousarray(n_alt, np.uint8), np.ascontiguousarray(host_keep, np.uint8),
                       None if af_user is None else np.ascontiguousarray(af_user, np.float64))
        p, r, a, k, u = self._sites
        self.S = len(p)
        self._check(self._lib.ibdgem_engine_upload_sites(self._h, C.c_int64(self.S), _ptr(p), _ptr(r), _ptr(a),
                                                         _ptr(k), _ptr(u)))

    def upload_panel(self, bits: np.ndarray, n_indiv: int):
        bits = np.ascontiguousarray(bits, np.uint32)
        self._bits = bits
        self.N = int(n_indiv)
        self._check(self._lib.ibdgem_engine_upload_panel(self._h, C.c_int64(bits.shape[0]), C.c_int32(n_indiv),
                                                         _ptr(bits), C.c_int64(bits.shape[1])))

    def clone_panel(self, src: "Engine"):
        """Panel copied device to device from another engine of this process (ibdgem_engine_clone_panel)."""
        self._bits = None
        self.N = src.N
        self._check(self._lib.ibdgem_engine_clone_panel(self._h, src._h))

    def set_panel_device(self, d_bits_ptr: int, n_sites: int, n_indiv: int, words_per_site: int):
        """Panel rows live in caller-owned device memory (see shard.replicate_panel); declare them
        readable piece by piece with panel_rows_ready()."""
        self._bits = None
        self.N = int(n_indiv)
        self._check(self._lib.ibdgem_engine_set_panel_device(self._h, C.c_int64(n_sites), C.c_int32(n_indiv),
                                                             C.c_void_p(d_bits_ptr), C.c_int64(words_per_site)))

    def panel_rows_ready(self, row_end: int, stream: int = 0):
        self._check(self._lib.ibdgem_engine_panel_rows_ready(self._h, C.c_int64(row_end), C.c_void_p(stream or None)))

    def set_window_shard(self, index: int, count: int):
        """Multi-GPU partition by windows (shared window maps): see include/ibdgem_b200.h."""
        self._check(self._lib.ibdgem_engine_set_window_shard(self._h, C.c_int32(index), C.c_int32(count)))

    def set_shard_compact_output(self, on: bool = True):
        """Window shards: the host score table is written as [T][shard windows][3] (one contiguous copy)."""
        self._check(self._lib.ibdgem_engine_set_shard_compact_output(self._h, C.c_int32(1 if on else 0)))

    def window_shard(self):
        """(w_begin, w_end, site_begin, site_end) of this engine's shard; prepares the window map."""
        wb, we, sb, se = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int64()
        self._check(self._lib.ibdgem_engine_window_shard(self._h, C.byref(wb), C.byref(we), C.byref(sb), C.byref(se)))
        return wb.value, we.value, sb.value, se.value

    def sync_uploads(self):
        self._check(self._lib.ibdgem_engine_sync_uploads(self._h))

    def prepare(self):
        self._check(self._lib.ibdgem_engine_prepare(self._h))

    def invalidate(self):
        self._check(self._lib.ibdgem_engine_invalidate(self._h))

    def get_site_table(self):
        f = np.zeros(self.S)
        st = np.zeros(self.S, np.uint8)
        lik7 = np.zeros((self.S, 7))
        self._check(self._lib.ibdgem_engine_get_site_table(self._h, _ptr(f), _ptr(st), _ptr(lik7)))
        return f, st, lik7

    # -- scoring ----------------------------------------------------------------------------
    def _alloc_scores(self, T, max_windows, expanded, device_out, linear=False):
        C_ = self.params.max_cov + 1
        s = Scores(np.zeros(T, np.int32), np.zeros((T, max_windows), np.uint64),
                   np.zeros((T, max_windows), np.uint64), np.zeros((T, max_windows), np.int32),
                   np.full((T, max_windows, 3), np.nan), np.zeros(T, np.uint64), np.zeros(T, np.uint64),
                   np.zeros(T, np.uint64), np.zeros((T, C_), np.uint64))
        if expanded:
            s.site_status = np.zeros((T, self.S), np.uint8)
            s.site_lik = np.zeros((T, self.S, 3))
        if linear:
            s.w_lik_linear = np.full((T, max_windows, 3), np.nan)
        cs = _CScores(max_windows, _ptr(s.n_windows), _ptr(s.w_start), _ptr(s.w_end), _ptr(s.w_nsites),
                      _ptr(s.w_loglik), _ptr(s.processed), _ptr(s.skipped), _ptr(s.final_total_cov),
                      _ptr(s.final_dist), _ptr(s.site_status), _ptr(s.site_lik), _ptr(s.w_lik_linear),
                      C.c_void_p(device_out) if device_out else None)
        return s, cs

    def default_max_windows(self):
        return self.S // max(self.params.window_size, 1) + 2

    def score_nonld(self, targets, tgt_counts=None, max_windows=None, expanded=False, device_out=0, linear=False) -> Scores:
        targets = np.ascontiguousarray(targets, np.int32)
        T = len(targets)
        s, cs = self._alloc_scores(T, max_windows or self.default_max_windows(), expanded, device_out, linear)
        tc = None if tgt_counts is None else np.ascontiguousarray(tgt_counts, np.uint8)
        self._check(self._lib.ibdgem_engine_score_nonld(self._h, C.c_int32(T), _ptr(targets), _ptr(tc), C.byref(cs)))
        return s

    def score_ld(self, targets, bg, pu_idx=-1, tgt_counts=None, max_windows=None, expanded=False,
                 device_out=0, linear=False) -> Scores:
        targets = np.ascontiguousarray(targets, np.int32)
        bg = np.ascontiguousarray(bg, np.int32)
        T = len(targets)
        s, cs = self._alloc_scores(T, max_windows or self.default_max_windows(), expanded, device_out, linear)
        tc = None if tgt_counts is None else np.ascontiguousarray(tgt_counts, np.uint8)
        self._check(self._lib.ibdgem_engine_score_ld(self._h, C.c_int32(T), _ptr(targets), C.c_int32(len(bg)),
                                                     _ptr(bg), C.c_int32(pu_idx), _ptr(tc), C.byref(cs)))
        s.extra["ld_path"] = self._lib.ibdgem_engine_last_ld_path(self._h)
        return s

    def score_ld_raw(self, targets: np.ndarray, bg: np.ndarray, pu_idx: int, cs: "_CScores"):
        """Lowest-overhead form for benchmarking: caller owns the ibdgem_scores struct."""
        self._check(self._lib.ibdgem_engine_score_ld(self._h, C.c_int32(len(targets)), _ptr(targets),
                                                     C.c_int32(len(bg)), _ptr(bg), C.c_int32(pu_idx), None,
                                                     C.byref(cs)))

    def score_nonld_raw(self, targets: np.ndarray, cs: "_CScores"):
        self._check(self._lib.ibdgem_engine_score_nonld(self._h, C.c_int32(len(targets)), _ptr(targets), None,
                                                        C.byref(cs)))

    def force_general_ld(self, on: bool):
        self._check(self._lib.ibdgem_engine_force_general_ld(self._h, C.c_int(1 if on else 0)))

    def last_ld_path(self) -> int:
        return self._lib.ibdgem_engine_last_ld_path(self._h)

    # -- hiddengem --------------------------------------------------------------------------
    def viterbi_batch(self, lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3):
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        nb = int(off[-1])
        state = np.zeros(nb, np.uint8)
        score = np.zeros((nb, 3))
        counts = np.zeros((nt, 3), np.int64)
        self._check(self._lib.hiddengem_viterbi_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik),
                                                      C.c_int32(1 if is_log else 0), C.c_double(p01),
                                                      C.c_double(p02), C.c_double(p12), _ptr(state), _ptr(score),
                                                      _ptr(counts)))
        return state, score, counts

    def viterbi_batch_raw(self, lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, state_ptr: int, score_ptr: int,
                          counts_ptr: int, p01=1e-3, p02=1e-6, p12=1e-3):
        """Caller-owned HOST buffers by address (pinned for asynchronous copies)."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        self._check(self._lib.hiddengem_viterbi_batch(self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_void_p(lik_ptr),
                                                      C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02),
                                                      C.c_double(p12), C.c_void_p(state_ptr), C.c_void_p(score_ptr),
                                                      C.c_void_p(counts_ptr)))

    def viterbi_batch_device(self, d_lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, d_state_ptr: int, d_score_ptr: int,
                             d_counts_ptr: int, table_stride: int = 0, p01=1e-3, p02=1e-6, p12=1e-3):
        """Device buffers in, device buffers out (hiddengem_viterbi_batch_device); bin_offsets stays on the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        self._check(self._lib.hiddengem_viterbi_batch_device(
            self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_int64(table_stride), C.c_void_p(d_lik_ptr),
            C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02), C.c_double(p12), C.c_void_p(d_state_ptr),
            C.c_void_p(d_score_ptr), C.c_void_p(d_counts_ptr)))

    def posterior_batch(self, lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3):
        """Per-bin posterior IBD-state probabilities over the path weights hiddengem maximises
        (hiddengem_posterior_batch): (posterior [n_bins, 3], expected [n_tables, 3])."""
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        post = np.zeros((int(off[-1]), 3))
        expected = np.zeros((nt, 3))
        self._check(self._lib.hiddengem_posterior_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik),
                                                        C.c_int32(1 if is_log else 0), C.c_double(p01),
                                                        C.c_double(p02), C.c_double(p12), _ptr(post), _ptr(expected)))
        return post, expected

    def posterior_batch_device(self, d_lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, d_posterior_ptr: int,
                               d_expected_ptr: int, table_stride: int = 0, p01=1e-3, p02=1e-6, p12=1e-3):
        """Device buffers in, device buffers out (hiddengem_posterior_batch_device); bin_offsets stays on the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        self._check(self._lib.hiddengem_posterior_batch_device(
            self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_int64(table_stride), C.c_void_p(d_lik_ptr),
            C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02), C.c_double(p12),
            C.c_void_p(d_posterior_ptr), C.c_void_p(d_expected_ptr)))

    def posterior_moments_batch(self, lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3, posterior=False):
        """Posterior mean and covariance of the bins per IBD state (hiddengem_posterior_moments_batch): (expected
        [n_tables, 3], cov [n_tables, 3, 3]), and with posterior=True also the per-bin posteriors [n_bins, 3]."""
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        post = np.zeros((int(off[-1]), 3)) if posterior else None
        expected = np.zeros((nt, 3))
        cov = np.zeros((nt, 3, 3))
        self._check(self._lib.hiddengem_posterior_moments_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik),
                                                                C.c_int32(1 if is_log else 0), C.c_double(p01),
                                                                C.c_double(p02), C.c_double(p12), _ptr(post), _ptr(expected),
                                                                _ptr(cov)))
        return (expected, cov, post) if posterior else (expected, cov)

    def posterior_moments_device(self, d_lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, d_expected_ptr: int,
                                 d_cov_ptr: int, d_posterior_ptr: int = 0, table_stride: int = 0, p01=1e-3, p02=1e-6,
                                 p12=1e-3):
        """Device buffers in, device buffers out (hiddengem_posterior_moments_device; d_posterior_ptr 0: none);
        bin_offsets stays on the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        self._check(self._lib.hiddengem_posterior_moments_device(
            self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_int64(table_stride), C.c_void_p(d_lik_ptr),
            C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02), C.c_double(p12),
            C.c_void_p(d_posterior_ptr or None), C.c_void_p(d_expected_ptr), C.c_void_p(d_cov_ptr)))

    def tract_counts_batch(self, lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3, cov=True):
        """Posterior expected switches between IBD states and IBD tracts per state (hiddengem_tract_counts_batch):
        (expected [n_tables, 3], switches [n_tables, 3, 3], tracts [n_tables, 3]), and with cov=True also the
        covariance of the tract counts [n_tables, 3, 3]."""
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        expected = np.zeros((nt, 3))
        switches = np.zeros((nt, 3, 3))
        tracts = np.zeros((nt, 3))
        tract_cov = np.zeros((nt, 3, 3)) if cov else None
        self._check(self._lib.hiddengem_tract_counts_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik),
                                                           C.c_int32(1 if is_log else 0), C.c_double(p01),
                                                           C.c_double(p02), C.c_double(p12), _ptr(expected),
                                                           _ptr(switches), _ptr(tracts), _ptr(tract_cov)))
        return (expected, switches, tracts, tract_cov) if cov else (expected, switches, tracts)

    def tract_counts_device(self, d_lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, d_expected_ptr: int,
                            d_switches_ptr: int, d_tracts_ptr: int, d_tract_cov_ptr: int = 0, table_stride: int = 0,
                            p01=1e-3, p02=1e-6, p12=1e-3):
        """Device buffers in, device buffers out (hiddengem_tract_counts_device; d_tract_cov_ptr 0: no covariance);
        bin_offsets stays on the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        self._check(self._lib.hiddengem_tract_counts_device(
            self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_int64(table_stride), C.c_void_p(d_lik_ptr),
            C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02), C.c_double(p12),
            C.c_void_p(d_expected_ptr), C.c_void_p(d_switches_ptr), C.c_void_p(d_tracts_ptr),
            C.c_void_p(d_tract_cov_ptr or None)))

    def tract_lengths_batch(self, lik, bin_offsets, thresholds, start=None, end=None, is_log=False, p01=1e-3, p02=1e-6,
                            p12=1e-3):
        """Posterior expected number of runs of each IBD state at least each threshold long
        (hiddengem_tract_lengths_batch): [n_tables, len(thresholds), 3].  With start / end (per bin, packed like lik)
        lengths are end[J] - start[i] + 1, otherwise bins."""
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        th = np.ascontiguousarray(thresholds, np.uint64)
        nt = len(off) - 1
        st = None if start is None else np.ascontiguousarray(start, np.uint64)
        en = None if end is None else np.ascontiguousarray(end, np.uint64)
        spectrum = np.zeros((nt, len(th), 3))
        self._check(self._lib.hiddengem_tract_lengths_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik),
                                                            C.c_int32(1 if is_log else 0), C.c_double(p01),
                                                            C.c_double(p02), C.c_double(p12), _ptr(st), _ptr(en),
                                                            C.c_int32(len(th)), _ptr(th), _ptr(spectrum)))
        return spectrum

    def tract_lengths_device(self, d_lik_ptr: int, bin_offsets: np.ndarray, is_log: bool, thresholds, d_spectrum_ptr: int,
                             d_start_ptr: int = 0, d_end_ptr: int = 0, table_stride: int = 0, p01=1e-3, p02=1e-6,
                             p12=1e-3):
        """Device buffers in, device buffers out (hiddengem_tract_lengths_device; d_start_ptr / d_end_ptr 0: lengths
        in bins); bin_offsets and thresholds stay on the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        th = np.ascontiguousarray(thresholds, np.uint64)
        self._check(self._lib.hiddengem_tract_lengths_device(
            self._h, C.c_int32(len(off) - 1), _ptr(off), C.c_int64(table_stride), C.c_void_p(d_lik_ptr),
            C.c_int32(1 if is_log else 0), C.c_double(p01), C.c_double(p02), C.c_double(p12),
            C.c_void_p(d_start_ptr or None), C.c_void_p(d_end_ptr or None), C.c_int32(len(th)), _ptr(th),
            C.c_void_p(d_spectrum_ptr)))

    def tracts_batch(self, lik, bin_offsets, is_log=False, p01=1e-3, p02=1e-6, p12=1e-3, posterior=True):
        """IBD tracts (runs of one Viterbi state) with likelihood sums and, with posterior, the mean and minimum
        posterior of their state (hiddengem_tracts_batch + hiddengem_last_tracts): (tract_offsets [n_tables + 1],
        tracts, a TRACT_DTYPE array)."""
        lik = np.ascontiguousarray(lik, np.float64)
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        toff = np.zeros(nt + 1, np.int64)
        self._check(self._lib.hiddengem_tracts_batch(self._h, C.c_int32(nt), _ptr(off), _ptr(lik), C.c_int32(1 if is_log else 0),
                                                     C.c_double(p01), C.c_double(p02), C.c_double(p12),
                                                     C.c_int32(1 if posterior else 0), _ptr(toff)))
        return toff, self.last_tracts(toff[-1])

    def tracts_device(self, d_lik_ptr: int, bin_offsets, is_log: bool, d_state_ptr: int, d_posterior_ptr: int = 0,
                      table_stride: int = 0):
        """Tracts of device states (and posteriors, 0: none) (hiddengem_tracts_device); bin_offsets stays on the host.
        Returns (tract_offsets, tracts) copied to the host."""
        off = np.ascontiguousarray(bin_offsets, np.int64)
        nt = len(off) - 1
        toff = np.zeros(nt + 1, np.int64)
        self._check(self._lib.hiddengem_tracts_device(self._h, C.c_int32(nt), _ptr(off), C.c_int64(table_stride),
                                                      C.c_void_p(d_lik_ptr), C.c_int32(1 if is_log else 0),
                                                      C.c_void_p(d_state_ptr), C.c_void_p(d_posterior_ptr or None), _ptr(toff)))
        return toff, self.last_tracts(toff[-1])

    def last_tracts(self, n: int):
        """The n records of the last successful tract call (hiddengem_last_tracts), as a TRACT_DTYPE array."""
        tracts = np.zeros(max(int(n), 1), TRACT_DTYPE)
        self._check(self._lib.hiddengem_last_tracts(self._h, _ptr(tracts), C.c_int32(0)))
        return tracts[: int(n)]

    def viterbi_last_flagged(self) -> int:
        """Tables of the last hiddengem call re-evaluated on the host in long double (near-tie guard)."""
        return int(self._lib.hiddengem_last_flagged(self._h))

    # -- instrumentation --------------------------------------------------------------------
    def enable_timing(self, on=True):
        self._check(self._lib.ibdgem_engine_enable_timing(self._h, C.c_int(1 if on else 0)))

    def reset_stats(self):
        self._check(self._lib.ibdgem_engine_reset_stats(self._h))

    def kernel_stats(self) -> dict:
        out = {}
        name = C.create_string_buffer(64)
        ms = C.c_double()
        n = C.c_int64()
        for k in range(self._lib.ibdgem_engine_num_kernels(self._h)):
            self._check(self._lib.ibdgem_engine_kernel_stats(self._h, C.c_int32(k), name, C.c_int32(64),
                                                             C.byref(ms), C.byref(n)))
            out[name.value.decode()] = (ms.value, n.value)
        return out

    def device_bytes(self) -> int:
        return int(self._lib.ibdgem_engine_device_bytes(self._h))
