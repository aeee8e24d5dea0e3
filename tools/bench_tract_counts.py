"""hiddengem posterior tract counts at C4 size (10,000 tables x 10,000 bins, the tables of tools/bench_posterior.py:
same generator and seed).  Prints one JSON line (and writes it to --out when given), with for each penalty set
(default, and p02 = 0, which runs the natural-log arithmetic):

  - device-resident time of hiddengem_tract_counts_device with and without the covariance of the tract counts, and of
    hiddengem_posterior_batch_device of this build, and with --parent-lib of another build of the library (e.g. the
    parent commit's): host clock around synchronised calls, warmed up, alternating over --reps repetitions;
  - the engine's per-kernel times (CUDA events) of each call, in a separate set of repetitions;
  - host-entry end-to-end time of hiddengem_tract_counts_batch from page-locked buffers, with and without the
    covariance;
  - the card's name and power limit, read in the same run.

`python tools/bench_tract_counts.py [--parent-lib PATH] --out FILE` on a GPU box."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


class OtherBuild:
    """hiddengem_posterior_batch_device of another build of libibdgem_b200.so, on its own engine."""

    def __init__(self, path):
        from ibdgem_b200.engine import _CParams
        self.lib = C.CDLL(os.path.abspath(path))
        self.lib.ibdgem_last_error.restype = C.c_char_p
        self.h = C.c_void_p()
        cp = _CParams(0.02, 20, 100, 0.0, 1.0, 0, 0)
        self._check(self.lib.ibdgem_engine_create(C.byref(cp), C.byref(self.h)))

    def _check(self, rc):
        if rc:
            raise RuntimeError(self.lib.ibdgem_last_error().decode())

    def posterior_device(self, d_lik, off, d_post, d_exp, p01, p02, p12):
        self._check(self.lib.hiddengem_posterior_batch_device(self.h, C.c_int32(len(off) - 1), off.ctypes.data_as(C.c_void_p), C.c_int64(0),
                                                              C.c_void_p(d_lik), C.c_int32(1), C.c_double(p01), C.c_double(p02),
                                                              C.c_double(p12), C.c_void_p(d_post), C.c_void_p(d_exp)))

    def close(self):
        self.lib.ibdgem_engine_destroy(self.h)


def stats(ts):
    return {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts)), "reps": len(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", type=int, default=10_000)
    ap.add_argument("--bins", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--parent-lib", default=None, help="another build of libibdgem_b200.so, timed alternately")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import ibdgem_b200 as ib
    if not torch.cuda.is_available():
        raise SystemExit("bench_tract_counts.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n_tables, n_bins = a.tables, a.bins
    nb = n_tables * n_bins
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=g, device=dev).repeat_interleave(200)[:nb]
    d_ll = torch.randn((nb, 3), generator=g, device=dev, dtype=torch.float64) * 10.0 - 150.0
    d_ll[torch.arange(nb, device=dev), seg] += 8.0  # planted IBD0/1/2 segments
    planted = torch.stack([(seg.view(n_tables, n_bins)[:, 0] == s) for s in range(3)], dim=1).double()
    runs_planted = planted + torch.stack([((seg.view(n_tables, n_bins)[:, 1:] == s) & (seg.view(n_tables, n_bins)[:, :-1] != s)).sum(dim=1)
                                          for s in range(3)], dim=1).double()
    del seg
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    d_post = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_post2 = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_exp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_exp2 = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_texp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_sw = torch.empty((n_tables, 3, 3), dtype=torch.float64, device=dev)
    d_tr = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_tc = torch.empty((n_tables, 3, 3), dtype=torch.float64, device=dev)
    d_sw2 = torch.empty((n_tables, 3, 3), dtype=torch.float64, device=dev)
    d_tr2 = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    h_ll = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
    h_ll.copy_(d_ll)
    h = [np.zeros(s) for s in ((n_tables, 3), (n_tables, 3, 3), (n_tables, 3), (n_tables, 3, 3))]
    other = OtherBuild(a.parent_lib) if a.parent_lib else None
    out = {"workload": "hiddengem posterior tract counts, C4: %d tables x %d bins of natural-log window scores "
                       "(tools/bench_posterior.py tables)" % (n_tables, n_bins), "card": card(),
           "torch_device": torch.cuda.get_device_name(dev), "runs": []}
    with ib.Engine(ib.Params(device=0)) as e:
        lib = e._lib
        for p01, p02, p12 in ((1e-3, 1e-6, 1e-3), (1e-3, 0.0, 1e-3)):
            pen = dict(p01=p01, p02=p02, p12=p12)

            def tc_cov():
                e.tract_counts_device(d_ll.data_ptr(), off, True, d_texp.data_ptr(), d_sw.data_ptr(), d_tr.data_ptr(), d_tc.data_ptr(), **pen)

            def tc_nocov():
                e.tract_counts_device(d_ll.data_ptr(), off, True, d_texp.data_ptr(), d_sw2.data_ptr(), d_tr2.data_ptr(), 0, **pen)

            def post():
                e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), **pen)

            def post_other():
                other.posterior_device(d_ll.data_ptr(), off, d_post2.data_ptr(), d_exp2.data_ptr(), p01, p02, p12)

            def host(with_cov):
                e._check(lib.hiddengem_tract_counts_batch(
                    e._h, C.c_int32(n_tables), off.ctypes.data_as(C.c_void_p), C.c_void_p(h_ll.data_ptr()), C.c_int32(1),
                    C.c_double(p01), C.c_double(p02), C.c_double(p12), *[x.ctypes.data_as(C.c_void_p) for x in h[:3]],
                    h[3].ctypes.data_as(C.c_void_p) if with_cov else None))

            calls = {"tract_counts_device_cov": tc_cov, "tract_counts_device_nocov": tc_nocov, "posterior_device": post}
            if other:
                calls["posterior_device_other_build"] = post_other
            for f in calls.values():
                f()
            times = {k: [] for k in calls}
            for _ in range(a.reps):  # alternating, host clock around synchronised calls (every entry synchronises)
                for k, f in calls.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    f()
                    times[k].append((time.perf_counter() - t0) * 1e3)
            same_mean = bool(torch.equal(d_texp, d_exp))
            same_without_cov = bool(torch.equal(d_sw, d_sw2) and torch.equal(d_tr, d_tr2))
            same_other = bool(torch.equal(d_post2, d_post) and torch.equal(d_exp2, d_exp)) if other else None
            e.enable_timing(True)
            kern = {}
            for k, f in calls.items():
                if k.endswith("other_build"):
                    continue
                e.reset_stats()
                for _ in range(a.reps):
                    f()
                kern[k] = {n: v[0] / a.reps for n, v in e.kernel_stats().items() if v[1]}
            e.enable_timing(False)
            th = {}
            for with_cov in (False, True):
                host(with_cov)
                ts = []
                for _ in range(max(3, a.reps // 3)):
                    t0 = time.perf_counter()
                    host(with_cov)
                    ts.append((time.perf_counter() - t0) * 1e3)
                th["with_cov" if with_cov else "without_cov"] = stats(ts)
            med = {k: float(np.median(v)) for k, v in times.items()}
            ksum = {k: sum(v.values()) for k, v in kern.items()}
            sd = torch.diagonal(d_tc, dim1=1, dim2=2).clamp(min=0).sqrt()
            run = {"penalties": pen,
                   "call_ms": {k: stats(v) for k, v in times.items()},
                   "kernels_ms": kern,
                   "cov_over_posterior": med["tract_counts_device_cov"] / med["posterior_device"],
                   "nocov_over_posterior": med["tract_counts_device_nocov"] / med["posterior_device"],
                   "cov_kernels_over_posterior_kernels": ksum["tract_counts_device_cov"] / ksum["posterior_device"],
                   "nocov_kernels_over_posterior_kernels": ksum["tract_counts_device_nocov"] / ksum["posterior_device"],
                   "host_entry_e2e_ms": th,
                   "means_equal_posterior_entry": same_mean,
                   "switches_tracts_equal_without_cov": same_without_cov,
                   "posterior_device_equal_to_other_build": same_other,
                   "finite": bool(torch.isfinite(d_tc).all() and torch.isfinite(d_tr).all() and torch.isfinite(d_sw).all()),
                   "median_tracts": [float(x) for x in d_tr.median(dim=0).values],
                   "median_planted_runs": [float(x) for x in runs_planted.median(dim=0).values],
                   "median_sd_tracts": [float(x) for x in sd.median(dim=0).values]}
            if other:
                run["posterior_this_over_other_build"] = med["posterior_device"] / med["posterior_device_other_build"]
            out["runs"].append(run)
    if other:
        other.close()
    out["buffers"] = "device-resident calls on torch allocations; host entry from page-locked buffers"
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
