"""hiddengem posterior moments at C4 size (10,000 tables x 10,000 bins, the tables of tools/bench_posterior.py: same
generator and seed).  Prints one JSON line (and writes it to --out when given), with for each penalty set (default,
and p02 = 0, which runs the natural-log arithmetic):

  - device-resident time of hiddengem_posterior_moments_device (no per-bin posteriors) and of
    hiddengem_posterior_batch_device of this build, and with --parent-lib of another build of the library (e.g. the
    parent commit's): host clock around synchronised calls, warmed up, alternating over --reps repetitions;
  - the engine's per-kernel times (CUDA events) of both calls, in a separate set of repetitions;
  - host-entry end-to-end time of hiddengem_posterior_moments_batch from page-locked buffers, with and without
    per-bin posteriors;
  - the card's name and power limit, read in the same run.

`python tools/bench_moments.py [--parent-lib PATH] --out FILE` on a GPU box."""
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
        raise SystemExit("bench_moments.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n_tables, n_bins = a.tables, a.bins
    nb = n_tables * n_bins
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=g, device=dev).repeat_interleave(200)[:nb]
    d_ll = torch.randn((nb, 3), generator=g, device=dev, dtype=torch.float64) * 10.0 - 150.0
    d_ll[torch.arange(nb, device=dev), seg] += 8.0  # planted IBD0/1/2 segments
    del seg
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    d_post = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_post2 = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_exp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_exp2 = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_mexp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_cov = torch.empty((n_tables, 3, 3), dtype=torch.float64, device=dev)
    h_ll = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
    h_ll.copy_(d_ll)
    h_post = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
    h_exp = np.zeros((n_tables, 3))
    h_cov = np.zeros((n_tables, 3, 3))
    other = OtherBuild(a.parent_lib) if a.parent_lib else None
    out = {"workload": "hiddengem posterior moments, C4: %d tables x %d bins of natural-log window scores (tools/bench_posterior.py "
                       "tables)" % (n_tables, n_bins), "card": card(), "torch_device": torch.cuda.get_device_name(dev), "runs": []}
    with ib.Engine(ib.Params(device=0)) as e:
        lib = e._lib
        for p01, p02, p12 in ((1e-3, 1e-6, 1e-3), (1e-3, 0.0, 1e-3)):
            pen = dict(p01=p01, p02=p02, p12=p12)

            def mom():
                e.posterior_moments_device(d_ll.data_ptr(), off, True, d_mexp.data_ptr(), d_cov.data_ptr(), **pen)

            def post():
                e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), **pen)

            def post_other():
                other.posterior_device(d_ll.data_ptr(), off, d_post2.data_ptr(), d_exp2.data_ptr(), p01, p02, p12)

            def host(with_post):
                e._check(lib.hiddengem_posterior_moments_batch(
                    e._h, C.c_int32(n_tables), off.ctypes.data_as(C.c_void_p), C.c_void_p(h_ll.data_ptr()), C.c_int32(1),
                    C.c_double(p01), C.c_double(p02), C.c_double(p12), C.c_void_p(h_post.data_ptr() if with_post else None),
                    h_exp.ctypes.data_as(C.c_void_p), h_cov.ctypes.data_as(C.c_void_p)))

            calls = {"moments_device": mom, "posterior_device": post}
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
            same_mean = bool(torch.equal(d_mexp, d_exp))
            same_other = bool(torch.equal(d_post2, d_post) and torch.equal(d_exp2, d_exp)) if other else None
            e.enable_timing(True)
            kern = {}
            for k, f in (("moments_device", mom), ("posterior_device", post)):
                e.reset_stats()
                for _ in range(a.reps):
                    f()
                kern[k] = {n: v[0] / a.reps for n, v in e.kernel_stats().items() if v[1]}
            e.enable_timing(False)
            th = {}
            for with_post in (False, True):
                host(with_post)
                ts = []
                for _ in range(max(3, a.reps // 3)):
                    t0 = time.perf_counter()
                    host(with_post)
                    ts.append((time.perf_counter() - t0) * 1e3)
                th["with_posteriors" if with_post else "without_posteriors"] = stats(ts)
            cov = torch.from_numpy(h_cov)
            run = {"penalties": pen,
                   "call_ms": {k: stats(v) for k, v in times.items()},
                   "kernels_ms": kern,
                   "moments_over_posterior": float(np.median(times["moments_device"]) / np.median(times["posterior_device"])),
                   "moments_kernels_over_posterior_kernels": sum(kern["moments_device"].values()) / sum(kern["posterior_device"].values()),
                   "host_entry_e2e_ms": th,
                   "means_equal_posterior_entry": same_mean,
                   "posterior_device_equal_to_other_build": same_other,
                   "cov_finite": bool(torch.isfinite(cov).all()),
                   "median_sd_bins": [float(x) for x in torch.diagonal(cov, dim1=1, dim2=2).clamp(min=0).sqrt().median(dim=0).values]}
            if other:
                run["posterior_this_over_other_build"] = float(np.median(times["posterior_device"]) / np.median(times["posterior_device_other_build"]))
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
