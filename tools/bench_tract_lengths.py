"""hiddengem posterior tract-length spectrum at C4 size (10,000 tables x 10,000 bins, the tables of
tools/bench_posterior.py and tools/bench_tract_counts.py: same generator and seed, 200-bin planted blocks).  Prints one
JSON line (and writes it to --out when given), with for each penalty set (default, and p02 = 0, which runs the
natural-log arithmetic) and each of K = 1 and K = 8 thresholds, in bins and with coordinates (bin i of every table
spans [5000 i + 1, 5000 i + 5000] bp, so X bins are 5000 X bp):

  - device-resident time of hiddengem_tract_lengths_device, alternating with hiddengem_tract_counts_device without the
    covariance: host clock around synchronised calls, warmed up, over --reps repetitions;
  - the engine's per-kernel times (CUDA events) of each call, in a separate set of repetitions;
  - host-entry end-to-end time of hiddengem_tract_lengths_batch from page-locked buffers;
  - the mean E[R_s(X)] per table at X = 50 and 100 bins beside the mean number of planted runs at least that long
    (a reported figure, not a check);
  - the card's name and power limit, read in the same run.

`python tools/bench_tract_lengths.py --out FILE` on a GPU box."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tools.bench_tract_counts import card, stats  # noqa: E402

BP = 5000  # bp per bin of the coordinate runs
THRESHOLDS = {1: [100], 8: [1, 10, 25, 50, 100, 150, 200, 400]}  # bins


def planted_runs_at_least(seg, xs):
    """Mean over tables of the number of maximal planted runs of each state at least x bins long, [len(xs), 3]."""
    import torch
    T, n = seg.shape
    head = torch.ones_like(seg, dtype=torch.bool)
    head[:, 1:] = seg[:, 1:] != seg[:, :-1]
    idx = torch.nonzero(head.flatten()).flatten()
    ends = torch.cat([idx[1:], torch.tensor([T * n], device=seg.device)])
    tab = idx // n
    ends = torch.minimum(ends, (tab + 1) * n)  # runs stop at table ends
    length = ends - idx
    state = seg.flatten()[idx]
    return [[float(((length >= x) & (state == s)).sum()) / T for s in range(3)] for x in xs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", type=int, default=10_000)
    ap.add_argument("--bins", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import ibdgem_b200 as ib
    if not torch.cuda.is_available():
        raise SystemExit("bench_tract_lengths.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n_tables, n_bins = a.tables, a.bins
    nb = n_tables * n_bins
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=g, device=dev).repeat_interleave(200)[:nb]
    d_ll = torch.randn((nb, 3), generator=g, device=dev, dtype=torch.float64) * 10.0 - 150.0
    d_ll[torch.arange(nb, device=dev), seg] += 8.0  # planted IBD0/1/2 segments
    planted = planted_runs_at_least(seg.view(n_tables, n_bins), [50, 100])
    del seg
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    pos = torch.arange(n_bins, device=dev, dtype=torch.int64).repeat(n_tables)
    d_bs = pos * BP + 1  # int64: the same bits as the uint64 coordinates the entries take
    d_be = pos * BP + BP
    del pos
    h_ll = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
    h_ll.copy_(d_ll)
    h_bs = torch.empty(nb, dtype=torch.int64, pin_memory=True)
    h_be = torch.empty(nb, dtype=torch.int64, pin_memory=True)
    h_bs.copy_(d_bs)
    h_be.copy_(d_be)
    d_texp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_sw = torch.empty((n_tables, 3, 3), dtype=torch.float64, device=dev)
    d_tr = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    out = {"workload": "hiddengem posterior tract lengths, C4: %d tables x %d bins of natural-log window scores "
                       "(tools/bench_posterior.py tables; coordinates %d bp per bin)" % (n_tables, n_bins, BP), "card": card(),
           "torch_device": torch.cuda.get_device_name(dev), "runs": []}
    with ib.Engine(ib.Params(device=0)) as e:
        lib = e._lib
        for p01, p02, p12 in ((1e-3, 1e-6, 1e-3), (1e-3, 0.0, 1e-3)):
            pen = dict(p01=p01, p02=p02, p12=p12)
            for K, xs in THRESHOLDS.items():
                for coords in (False, True):
                    th = np.array([x * BP if coords else x for x in xs], np.uint64)
                    d_spec = torch.empty((n_tables, K, 3), dtype=torch.float64, device=dev)
                    h_spec = np.zeros((n_tables, K, 3))

                    def tl():
                        e.tract_lengths_device(d_ll.data_ptr(), off, True, th, d_spec.data_ptr(), d_bs.data_ptr() if coords else 0,
                                               d_be.data_ptr() if coords else 0, **pen)

                    def tc():
                        e.tract_counts_device(d_ll.data_ptr(), off, True, d_texp.data_ptr(), d_sw.data_ptr(), d_tr.data_ptr(), 0, **pen)

                    def host():
                        e._check(lib.hiddengem_tract_lengths_batch(
                            e._h, C.c_int32(n_tables), off.ctypes.data_as(C.c_void_p), C.c_void_p(h_ll.data_ptr()), C.c_int32(1),
                            C.c_double(p01), C.c_double(p02), C.c_double(p12), C.c_void_p(h_bs.data_ptr() if coords else None),
                            C.c_void_p(h_be.data_ptr() if coords else None), C.c_int32(K), th.ctypes.data_as(C.c_void_p),
                            h_spec.ctypes.data_as(C.c_void_p)))

                    calls = {"tract_lengths_device": tl, "tract_counts_device_nocov": tc}
                    for f in calls.values():
                        f()
                    times = {k: [] for k in calls}
                    for _ in range(a.reps):  # alternating, host clock around synchronised calls (every entry synchronises)
                        for k, f in calls.items():
                            torch.cuda.synchronize()
                            t0 = time.perf_counter()
                            f()
                            times[k].append((time.perf_counter() - t0) * 1e3)
                    e.enable_timing(True)
                    kern = {}
                    for k, f in calls.items():
                        e.reset_stats()
                        for _ in range(a.reps):
                            f()
                        kern[k] = {n: v[0] / a.reps for n, v in e.kernel_stats().items() if v[1]}
                    e.enable_timing(False)
                    host()
                    ts = []
                    for _ in range(max(3, a.reps // 3)):
                        t0 = time.perf_counter()
                        host()
                        ts.append((time.perf_counter() - t0) * 1e3)
                    spec = d_spec.cpu().numpy()
                    med = {k: float(np.median(v)) for k, v in times.items()}
                    run = {"penalties": pen, "K": K, "lengths": "bp" if coords else "bins", "thresholds": [int(x) for x in th],
                           "call_ms": {k: stats(v) for k, v in times.items()},
                           "kernels_ms": kern,
                           "lengths_over_tract_counts_nocov": med["tract_lengths_device"] / med["tract_counts_device_nocov"],
                           "host_entry_e2e_ms": stats(ts),
                           "host_equals_device": bool(np.array_equal(h_spec, spec)),
                           "finite": bool(np.isfinite(spec).all())}
                    if xs[0] == 1:  # X = 1 bin against E[T_s] of the tract-count call
                        tr = d_tr.cpu().numpy()
                        run["x1_vs_tract_counts_max_rel"] = float(np.max(np.abs(spec[:, 0] - tr) / np.maximum(1.0, np.abs(tr))))
                    for x, want in zip((50, 100), planted):
                        if x in xs:
                            run[f"mean_runs_at_least_{x}_bins"] = [float(v) for v in spec[:, xs.index(x)].mean(axis=0)]
                            run[f"mean_planted_runs_at_least_{x}_bins"] = want
                    out["runs"].append(run)
    out["buffers"] = "device-resident calls on torch allocations; host entry from page-locked buffers"
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
