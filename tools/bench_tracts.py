"""hiddengem IBD tracts at C4 size (10,000 tables x 10,000 bins, the tables of tools/bench_posterior.py: same generator
and seed), default penalties.  Prints one JSON line (and writes it to --out when given):

  - device-resident: the tract kernels' times (kernel_stats, CUDA events) and hiddengem_tracts_device as a synchronised
    call (host clock), on the device Viterbi states and posteriors; bytes per bin and the HBM fraction on the compulsory
    bytes (1 state byte + 24 B of likelihoods + 24 B of posteriors per bin; the records are a few MB);
  - host entry end to end from page-locked buffers: hiddengem_tracts_batch with and without posteriors, against what a
    caller does today, hiddengem_viterbi_batch + hiddengem_posterior_batch on the same buffers (per-bin arrays down);
  - the number of tracts, and the card's name and power limit, read in the same run.

`python tools/bench_tracts.py --out FILE` on a GPU box."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _stats(ts):
    return {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts)), "reps": len(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", type=int, default=10_000)
    ap.add_argument("--bins", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import ibdgem_b200 as ib
    from bench_aux import hbm_peak
    from bench_posterior import card
    if not torch.cuda.is_available():
        raise SystemExit("bench_tracts.py needs a CUDA device")
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
    p01, p02, p12 = 1e-3, 1e-6, 1e-3
    out = {"workload": "hiddengem tracts, C4: %d tables x %d bins of natural-log window scores (tools/bench_posterior.py tables), "
                       "default penalties" % (n_tables, n_bins), "card": card(), "torch_device": torch.cuda.get_device_name(dev)}
    with ib.Engine(ib.Params(device=0)) as e:
        d_state = torch.empty((nb,), dtype=torch.uint8, device=dev)
        d_counts = torch.empty((n_tables, 3), dtype=torch.int64, device=dev)
        d_score = torch.empty((nb, 3), dtype=torch.float64, device=dev)
        e.viterbi_batch_device(d_ll.data_ptr(), off, True, d_state.data_ptr(), d_score.data_ptr(), d_counts.data_ptr())
        del d_score
        d_post = torch.empty((nb, 3), dtype=torch.float64, device=dev)
        d_exp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
        e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr())
        del d_exp
        lib = e._lib
        toff = np.zeros(n_tables + 1, np.int64)

        def dev_call(post=True):
            e._check(lib.hiddengem_tracts_device(e._h, C.c_int32(n_tables), off.ctypes.data_as(C.c_void_p), C.c_int64(0),
                                                 C.c_void_p(d_ll.data_ptr()), C.c_int32(1), C.c_void_p(d_state.data_ptr()),
                                                 C.c_void_p(d_post.data_ptr() if post else None), toff.ctypes.data_as(C.c_void_p)))

        dev_call()
        n_tracts = int(toff[-1])
        td = []
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev_call()
            td.append((time.perf_counter() - t0) * 1e3)
        e.enable_timing(True)
        e.reset_stats()
        for _ in range(a.reps):
            dev_call()
        kt = {k: v[0] / a.reps for k, v in e.kernel_stats().items() if v[1]}
        e.reset_stats()
        for _ in range(a.reps):
            dev_call(False)
        kt_nopost = {k: v[0] / a.reps for k, v in e.kernel_stats().items() if v[1]}
        e.enable_timing(False)
        counts = d_counts.cpu().numpy()
        st = d_state.view(n_tables, n_bins)
        assert n_tracts == int((st[:, 1:] != st[:, :-1]).sum()) + n_tables
        del d_post
        # host entries end to end, page-locked buffers
        h_ll = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
        h_ll.copy_(d_ll)
        del d_ll
        torch.cuda.empty_cache()
        h_state = torch.empty((nb,), dtype=torch.uint8, pin_memory=True)
        h_score = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
        h_post = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
        h_counts = np.zeros((n_tables, 3), np.int64)
        h_exp = np.zeros((n_tables, 3))
        poff = off.ctypes.data_as(C.c_void_p)

        def tracts_host(post):
            e._check(lib.hiddengem_tracts_batch(e._h, C.c_int32(n_tables), poff, C.c_void_p(h_ll.data_ptr()), C.c_int32(1), C.c_double(p01),
                                                C.c_double(p02), C.c_double(p12), C.c_int32(1 if post else 0), toff.ctypes.data_as(C.c_void_p)))

        def today():
            e._check(lib.hiddengem_viterbi_batch(e._h, C.c_int32(n_tables), poff, C.c_void_p(h_ll.data_ptr()), C.c_int32(1), C.c_double(p01),
                                                 C.c_double(p02), C.c_double(p12), C.c_void_p(h_state.data_ptr()),
                                                 C.c_void_p(h_score.data_ptr()), h_counts.ctypes.data_as(C.c_void_p)))
            e._check(lib.hiddengem_posterior_batch(e._h, C.c_int32(n_tables), poff, C.c_void_p(h_ll.data_ptr()), C.c_int32(1), C.c_double(p01),
                                                   C.c_double(p02), C.c_double(p12), C.c_void_p(h_post.data_ptr()),
                                                   h_exp.ctypes.data_as(C.c_void_p)))

        tracts_host(True)
        tracts_host(False)
        today()
        th_post, th_nopost, t_today = [], [], []
        for _ in range(max(3, a.reps // 2)):  # alternating, host clock (every entry synchronises)
            for fn, acc in ((lambda: tracts_host(True), th_post), (lambda: tracts_host(False), th_nopost), (today, t_today)):
                t0 = time.perf_counter()
                fn()
                acc.append((time.perf_counter() - t0) * 1e3)
        tracts_host(True)
        assert int(toff[-1]) == n_tracts
        recs = e.last_tracts(n_tracts)
        table = np.repeat(np.arange(n_tables), np.diff(toff))
        per_state = np.zeros((n_tables, 3), np.int64)
        np.add.at(per_state, (table, recs["state"]), recs["n_bins"])
        assert (per_state == counts).all() and (h_counts == counts).all()
    hbm, src = hbm_peak()
    ms_k = kt.get("tract_count", 0.0) + kt.get("tract_emit", 0.0)
    bpb = 1 + 24 + 24
    gbs = nb * bpb / 1e9 / (ms_k * 1e-3)
    up_gb = nb * 24 / 1e9
    out.update({
        "n_tracts": n_tracts, "mean_tract_bins": nb / n_tracts,
        "tract_kernels_ms": kt, "tract_kernels_no_posterior_ms": kt_nopost,
        "device_call_ms": dict(_stats(td), clock="host, around synchronised hiddengem_tracts_device calls"),
        "compulsory_bytes_per_bin": bpb, "records_MB": n_tracts * 64 / 1e6,
        "hbm_peak_GBs": hbm, "hbm_peak_source": src,
        "roofline_compulsory": {"achieved_GBs": gbs, "frac": gbs / hbm, "floor_ms": nb * bpb / (hbm * 1e9) * 1e3},
        "host_tracts_batch_ms": dict(_stats(th_post), buffers="page-locked", posterior=True),
        "host_tracts_batch_no_posterior_ms": dict(_stats(th_nopost), buffers="page-locked", posterior=False),
        "host_viterbi_plus_posterior_ms": dict(_stats(t_today), buffers="page-locked",
                                               note="hiddengem_viterbi_batch + hiddengem_posterior_batch: states, scores and posteriors come down"),
        "upload_GB": up_gb,
        "working_set_note": "likelihoods and posteriors are 2.4 GB each, far beyond the 126 MB L2",
    })
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
