"""hiddengem posterior at C4 size (10,000 tables x 10,000 bins, the tables of tools/bench_aux.py leg_c4: same generator
and seed), beside the Viterbi pass on the same tables.  Prints one JSON line (and writes it to --out when given):

  - device-resident time of hiddengem_posterior_batch_device and of hiddengem_viterbi_batch_device: host clock around
    a synchronised call, warmed up, the two alternating over --reps repetitions (median and spread), then the engine's
    per-kernel times (CUDA events) in a separate set of repetitions;
  - bytes moved and the HBM roofline fraction on the compulsory traffic (48 B per bin: 24 in, 24 out) and on the traffic
    of the kernels as built (per bin: 24 read by each of the two passes, 24 written, 3 of alpha checkpoints);
  - host-entry end-to-end time (page-locked host buffers through hiddengem_posterior_batch);
  - the card's name and power limit, read in the same run.

`python tools/bench_posterior.py [--p01 P --p02 P --p12 P] --out FILE` on a GPU box.  Penalties with a zero (for
example --p02 0) or spread wider than 2^400 run the kernels in natural-log arithmetic (kernel_stats counts those launches
again as posterior_fwd_log / posterior_bwd_log)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", type=int, default=10_000)
    ap.add_argument("--bins", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--p01", type=float, default=1e-3)
    ap.add_argument("--p02", type=float, default=1e-6)
    ap.add_argument("--p12", type=float, default=1e-3)
    a = ap.parse_args()
    import torch
    import ibdgem_b200 as ib
    from bench_aux import hbm_peak
    if not torch.cuda.is_available():
        raise SystemExit("bench_posterior.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n_tables, n_bins = a.tables, a.bins
    nb = n_tables * n_bins
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    seg = torch.randint(0, 3, (nb // 200 + 1,), generator=g, device=dev).repeat_interleave(200)[:nb]
    d_ll = torch.randn((nb, 3), generator=g, device=dev, dtype=torch.float64) * 10.0 - 150.0
    d_ll[torch.arange(nb, device=dev), seg] += 8.0  # planted IBD0/1/2 segments
    seg = seg.to(torch.uint8)
    off = np.arange(n_tables + 1, dtype=np.int64) * n_bins
    d_post = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_exp = torch.empty((n_tables, 3), dtype=torch.float64, device=dev)
    d_state = torch.empty((nb,), dtype=torch.uint8, device=dev)
    d_score = torch.empty((nb, 3), dtype=torch.float64, device=dev)
    d_counts = torch.empty((n_tables, 3), dtype=torch.int64, device=dev)
    out = {"workload": "hiddengem posterior, C4: %d tables x %d bins of natural-log window scores (tools/bench_aux.py leg_c4 "
                       "tables), device-resident" % (n_tables, n_bins), "card": card(), "torch_device": torch.cuda.get_device_name(dev),
           "penalties": {"p01": a.p01, "p02": a.p02, "p12": a.p12}}
    pen = dict(p01=a.p01, p02=a.p02, p12=a.p12)
    with ib.Engine(ib.Params(device=0)) as e:
        def post():
            e.posterior_batch_device(d_ll.data_ptr(), off, True, d_post.data_ptr(), d_exp.data_ptr(), **pen)

        def vit():
            e.viterbi_batch_device(d_ll.data_ptr(), off, True, d_state.data_ptr(), d_score.data_ptr(), d_counts.data_ptr(), **pen)

        post()
        vit()
        tp, tv = [], []
        for _ in range(a.reps):  # alternating, host clock around synchronised calls (both entries synchronise)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            post()
            tp.append((time.perf_counter() - t0) * 1e3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            vit()
            tv.append((time.perf_counter() - t0) * 1e3)
        e.enable_timing(True)
        e.reset_stats()
        for _ in range(a.reps):
            post()
        kp = {k: v[0] / a.reps for k, v in e.kernel_stats().items() if v[1]}
        e.reset_stats()
        for _ in range(a.reps):
            vit()
        kv = {k: v[0] / a.reps for k, v in e.kernel_stats().items() if v[1]}
        e.enable_timing(False)
        rec_post = float((d_post.argmax(dim=1).to(torch.uint8) == seg).float().mean())
        rec_vit = float((d_state == seg).float().mean())
        row_err = float((d_post.sum(dim=1) - 1.0).abs().max())
        # host entry end to end: page-locked buffers
        h_ll = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
        h_ll.copy_(d_ll)
        h_post = torch.empty((nb, 3), dtype=torch.float64, pin_memory=True)
        h_exp = np.zeros((n_tables, 3))
        lib = e._lib

        def host():
            e._check(lib.hiddengem_posterior_batch(e._h, C.c_int32(n_tables), off.ctypes.data_as(C.c_void_p), C.c_void_p(h_ll.data_ptr()),
                                                   C.c_int32(1), C.c_double(a.p01), C.c_double(a.p02), C.c_double(a.p12),
                                                   C.c_void_p(h_post.data_ptr()), h_exp.ctypes.data_as(C.c_void_p)))

        host()
        th = []
        for _ in range(max(3, a.reps // 3)):
            t0 = time.perf_counter()
            host()
            th.append((time.perf_counter() - t0) * 1e3)
        assert torch.equal(h_post, d_post.cpu())
    hbm, src = hbm_peak()
    mp, mv = float(np.median(tp)), float(np.median(tv))
    ms_k = sum(kp.values())
    built = 24 * 2 + 24 + 2 * 24 / 16  # per bin: lik read by both passes, posterior written, checkpoints written and read

    def roof(bpb, ms):
        gbs = nb * bpb / 1e9 / (ms * 1e-3)
        return {"bytes_per_bin": bpb, "achieved_GBs": gbs, "frac": gbs / hbm}

    out.update({
        "posterior_ms": {"median": mp, "min": min(tp), "max": max(tp), "reps": a.reps, "clock": "host, around synchronised calls"},
        "viterbi_ms": {"median": mv, "min": min(tv), "max": max(tv), "reps": a.reps, "clock": "host, around synchronised calls"},
        "posterior_over_viterbi": mp / mv,
        "posterior_kernels_ms": kp, "viterbi_kernels_ms": kv,
        "hbm_peak_GBs": hbm, "hbm_peak_source": src,
        "roofline_compulsory": roof(48.0, ms_k), "roofline_as_built": roof(built, ms_k),
        "roofline_alpha_stored_design_bytes_per_bin": 120.0,
        "host_entry_e2e_ms": {"median": float(np.median(th)), "min": min(th), "max": max(th), "buffers": "page-locked"},
        "planted_state_recovery": {"posterior_argmax": rec_post, "viterbi": rec_vit},
        "max_row_sum_error": row_err,
        "working_set_note": "inputs and outputs are 2.4 GB each, far beyond the 126 MB L2",
    })
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
