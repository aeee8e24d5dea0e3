#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native IBDGem engine.

Metric (BASELINE.json): LD genotype-comparisons/s, one comparison = one
site x target x background-individual x 1-of-4 haplotype pairing (the multiply at
src/ibdgem.c:716-719 of the reference).  Workload at N=1: BASELINE.json configs[2] — `--LD`
scoring of a synthetic chr20-scale panel, 1,000,000 sites x 2,504 phased samples, 1,000 targets,
window 1,000 sites (SURVEY.md §8d "C3", depth >= 1 variant).  At N>1 every rank scores its own
1,000 targets against the replicated panel (weak scaling) and stores its window scores into the
gathered table in rank 0's HBM over NVLink (CUDA IPC peer stores; fallback: one NCCL all_gather).

The other configurations of BASELINE.json ride on the same JSON line under "aux" (tools/bench_aux.py):
c2 (non-LD), c4 (hiddengem), c5 (10k targets x 5k background; windows partitioned across the ranks at every N),
strong_c3 (N>1: C3 in full, windows partitioned), ld_v (C3 with -v), flat_rows, cli_e2e, int8_peak.

    python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
    python bench.py --impl reference ...                     (the reference's CPU binary)

Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "LD genotype-comparisons/s (site x target x bg x 4)"
UNIT = "comparisons/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--targets", type=int, default=1000)
    ap.add_argument("--window", type=int, default=1000)
    ap.add_argument("--cpu-sites", type=int, default=10_000, help="site sample for the CPU baseline")
    ap.add_argument("--cpu-targets", type=int, default=16, help="targets of the single-core CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the secondary legs (C2, C4, -v, flat rows, CLI, int8 peak)")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 leg (10k targets x 5k background, 15k-individual panel)")
    ap.add_argument("--force-general", action="store_true", help="A/B: CUDA-core --LD path")
    ap.add_argument("--panel-pieces", type=int, default=int(os.environ.get("IBDGEM_BENCH_PANEL_PIECES", "-1")),
                    help="N>1: the panel is replicated over NVLink in this many pieces (0 = every rank uploads all "
                         "of it; default max(2, 16 // N): ~40 MB per rank and piece at C3; measured at N=2: "
                         "0 -> 12.8 ms, 1 -> 15.6, 4 -> 11.6, 8 -> 10.7, 16 -> 12.1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's results of the last timed step as DIR/<name>.npy "
                         "(targets, n_windows, and w_start, w_end, w_nsites, w_loglik of every window, target after "
                         "target); under 64 MB in all, larger results keep a fixed seeded sample of the targets")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 60_000_000  # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(path, targets, n_windows, w_start, w_end, w_nsites, w_loglik):
    """Writes the window scores a caller of the --LD scoring path receives, one float64 .npy file per
    array.  Only a target's first n_windows slots hold results, so the per-window arrays keep just those,
    target after target ([sum of n_windows] and [sum of n_windows, 3]); n_windows splits them again.
    When all of it could exceed DUMP_LIMIT_BYTES, a fixed seeded sample of the targets is kept, in target order."""
    T, maxW = w_loglik.shape[:2]
    per_target = 8 * (1 + 1 + maxW * (3 + 3))  # targets, n_windows, w_start/w_end/w_nsites, w_loglik
    rows = np.arange(T)
    if T * per_target > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(T, DUMP_LIMIT_BYTES // per_target, replace=False))
    nw = n_windows[rows].astype(np.int64)
    valid = np.arange(maxW)[None, :] < nw[:, None]

    def windows(a):
        return a[rows][valid].astype(np.float64)

    os.makedirs(path, exist_ok=True)
    for name, a in (("targets", targets[rows].astype(np.float64)), ("n_windows", nw.astype(np.float64)),
                    ("w_start", windows(w_start)), ("w_end", windows(w_end)), ("w_nsites", windows(w_nsites)),
                    ("w_loglik", windows(w_loglik))):
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# reference CPU arm helpers
def write_reference_sample(dirpath, bits_np, H, n_ref, n_alt, pos, n_sites):
    """IMPUTE triple + pileup for the first n_sites of the workload (same seeded data)."""
    from ibdgem_b200.synth import unpack_rows
    os.makedirs(dirpath, exist_ok=True)
    hap = unpack_rows(bits_np, H, np.arange(n_sites))
    txt = np.full((n_sites, 2 * H), ord(" "), np.uint8)
    txt[:, 0::2] = hap + ord("0")
    txt[:, -1] = ord("\n")
    txt.tofile(os.path.join(dirpath, "p.hap"))
    with open(os.path.join(dirpath, "p.legend"), "w") as fh:
        fh.write("ID pos allele0 allele1\n")
        fh.write("".join("s%d %d A G\n" % (i, int(pos[i])) for i in range(n_sites)))
    with open(os.path.join(dirpath, "p.indv"), "w") as fh:
        fh.write("".join("i%d\n" % i for i in range(H // 2)))
    with open(os.path.join(dirpath, "u.pileup"), "w") as fh:
        for i in range(n_sites):
            b = "A" * int(n_ref[i]) + "G" * int(n_alt[i])
            c = len(b)
            fh.write("20\t%d\tN\t%d\t%s\t%s\t%s\n" % (int(pos[i]), c, b or "*", "I" * c or "*", "]" * c or "*"))


def run_reference_procs(binary, dirpath, target_lists, window, ld=True, tag="out"):
    """One process per target list (the reference is single-threaded; independent processes
    sharded with -S are how it uses more than one core).  Returns wall seconds."""
    procs = []
    for k, tl in enumerate(target_lists):
        with open(os.path.join(dirpath, "targets_%d.txt" % k), "w") as fh:
            fh.write("".join("i%d\n" % t for t in tl))
        os.makedirs(os.path.join(dirpath, "%s_%d" % (tag, k)), exist_ok=True)
    t0 = time.perf_counter()
    for k, tl in enumerate(target_lists):
        procs.append(subprocess.Popen([binary, "-H", "p.hap", "-L", "p.legend", "-I", "p.indv", "-P", "u.pileup"] +
                                      (["--LD"] if ld else []) + ["-w", str(window), "-S", "targets_%d.txt" % k,
                                                                  "-O", "%s_%d" % (tag, k)],
                                      cwd=dirpath, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("reference binary failed")
    return time.perf_counter() - t0


def host_sample(args, seed=1):
    """The first cpu_sites sites of the synthetic workload, generated on the host with numpy."""
    from ibdgem_b200.synth import synth_panel_numpy
    return synth_panel_numpy(args.cpu_sites, args.samples, seed=seed)


def cpu_baseline(args, sample=None, n_procs=1, targets_per_proc=None, tmp=None, with_o2=False):
    """Times the reference's own CPU implementation of the path on a bounded sample: the first
    cpu_sites sites of the workload, targets_per_proc targets per process, full background."""
    d = sample if sample is not None else host_sample(args)
    S1 = args.cpu_sites
    H = 2 * args.samples
    tpp = targets_per_proc or args.cpu_targets
    inf = int(((d["n_ref"][:S1].astype(int) + d["n_alt"][:S1]) >= 1).sum())
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "ibdgem")
    own_tmp = tmp is None
    if own_tmp:
        tmp = tempfile.mkdtemp(prefix="ibdgem_cpu_")
    extra = {}
    try:
        if os.path.exists(ref_bin):
            if not os.path.exists(os.path.join(tmp, "p.hap")):
                write_reference_sample(tmp, d["bits"], H, d["n_ref"], d["n_alt"], d["pos"], S1)
            lists = [[(k * tpp + j) % args.samples for j in range(tpp)] for k in range(n_procs)]
            wall = run_reference_procs(ref_bin, tmp, lists, args.window)
            comps = n_procs * tpp * inf * (args.samples - 1) * 4
            kind = "reference"
            note = "oracle/_ref/ibdgem (unmodified reference, as-shipped flags -ggdb3 = -O0)"
            if with_o2 and os.path.exists(ref_bin + ".O2"):  # SURVEY.md 8(d): state both builds
                wall2 = run_reference_procs(ref_bin + ".O2", tmp, lists, args.window, tag="out_o2")
                extra = {"value_O2": comps / wall2, "O2_note": "same sample, reference sources built with -O2: %.2f s wall" % wall2}
        else:
            import oracle
            from ibdgem_b200.synth import unpack_rows
            hap = unpack_rows(d["bits"], H, np.arange(S1))
            prm = oracle.Params(window=args.window, ld_mode=1)
            t0 = time.perf_counter()
            comps = oracle.ld_loop_bench(prm, d["n_ref"][:S1], d["n_alt"][:S1], hap, np.arange(tpp, dtype=np.int32),
                                         np.arange(args.samples, dtype=np.int32))
            wall = time.perf_counter() - t0
            kind = "port"
            note = "oracle/liboracle.so orc_ld_loop_bench (C restatement of src/ibdgem.c:673-721, -O2)"
            n_procs = 1
    finally:
        if own_tmp:
            shutil.rmtree(tmp, ignore_errors=True)
    out = dict(value=comps / wall, unit=UNIT, cores=n_procs, kind=kind,
               sample="%s; first %d sites x %d target(s) per process x %d process(es) x %d background, --LD -w %d, "
                      "%.2f s wall" % (note, S1, tpp, n_procs, args.samples - 1, args.window, wall))
    out.update(extra)
    return out, comps, wall


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_procs = max(1, min(os.cpu_count() or 1, 64))
    sample = host_sample(args)
    tpp = max(1, args.cpu_targets // 4)
    vals = []
    last = None
    tmp = tempfile.mkdtemp(prefix="ibdgem_ref_")
    try:
        for i in range(args.warmup + args.steps):
            cb, comps, wall = cpu_baseline(args, sample, n_procs, tpp, tmp)
            if i >= args.warmup:
                vals.append((comps, wall))
            last = cb
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    comps = sum(c for c, _ in vals)
    wall = sum(w for _, w in vals)
    v = comps / wall
    last["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall / max(len(vals), 1) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "--LD scoring, bounded CPU sample of C3 per step: first %d sites x %d targets (%d per "
                               "process, one process per host core, %d cores) x %d background, window %d" % (
                                   args.cpu_sites, n_procs * tpp, tpp, n_procs, args.samples - 1, args.window)},
        "cpu_baseline": last,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML from a thread, every
    few ms; nvidia-smi would manage one sample per step)."""

    def __init__(self, index, period_s=0.004):
        import threading
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}

            def run():
                while not self._stop.is_set():
                    try:
                        self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for n, bit in names.items():
                            if r & bit:
                                self.reasons.add(n)
                        self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    except Exception:
                        pass
                    time.sleep(period_s)

            self._thread = threading.Thread(target=run, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        if self._thread is None:
            return out
        self._stop.set()
        self._thread.join(timeout=2)
        if self.samples:
            out = {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                   "reasons": sorted(self.reasons), "samples": len(self.samples),
                   "power_w_max": max(self.power) if self.power else None}
        return out


def aux_legs(args, torch, ib, eng, bits, pos, n_ref, n_alt, ref_tmp, ref_wall, peaks, achieved_tops):
    """Secondary legs on one GPU (tools/bench_aux.py); a leg that fails is reported, not fatal."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_aux as ba
    eng.close()  # the headline engine's operands (~8.5 GB) are not needed any more
    torch.cuda.empty_cache()
    S, N, T, W = args.sites, args.samples, args.targets, args.window
    full = (S, N, T, W) == (1_000_000, 2504, 1000, 1000)
    aux = {}

    def leg(name, fn):
        t0 = time.perf_counter()
        try:
            aux[name] = fn()
        except Exception as ex:  # noqa: BLE001
            aux[name] = {"failed": repr(ex)[:300]}
        aux[name]["leg_wall_s"] = round(time.perf_counter() - t0, 2)

    leg("int8_peak", lambda: ba.leg_int8_peak(torch))
    if "burst_tops" in aux["int8_peak"]:
        aux["int8_peak"]["ld_mma_frac_of_burst"] = achieved_tops / aux["int8_peak"]["burst_tops"]
        aux["int8_peak"]["ld_mma_frac_of_sustained"] = achieved_tops / aux["int8_peak"]["sustained_tops"]
    # C3 with the pileup's source outside the background: no row has a dominant column, ~6 % of the
    # accumulator elements pass the screen (DESIGN.md 4.1) — the forensic common case
    def flat():
        r2, a2 = ba.make_counts(bits, N - 1, 3, 1)
        return ba.leg_ld(torch, ib, bits, pos, r2, a2, N, T, W, args.steps, 0, np.arange(N - 1, dtype=np.int32),
                         "C3 shape, reads drawn from individual %d, background = individuals 0..%d (source not in it)" % (N - 1, N - 2))
    leg("flat_rows", flat)
    # C3 with -v, the flag the reference recommends (README.md:180; src/ibdgem.c:584-587): per-target windows
    leg("ld_v", lambda: ba.leg_ld(torch, ib, bits, pos, n_ref, n_alt, N, T, W, args.steps, 1, None,
                                  "C3 shape with -v (variable sites only): per-target window maps"))
    leg("c2", lambda: ba.leg_c2(torch, ib, bits, pos, N, args.steps, ref_tmp, args.cpu_sites))
    if full:
        leg("c4", lambda: ba.leg_c4(torch, ib, 3, 10_000, 10_000, ref_tmp))
    else:
        leg("c4", lambda: ba.leg_c4(torch, ib, 3, 500, 2_000, ref_tmp))
    if ref_wall is not None:
        leg("cli_e2e", lambda: ba.leg_cli(ref_tmp, W, ref_wall, args.cpu_targets))
    return aux


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import ibdgem_b200 as ib
    from ibdgem_b200.engine import _CScores
    from ibdgem_b200.shard import gather_window_scores
    from ibdgem_b200.synth import synth_panel_torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    # stdout carries exactly one JSON line: whatever libraries print on fd 1 meanwhile (NCCL's version
    # banner, for one) goes to stderr
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # (NCCL_DEBUG is left to the caller: fd 1 already points at stderr, so INFO lines cannot reach the JSON line)
        dist.init_process_group("nccl", device_id=dev)

    S, N, T, W = args.sites, args.samples, args.targets, args.window
    d = synth_panel_torch(S, N, seed=1, device=dev)  # pinned host tensors, identical on every rank
    bits = d["bits"].numpy().view(np.uint32)
    pos = d["pos"].numpy().view(np.uint64)
    n_ref, n_alt, keep = d["n_ref"].numpy(), d["n_alt"].numpy(), d["keep"].numpy()
    # weak scaling: every rank scores its own T targets
    targets = ((rank * T + np.arange(T)) % N).astype(np.int32)
    bg = np.arange(N, dtype=np.int32)
    inf_sites = int(((n_ref.astype(np.int64) + n_alt) >= 1).sum())
    comps_rank = inf_sites * int(T) * (N - 1) * 4
    maxW = S // W + 2

    eng = ib.Engine(ib.Params(window_size=W, device=local_rank))
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.enable_timing(True)
    if args.force_general:
        eng.force_general_ld(True)

    # pinned result buffers + a device tensor for the gather
    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    o_nw = pinned((T,), torch.int32)
    o_ws, o_we = pinned((T, maxW), torch.int64), pinned((T, maxW), torch.int64)
    o_wn = pinned((T, maxW), torch.int32)
    o_ll = pinned((T, maxW, 3), torch.float64)
    # The gathered score table [world * T][maxW][3] lives in rank 0's HBM and is mapped into every rank (CUDA
    # IPC): each rank's engine stores its own block there, window range by window range, over NVLink — the
    # gather needs no collective call and no rendezvous inside the step.  Fallback (IPC unavailable): one
    # NCCL all_gather per step, as in round 1.
    from ibdgem_b200.shard import PeerTable
    table = PeerTable(world * T, maxW, local_rank)
    d_ll = None
    if table.ok:
        if table.is_root:
            table.tensor().fill_(float("nan"))
        dst = table.block_ptr(rank * T)
    else:
        d_ll = torch.empty((T, maxW, 3), dtype=torch.float64, device=dev)
        dst = d_ll.data_ptr()
    cs = _CScores(maxW, o_nw.data_ptr(), o_ws.data_ptr(), o_we.data_ptr(), o_wn.data_ptr(), o_ll.data_ptr(),
                  None, None, None, None, None, None, None, dst)

    # N > 1: the packed panel is the same on every rank, so each rank copies 1/N of it over PCIe and the
    # ranks all_gather the pieces over NVLink (shard.replicate_panel) instead of N full uploads
    if args.panel_pieces < 0:
        args.panel_pieces = max(2, 16 // world)
    replicate = world > 1 and args.panel_pieces > 0
    if replicate:
        from ibdgem_b200.shard import panel_pieces, replicate_panel
        _, padded_rows = panel_pieces(S, world, args.panel_pieces)
        d_panel = torch.empty((padded_rows, bits.shape[1]), dtype=torch.int32, device=dev)
        up_stream = torch.cuda.Stream(device=dev)

    def upload():
        eng.upload_sites(pos, n_ref, n_alt, keep)
        if replicate:
            up_stream.wait_stream(stream)
            replicate_panel(eng, d["bits"], d_panel, N, pieces=args.panel_pieces, stream=up_stream)
        else:
            eng.upload_panel(bits, N)

    def score():
        # one step = the whole path from the packed inputs resident in HBM: allele-frequency popcount
        # + per-site table + window map (prepare), the cached window operands, then --LD scoring.
        # invalidate() discards every derived device array of the previous step (nothing is cached
        # across steps except the allocations).
        eng.invalidate()
        eng.score_ld_raw(targets, bg, -1, cs)  # includes the store of this rank's block into the root's table
        if world > 1 and d_ll is not None:
            gather_window_scores(d_ll, world * T)  # fallback: one NCCL all_gather of [T][maxW][3] fp64 per rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            every = torch.zeros(world, device=dev, dtype=torch.float64)
            dist.all_gather_into_tensor(every, ms)
            timed.per_rank = [float(x) / steps for x in every.tolist()]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- value: inputs resident in HBM ---------------------------------------------------------
    upload()
    eng.sync_uploads()  # the panel is resident before the first step, not still arriving in chunks
    torch.cuda.synchronize()
    eng.prepare()
    for _ in range(max(args.warmup, 3)):
        score()
    gather_check = None
    if world > 1 and table.ok:
        # outside the timed region: the root's table must equal an NCCL all_gather of every rank's host results
        barrier()
        every = gather_window_scores(o_ll.to(dev), world * T)
        if rank == 0:
            gather_check = bool(torch.equal(torch.nan_to_num(every, nan=-1.0), torch.nan_to_num(table.tensor(), nan=-1.0)))
        del every
        barrier()
    eng.reset_stats()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total = timed(score, args.steps)
    rank_ms = getattr(timed, "per_rank", None)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # the e2e steps below overwrite the same host buffers, so the last timed step's results are saved now
        dump_outputs(args.dump_outputs, targets, o_nw.numpy(), o_ws.numpy(), o_we.numpy(), o_wn.numpy(), o_ll.numpy())
    stats = eng.kernel_stats()
    ld_path = eng.last_ld_path()
    ms_step = ms_total / args.steps
    value = comps_rank * world / (ms_step * 1e-3)

    # ---- e2e: host buffers in, host results out, every step -------------------------------------
    def e2e_step():
        upload()
        score()

    # the per-launch event pairs are only needed for the roofline of the device-resident loop above
    eng.enable_timing(bool(os.environ.get("IBDGEM_TIMELINE")))
    for _ in range(2):
        e2e_step()
    e2e_steps = max(2, min(args.steps, 3))
    ms_e2e = timed(e2e_step, e2e_steps) / e2e_steps
    h2d = (bits.nbytes // world if replicate else bits.nbytes) + pos.nbytes + n_ref.nbytes + n_alt.nbytes + keep.nbytes + targets.nbytes + bg.nbytes
    d2h = o_nw.numel() * 4 + o_ws.numel() * 8 * 2 + o_wn.numel() * 4 + o_ll.numel() * 8
    e2e_value = comps_rank * world / (ms_e2e * 1e-3)

    # ---- partition by windows: strong scaling of C3, and C5 (all ranks take part) -----------------
    multi = {}
    dev_bytes = eng.device_bytes()
    if not args.no_aux:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_aux as ba
        eng.close()
        table.close()
        torch.cuda.empty_cache()

        def mleg(name, fn):
            t0 = time.perf_counter()
            try:
                r = fn()
            except Exception as ex:  # noqa: BLE001
                r = {"failed": repr(ex)[:300]}
            if rank == 0 and r is not None:
                r["leg_wall_s"] = round(time.perf_counter() - t0, 2)
                multi[name] = r

        if world > 1:
            mleg("strong_c3", lambda: ba.leg_window_sharded(
                torch, ib, world, rank, d["bits"], pos, n_ref, n_alt, N, np.arange(T, dtype=np.int32), bg, W, args.steps,
                "C3 in full on %d GPU(s): %d sites x %d-sample panel, %d targets in total, window %d" % (world, S, N, T, W)))
        if (S, N, W) == (1_000_000, 2504, 1000) and not args.no_c5:
            def c5():
                d5 = ba.c5_inputs(torch, S, 15_000)
                return ba.leg_window_sharded(
                    torch, ib, world, rank, d5["bits"], d5["pos"].numpy().view(np.uint64), d5["n_ref"].numpy(), d5["n_alt"].numpy(),
                    15_000, np.arange(10_000, dtype=np.int32), np.arange(10_000, 15_000, dtype=np.int32), W, max(2, min(args.steps, 3)),
                    "C5 (BASELINE.json configs[4]): %d sites x 15,000-individual panel, 10,000 targets x 5,000 disjoint "
                    "background individuals, window %d, reads drawn from background individual 10,000" % (S, W))
            mleg("c5", c5)

    if rank == 0:
        launches = int(sum(n for _, n in stats.values()))
        dom = "ld_mma" if ld_path == 1 else "ld_general"
        dom_ms, dom_n = stats[dom]
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except OSError:
            pass
        # Algorithmic work of the dominant kernel (DESIGN.md "Roofline"): one multiply-accumulate of the
        # weighted binary contraction sum_s n_s h_s k_s per comparison = 2 op / comparison.  The kernel
        # runs it as int8 on tcgen05 (kind::i8), whose rate is 2x the bf16 rate, so the denominator is
        # 2 x the measured dense bf16 figure of MEASURED_PEAKS.json (sustained: the kernel is timed
        # inside a long step).  That figure was taken at the power-capped clock of a bf16 GEMM
        # (~1.35 GHz); 0/1 x small-integer operands toggle few bits and this kernel holds the full
        # boost clock, so frac can exceed 1 — pipe_peak_at_clock is the hardware ceiling
        # (148 SMs x 8192 int8 MAC/clk x 2) at the SM clock sampled during the run.
        flop_per_launch = 2.0 * comps_rank * args.steps / max(dom_n, 1)
        avg_ms = dom_ms / max(dom_n, 1)
        achieved = flop_per_launch / (avg_ms * 1e-3) / 1e12 if avg_ms > 0 else 0.0
        bf16 = peaks.get("bf16_tflops_sustained") or 1400.0
        peak = 2.0 * bf16 if ld_path == 1 else bf16
        sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        pipe_peak = 148 * 8192 * 2 * sm_mhz * 1e6 / 1e12
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                traffic = json.load(fh).get(dom)
        except (OSError, ValueError):
            pass
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "kernel": dom, "avg_launch_ms": avg_ms,
                    "launches": dom_n,
                    "peak_source": ("2 x bf16_tflops_sustained of measured MEASURED_PEAKS.json (int8 tcgen05 rate "
                                    "= 2 x bf16)" if ld_path == 1 else "bf16_tflops_sustained of measured") if peaks
                    else "fallback 1.4 PFLOP/s sustained bf16",
                    "pipe_peak_at_clock": pipe_peak, "frac_of_pipe_peak": achieved / pipe_peak,
                    "note": "frac can exceed 1: the bf16 denominator was measured power-capped (~1.35 GHz, ~1 kW); this "
                            "int8 kernel on 0/1 operands holds the full SM clock (see clocks) at ~300 W. "
                            "frac_of_pipe_peak is against 148 SM x 8192 int8 MAC/clk x 2 at the sampled clock.",
                    "kernel_share_of_step": dom_ms / (ms_total) if ms_total > 0 else None,
                    "kernels_ms_per_step": {k: v[0] / args.steps for k, v in stats.items() if v[1]}}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C3 --LD scoring: %d sites x %d-sample phased panel, %d targets per GPU, "
                                   "window %d, depth Poisson(2)+1 (BASELINE.json configs[2]); the pileup's reads are drawn "
                                   "from individual 0, who IS in the background (SURVEY.md 8d) — the other case is "
                                   "aux.flat_rows" % (S, N, T, W),
                       "sites": S, "samples": N, "targets_per_gpu": T, "window": W,
                       "parallelism": "targets sharded across %d GPU(s), panel replicated%s, window scores gathered into "
                                      "rank 0's HBM by peer stores over NVLink" % (world, (" (e2e: each rank uploads 1/%d of it over PCIe, "
                                                                 "%d all_gather pieces over NVLink)" % (world, args.panel_pieces))
                                                         if replicate else ""),
                       "ld_path": "tensor (tcgen05 int8 window GEMM + fused LSE)" if ld_path == 1 else "general CUDA-core",
                       "l2": "inputs larger than L2 (packed panel %.0f MB, operands %.1f GB)" % (
                           bits.nbytes / 1e6, dev_bytes / 1e9)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "bytes_are": "per rank",
                    "ms_per_step": ms_e2e},
            "gpu_launches": launches,
            "roofline": roofline,
        }
        if rank_ms:
            out["ms_per_step_by_rank"] = rank_ms  # value uses the maximum
        if world > 1:
            out["gather"] = {"how": ("every rank stores its [T][maxW][3] fp64 block into rank 0's HBM over NVLink (CUDA IPC "
                                     "mapping, cudaMemcpy2DAsync per window range from inside the score call); no collective, "
                                     "no rendezvous inside the step") if table.ok or gather_check is not None else
                                    "fallback: one NCCL all_gather_into_tensor per step",
                             "bytes_per_rank": int(T * (S // W) * 24), "equals_nccl_all_gather": gather_check}
        if multi:
            out.setdefault("aux", {}).update(multi)
        ref_tmp = tempfile.mkdtemp(prefix="ibdgem_cpu_")
        try:
            ref_wall = None
            if world == 1 and not args.no_cpu_baseline:
                cb, _, ref_wall = cpu_baseline(args, tmp=ref_tmp, with_o2=True)
                out["cpu_baseline"] = cb
            if world == 1 and not args.no_aux:
                out.setdefault("aux", {}).update(
                    aux_legs(args, torch, ib, eng, bits, pos, n_ref, n_alt, ref_tmp, ref_wall, peaks, achieved))
                i8 = out["aux"].get("int8_peak", {})
                if "burst_tops" in i8:  # the int8 tensor peak measured on THIS box, next to the 2 x bf16 inference
                    roofline["int8_peak_measured_here"] = {"burst": i8["burst_tops"], "sustained": i8["sustained_tops"], "unit": "TOP/s"}
                    roofline["frac_of_int8_burst"] = achieved / i8["burst_tops"]
                    roofline["frac_of_int8_sustained"] = achieved / i8["sustained_tops"]
        finally:
            shutil.rmtree(ref_tmp, ignore_errors=True)
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    eng.close()
    table.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
