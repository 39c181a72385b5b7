#!/usr/bin/env python3
"""bench.py -- throughput of the ELECTOR POA hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          (N>1: launched by torchrun)
  python bench.py --impl reference --gpus N --steps K --warmup W

One step = one pass of the hot path (three-way POA of every window of every triplet, then
the per-read merge + tally + global counter sum) over the workload: BASELINE.json
configs[1], 10 000 triplets of 10 kb reads at 10 % / 1 % error, cut into ~1.95 M windows by
the unchanged reference splitter.  Per-GPU work is fixed (weak scaling): rank r owns read
ids [r*10000, (r+1)*10000).  The window arrays (~300 MB) exceed the 126 MB L2, so no
flush is needed between steps.

  value     triplets/s with the window arrays already resident in HBM (elector_poa_run_device +
            elector_merge_tally_device + elector_tally_sum_device)
  e2e       the same through the host-buffer C-ABI call (elector_pipeline_run2): pinned host arrays in (letters 2-bit
            packed once outside the call, 32-bit offsets), merged per-read MSA rows + per-read counters out, H2D/D2H
            inside the timed region; e2e.modes times the other wire formats of the call (bytes in / window rows out as
            in round 1, 4-bit merged rows, counters only)
  roofline  INT32 issue roofline of the DP kernel (15 integer ops per DP cell, SURVEY.md 8d)
            against the peak measured on this device by elector_int32_peak
  cpu_baseline  the reference poa binary (oracle/_ref/poa) or the oracle port, timed on
            this box's host cores on a bounded prefix of the same workload
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

INT_OPS_PER_CELL = 15  # SURVEY.md 8d convention


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks + throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def cpu_reference_throughput(wl, n_triplets, procs, kind):
    """Times the reference's CPU implementation on the first n_triplets triplets of wl.
    kind 'reference': oracle/_ref/poa, one single-threaded process per shard file, `procs`
    concurrently (how elector/alignment.py:117-119 runs it), shards balanced by windows.
    kind 'port': the oracle (oracle/poa_oracle.c) with `procs` OpenMP threads."""
    import workloads
    sub = workloads.slice_windows(wl, 0, n_triplets)
    n = len(sub["ref_off"]) - 1
    lr, lc, lu = np.diff(sub["ref_off"]), np.diff(sub["cor_off"]), np.diff(sub["unc_off"])
    if kind == "port":
        from oracle import oracle
        t0 = time.perf_counter()
        o = oracle.batch(sub["ref"], sub["ref_off"], sub["cor"], sub["cor_off"], sub["unc"], sub["unc_off"], nthreads=procs)
        dt = time.perf_counter() - t0
        cells = int(o["cells"].sum())
    else:
        work = tempfile.mkdtemp(prefix="elref_")
        try:
            bounds = [(n * i) // procs for i in range(procs + 1)]
            for i in range(procs):
                a, b = bounds[i], bounds[i + 1]
                for key, name in (("ref", "out1"), ("unc", "out2"), ("cor", "out3")):
                    off, seq = sub[key + "_off"], sub[key]
                    with open("%s/%s%d" % (work, name, i), "wb") as f:
                        for w in range(a, b):
                            f.write(b">w%d\n" % w)
                            f.write(seq[int(off[w]):int(off[w + 1])].tobytes())
                            f.write(b"\n")
            exe, mat = os.path.join(ROOT, "oracle", "_ref", "poa"), os.path.join(ROOT, "oracle", "_ref", "blosum80.mat")
            t0 = time.perf_counter()
            ps = [subprocess.Popen([exe, "-pir", "%s/smsa%d" % (work, i), "-preserve_seqorder", "-corrected_reads_fasta",
                                    "%s/out3%d" % (work, i), "-reference_reads_fasta", "%s/out1%d" % (work, i),
                                    "-uncorrected_reads_fasta", "%s/out2%d" % (work, i), "-preserve_seqorder", "-threads", "1",
                                    "-pathMatrix", mat], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                  for i in range(procs) if bounds[i + 1] > bounds[i]]
            for p in ps:
                p.wait()
            dt = time.perf_counter() - t0
            cells = int((lr * lc + np.maximum(lr, lc) * lu).sum())  # lower bound on the cells (len(P1) >= max(lr, lc))
        finally:
            shutil.rmtree(work, ignore_errors=True)
    return {"seconds": dt, "triplets_per_s": n_triplets / dt, "windows_per_s": n / dt, "gcups": cells / dt / 1e9,
            "windows": n, "triplets": n_triplets}


DUMP_WINDOWS = 1 << 16          # windows whose per-window results are written
DUMP_READS = 1 << 16            # reads whose per-read counters are written
DUMP_ROW_LETTERS = 4 << 20      # at most this many MSA row columns (3 per window column) are written


def dump_outputs(out_dir, wl, d_rows, d_rowoff, d_stride, d_nring, d_s1, d_s2, d_cells, d_cnt, d_sums):
    """What elector_poa_run_device + elector_merge_tally_device + elector_tally_sum_device left in their output buffers, as
    float64 .npy files of at most ~50 MB in all: the global counters, and for samples of reads and of windows drawn with a
    fixed seed from their counts alone (the same ones for the same arguments) the per-read counters, and per window the
    ring length, DP scores, cell count and the three MSA rows, concatenated in the order rows_window_index lists them.
    The rows stop at DUMP_ROW_LETTERS columns, counted from the input lengths, so that the cut does not depend on what
    was computed."""
    import torch
    n, n_trip = len(wl["ref_off"]) - 1, len(wl["read_first"]) - 1
    rng = np.random.default_rng(12345)
    win = np.sort(rng.choice(n, min(n, DUMP_WINDOWS), replace=False))
    reads = np.sort(rng.choice(n_trip, min(n_trip, DUMP_READS), replace=False))
    nring = d_nring.cpu().numpy()
    out = {"sums": d_sums.cpu().numpy(), "read_index": reads, "counters": d_cnt.cpu().numpy().reshape(n_trip, -1)[reads],
           "window_index": win, "nring": nring[win], "score1": d_s1.cpu().numpy()[win], "score2": d_s2.cpu().numpy()[win],
           "cells": d_cells.cpu().numpy()[win]}
    # nring <= ref + cor + unc letters of the window: the row budget is cut on that bound
    bound = sum(np.diff(wl[k])[win] for k in ("ref_off", "cor_off", "unc_off"))
    rwin = win[:int(np.searchsorted(np.cumsum(3 * bound), DUMP_ROW_LETTERS, side="right"))]
    ro, st, nr = d_rowoff.cpu().numpy()[rwin], d_stride.cpu().numpy()[rwin].astype(np.int64), nring[rwin].astype(np.int64)
    starts = (ro[:, None] + st[:, None] * np.arange(3)).ravel()      # window-major, rows ref / cor / unc
    lens = np.repeat(nr, 3)
    idx = np.repeat(starts - np.concatenate(([0], np.cumsum(lens)[:-1])), lens) + np.arange(int(lens.sum()))
    out["rows_window_index"] = rwin
    out["rows"] = d_rows[torch.from_numpy(idx).to(d_rows.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1)
    ap.add_argument("--reads", type=int, default=0, help="triplets per GPU (default: the config's full size, capped at 10000)")
    ap.add_argument("--cpu-triplets", type=int, default=0, help="triplets of the CPU baseline sample (default: sized for ~10-20 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-main-only", action="store_true", help="time only the headline wire format and the byte path")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the headline path computed as DIR/<name>.npy "
                                                          "(float64; per-window results and MSA rows of a fixed sample of windows). The same "
                                                          "arguments give the same inputs only from the same window source: compare dumps of "
                                                          "runs whose JSON line has the same config.windows_from (the windows are cut by "
                                                          "oracle/_ref/masterSplitter where it is built, else synthesised directly)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)

    import workloads
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    n_reads = args.reads or min(workloads.CONFIG_READS[args.config], 10000)
    ncores = os.cpu_count() or 1
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "poa"))
    workload_name = workloads.CONFIG_NAMES[args.config] + (" [%d triplets per GPU]" % n_reads)

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        kind = "reference" if have_ref else "port"
        # bounded sample: ~26 triplets/s/core for 10 kb reads (BASELINE.md section 2) -> ~15 s per step
        per_step = args.cpu_triplets or int(min(n_reads, max(16, ncores * 26 * 12)))
        wl = workloads.make_windows(args.config, per_step, 0)
        per_step = len(wl["read_first"]) - 1
        for _ in range(args.warmup):
            cpu_reference_throughput(wl, max(1, per_step // 8), ncores, kind)
        times, last = [], None
        for _ in range(max(1, args.steps)):
            last = cpu_reference_throughput(wl, per_step, ncores, kind)
            times.append(last["seconds"])
        val = per_step * len(times) / sum(times)
        sample = "first %d triplets (%d windows) of the workload per step" % (per_step, last["windows"])
        print(json.dumps({
            "impl": "reference", "metric": "triplets_per_sec", "value": val, "unit": "triplets/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "gcups": last["gcups"], "windows_per_sec": last["windows_per_s"],
            "config": {"workload": workload_name, "windows_from": wl["source"], "sample": sample},
            "cpu_baseline": {"value": val, "unit": "triplets/s", "cores": ncores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "triplets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ------------------------------------------------------------------ our arm
    # one rank per GPU: keep the rank's threads (and the pinned buffers they first touch) on the CPUs next to its GPU;
    # with 8 ranks the host side of the pipelined call is otherwise bound by cross-socket traffic
    full_affinity = os.sched_getaffinity(0)
    numa_cpus = None
    if world > 1 and not os.environ.get("ELECTOR_NO_AFFINITY"):
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
            numa_cpus = len(os.sched_getaffinity(0))
        except Exception:
            numa_cpus = None
    import ctypes
    import torch
    import elector_b200
    from elector_b200 import TALLY_FIELDS
    if world > 1:
        import torch.distributed as dist
        # rank 0 prints ONE JSON line on stdout: NCCL's log goes to stderr, and its version banner (a printf to stdout at
        # the VERSION and WARN levels) is switched off unless the caller asked for INFO or more
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K = len(TALLY_FIELDS)

    wl = workloads.make_windows(args.config, n_reads, rank * n_reads)
    n_trip = len(wl["read_first"]) - 1
    n = len(wl["ref_off"]) - 1
    ctx = elector_b200.PoaContext(device=local)
    lib = ctx._lib

    # host (pinned) and device copies of the inputs
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    hp = {k: pinned(wl[k]) for k in ("ref", "ref_off", "cor", "cor_off", "unc", "unc_off", "read_first")}
    dv = {k: hp[k][0].to(dev, non_blocking=False) for k in hp if k != "read_first"}
    hptr = {k: hp[k][1].ctypes.data for k in hp}
    bound = int(lib.elector_poa_rows_bound(n, hptr["ref_off"], hptr["cor_off"], hptr["unc_off"]))
    d_rows = torch.empty(bound, dtype=torch.uint8, device=dev)
    d_rowoff = torch.empty(n, dtype=torch.int64, device=dev)
    d_stride = torch.empty(n, dtype=torch.int32, device=dev)
    d_nring = torch.empty(n, dtype=torch.int32, device=dev)
    d_s1 = torch.empty(n, dtype=torch.int32, device=dev)
    d_s2 = torch.empty(n, dtype=torch.int32, device=dev)
    d_cells = torch.empty(n, dtype=torch.int64, device=dev)
    d_used = torch.zeros(1, dtype=torch.int64, device=dev)
    d_cnt = torch.zeros(n_trip * K, dtype=torch.int64, device=dev)
    d_sums = torch.zeros(K, dtype=torch.int64, device=dev)
    h_rows = torch.empty(bound, dtype=torch.uint8).pin_memory()
    h_out = {"row_off": torch.empty(n, dtype=torch.int64).pin_memory(), "stride": torch.empty(n, dtype=torch.int32).pin_memory(),
             "nring": torch.empty(n, dtype=torch.int32).pin_memory(), "counters": torch.empty(n_trip * K, dtype=torch.int64).pin_memory(),
             "sums": torch.empty(K, dtype=torch.int64).pin_memory()}
    h_used = torch.zeros(1, dtype=torch.int64).pin_memory()
    torch.cuda.synchronize()
    phase = {"p1": 0.0, "tot": 0.0, "launches": 0, "tally_ms": 0.0}

    def step_device():
        """inputs resident in HBM: POA (both phases) -> merge -> tally -> global counters [-> all-reduce]"""
        ctx._check(lib.elector_poa_run_device(ctx._ctx, n, dv["ref"].data_ptr(), dv["ref_off"].data_ptr(), dv["cor"].data_ptr(),
                                              dv["cor_off"].data_ptr(), dv["unc"].data_ptr(), dv["unc_off"].data_ptr(),
                                              hptr["ref_off"], hptr["cor_off"], hptr["unc_off"],
                                              d_rows.data_ptr(), bound, d_rowoff.data_ptr(), d_stride.data_ptr(), d_nring.data_ptr(),
                                              d_s1.data_ptr(), d_s2.data_ptr(), d_cells.data_ptr(), d_used.data_ptr()))
        a, b = ctypes.c_float(0), ctypes.c_float(0)
        lib.elector_last_phase_ms(ctx._ctx, ctypes.byref(a), ctypes.byref(b))
        m, k = ctx.last_kernel_ms()
        phase["p1"] += a.value; phase["tot"] += b.value; phase["launches"] += k
        h_used.copy_(d_used)
        ctx._check(lib.elector_merge_tally_device(ctx._ctx, n_trip, hptr["read_first"], n, d_rows.data_ptr(), int(h_used.item()),
                                                  d_rowoff.data_ptr(), d_stride.data_ptr(), d_nring.data_ptr(), d_cnt.data_ptr()))
        m, k = ctx.last_kernel_ms()
        phase["tally_ms"] += m; phase["launches"] += k
        d_sums.zero_()
        torch.cuda.current_stream().synchronize()   # the library launches on its own stream
        ctx._check(lib.elector_tally_sum_device(ctx._ctx, n_trip, d_cnt.data_ptr(), d_sums.data_ptr()))
        phase["launches"] += 1
        if world > 1:
            dist.all_reduce(d_sums)       # the one collective of the path: 24 int64 counters

    # ---- end to end: the call a user makes, host buffers in / out, copies inside the timed region ----
    # Four wire formats of the same call (include/elector_poa.h, elector_pipeline_run2).  The headline `e2e` is the first:
    # what ELECTOR consumes after alignment.py (the merged per-read MSA that Donatello appends to msa.fa, losslessly as 4-bit
    # columns, and the per-read counters of computeStats.py) from what its caller has (the reads, packed once outside the call).
    from elector_b200.poa import PipelineIoC, pack_letters
    packed = [pack_letters(wl[k]) for k in ("ref", "cor", "unc")]      # outside the timed region, like reading the FASTA files
    pk_pinned = []
    for pk in packed:
        t_bits, a_bits = pinned(pk.bits); t_pos, a_pos = pinned(pk.exc_pos if len(pk.exc_pos) else np.zeros(1, np.int64)); t_byt, a_byt = pinned(pk.exc_byte if len(pk.exc_byte) else np.zeros(1, np.uint8))
        pk_pinned.append((t_bits, t_pos, t_byt))
        pk.bits, n_e = a_bits, len(pk.exc_pos)
        pk.exc_pos, pk.exc_byte = a_pos[:n_e], a_byt[:n_e]
    pk_c = [pk.c_struct() for pk in packed]
    len32 = [pinned(np.diff(wl[k]).astype(np.int32)) for k in ("ref_off", "cor_off", "unc_off")]   # 32-bit window lengths: what crosses the link
    len16 = [pinned(np.diff(wl[k]).astype(np.uint16)) for k in ("ref_off", "cor_off", "unc_off")]  # ... or 16-bit ones (the headline mode)
    assert max(int(np.diff(wl[k]).max()) for k in ("ref_off", "cor_off", "unc_off")) < 65536
    m_cap = int(lib.elector_merged_bound(n, n_trip, hptr["ref_off"], hptr["cor_off"], hptr["unc_off"]))
    h_m = [torch.empty(m_cap, dtype=torch.uint8).pin_memory() for _ in range(3)]
    h_moff, h_mlen = torch.empty(n_trip, dtype=torch.int64).pin_memory(), torch.empty(n_trip, dtype=torch.int32).pin_memory()
    h_esc_pos, h_esc_byte, h_nesc = torch.empty(1 << 20, dtype=torch.int64).pin_memory(), torch.empty(1 << 20, dtype=torch.uint8).pin_memory(), torch.zeros(1, dtype=torch.int64)

    def make_io(mode):
        io = PipelineIoC()
        io.n_windows, io.n_reads = n, n_trip
        io.ref_off, io.cor_off, io.unc_off, io.read_first = hptr["ref_off"], hptr["cor_off"], hptr["unc_off"], hptr["read_first"]
        if mode != "packed_in_counters_out":
            io.nring = h_out["nring"].data_ptr()
        io.counters_out, io.sums_out = h_out["counters"].data_ptr(), h_out["sums"].data_ptr()
        if mode == "bytes_in_window_rows_out":
            io.ref, io.cor, io.unc = hptr["ref"], hptr["cor"], hptr["unc"]
            io.rows_out, io.rows_cap, io.row_off, io.row_stride = h_rows.data_ptr(), bound, h_out["row_off"].data_ptr(), h_out["stride"].data_ptr()
        else:
            io.pref, io.pcor, io.punc = (ctypes.addressof(c) for c in pk_c)
            if mode == "packed_in_merged_columns_out":
                io.ref_len16, io.cor_len16, io.unc_len16 = (t[1].ctypes.data for t in len16)
            else:
                io.ref_len, io.cor_len, io.unc_len = (t[1].ctypes.data for t in len32)
            if mode != "packed_in_counters_out":
                io.m_ref, io.m_cor, io.m_unc, io.m_cap = h_m[0].data_ptr(), h_m[1].data_ptr(), h_m[2].data_ptr(), m_cap
                io.m_off, io.m_len = h_moff.data_ptr(), h_mlen.data_ptr()
                if mode in ("packed_in_merged_nibbles_out", "packed_in_merged_columns_out"):
                    io.m_nibbles = 1 if mode == "packed_in_merged_nibbles_out" else 2
                    io.m_esc_pos, io.m_esc_byte, io.m_esc_cap, io.m_n_esc = h_esc_pos.data_ptr(), h_esc_byte.data_ptr(), 1 << 20, h_nesc.data_ptr()
        return io

    E2E_MODES = ["packed_in_merged_columns_out", "packed_in_merged_nibbles_out", "bytes_in_window_rows_out", "packed_in_merged_rows_out", "packed_in_counters_out"]
    ios = {m: make_io(m) for m in E2E_MODES}

    def make_step(mode):
        io = ios[mode]

        def step():
            ctx._check(lib.elector_pipeline_run2(ctx._ctx, ctypes.byref(io)))
            if world > 1:
                t = h_out["sums"].to(dev)
                dist.all_reduce(t)
                h_out["sums"].copy_(t)
        return step
    step_e2e = make_step(E2E_MODES[0])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """device time of `steps` calls: CUDA events on the library's launching stream, max over ranks"""
        barrier()
        ctx._check(lib.elector_event_record(ctx._ctx, 0))
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        ctx._check(lib.elector_event_record(ctx._ctx, 1))
        ms = ctypes.c_float(0)
        ctx._check(lib.elector_event_elapsed_ms(ctx._ctx, ctypes.byref(ms)))
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        barrier()
        t = torch.tensor([max(ms.value, 0.0), wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    for _ in range(args.warmup):
        step_device()
    for k in phase:
        phase[k] = 0
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, dev_wall = timed(step_device, args.steps)
    clocks = sampler.summary()
    # the library's stream events bracket the steps; the tally launches and the all-reduce end on other streams, so the
    # wall clock around the synchronised loop is the safe upper bound: report the larger of the two
    step_ms = max(dev_ms, dev_wall) / args.steps
    cells = int(d_cells.sum().item())
    used = int(d_used.item())
    sums_dev = d_sums.cpu().numpy().copy()
    e2e_modes = {}
    nesc = {"packed_in_merged_nibbles_out": 0, "packed_in_merged_columns_out": 0}
    sums_e2e = None
    for mode in (E2E_MODES if not args.e2e_main_only else E2E_MODES[:3]):
        fn = make_step(mode)
        for _ in range(args.warmup):
            fn()
        ms_, wall_ = timed(fn, args.steps)
        e2e_modes[mode] = max(ms_, wall_) / args.steps
        if mode in nesc:
            nesc[mode] = int(h_nesc[0])
        if mode == E2E_MODES[0]:
            sums_e2e = h_out["sums"].numpy().copy()
            merged_cols = int(h_mlen.numpy().astype(np.int64).sum())
    e2e_step_ms = e2e_modes[E2E_MODES[0]]
    # the byte path once more, last: the parity check below reads its window rows
    step_rows = make_step("bytes_in_window_rows_out")
    step_rows()

    # parity spot check of what was just timed (not in the timed region): first 2000 windows vs the oracle,
    # and the two paths (device-resident / pipelined host call) against each other
    parity = None
    try:
        from oracle import oracle
        k = min(n, 2000)
        o = oracle.batch(wl["ref"], wl["ref_off"][:k + 1], wl["cor"], wl["cor_off"][:k + 1], wl["unc"], wl["unc_off"][:k + 1], nthreads=min(8, ncores))
        nr = h_out["nring"].numpy()[:k]
        ok = bool(np.array_equal(nr, o["nring"]))
        rows = h_rows.numpy()
        ro, st = h_out["row_off"].numpy(), h_out["stride"].numpy()
        for w in range(k):
            if not ok:
                break
            for s in range(3):
                a = rows[ro[w] + s * st[w]: ro[w] + s * st[w] + nr[w]]
                b = o["rows"][o["row_off"][w] + s * nr[w]: o["row_off"][w] + (s + 1) * nr[w]]
                if not np.array_equal(a, b):
                    ok = False
                    break
        ok = ok and bool(np.array_equal(sums_dev, sums_e2e))
        ok = ok and bool(np.array_equal(h_out["counters"].numpy(), d_cnt.cpu().numpy()))
        parity = "bit-exact vs oracle on %d windows; device and host paths agree on all per-read counters" % k if ok else "MISMATCH"
    except Exception as e:  # the oracle is only a checker here
        parity = "not checked (%s)" % e

    # roofline of the dominant kernel (poa_dp2_kernel: DP2 phase incl. its sort), and of the DP1 phase beside it
    mixed, alu = ctypes.c_double(0), ctypes.c_double(0)
    ctx._check(lib.elector_int32_peak(ctx._ctx, ctypes.byref(mixed), ctypes.byref(alu)))
    lr, lc = np.diff(wl["ref_off"]), np.diff(wl["cor_off"])
    cells1 = int((lr * lc).sum())
    # DP1 cells the kernels really sweep: windows whose corrected letters are the reference letters are recognised by
    # the size sort and skip phase 1 (their DP1 has one possible result); the algorithmic count above includes them
    lu_ = np.diff(wl["unc_off"])
    cand = np.flatnonzero((lr == lc) & (lr <= 256) & (lu_ <= 256))
    if len(cand):
        ln = lr[cand]
        pos = np.arange(int(ln.sum()), dtype=np.int64) - np.repeat(np.cumsum(ln) - ln, ln)
        diff = wl["ref"][np.repeat(wl["ref_off"][cand], ln) + pos] != wl["cor"][np.repeat(wl["cor_off"][cand], ln) + pos]
        ident = cand[np.add.reduceat(diff.astype(np.int32), np.cumsum(ln) - ln) == 0]
    else:
        ident = cand
    cells1_swept = cells1 - int((lr[ident] * lc[ident]).sum())
    cells2 = cells - cells1
    p1_s = phase["p1"] / 1e3 / args.steps
    p2_s = (phase["tot"] - phase["p1"]) / 1e3 / args.steps
    poa_s = phase["tot"] / 1e3 / args.steps
    ach2 = INT_OPS_PER_CELL * cells2 / p2_s / 1e12
    ach1 = INT_OPS_PER_CELL * cells1 / p1_s / 1e12
    hbm_peak = 6552.6
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    issue = None
    try:   # ncu view of the same launch set (tools/ncu_issue.py on the launch list of the round's evidence run)
        issue = json.load(open(os.path.join(ROOT, "profiles", "issue.json")))
    except Exception:
        pass
    letters = int(wl["ref_off"][-1] + wl["cor_off"][-1] + wl["unc_off"][-1])
    in_bytes = letters + 3 * 8 * (n + 1) + 8 * (n_trip + 1)                     # byte path: 1 B per letter, 64-bit offsets
    in_packed = sum((pk.n_letters + 3) // 4 + 9 * len(pk.exc_pos) for pk in packed) + 3 * 4 * n + 8 * (n_trip + 1)
    out_rows = used + n * (8 + 4 + 4) + n_trip * K * 8 + K * 8                   # byte path: window rows, their offsets, counters
    out_merged = 3 * merged_cols + n * 4 + n_trip * (8 + 4 + K * 8) + K * 8     # merged rows as bytes, nring, m_off / m_len, counters
    wire = {"packed_in_merged_rows_out": (in_packed, out_merged), "bytes_in_window_rows_out": (in_bytes, out_rows),
            "packed_in_merged_nibbles_out": (in_packed, out_merged - 3 * merged_cols + 3 * ((merged_cols + 1) // 2) + 9 * nesc["packed_in_merged_nibbles_out"]),
            "packed_in_merged_columns_out": (in_packed - 3 * 2 * n, out_merged - 2 * merged_cols + 9 * nesc["packed_in_merged_columns_out"]),
            "packed_in_counters_out": (in_packed, n_trip * K * 8 + K * 8)}
    out_bytes = wire[E2E_MODES[0]][1]
    alg_bytes = in_bytes + used + n * 36

    value = n_trip * world / (step_ms / 1e3)
    e2e_val = n_trip * world / (e2e_step_ms / 1e3)
    line = {
        "metric": "triplets_per_sec", "value": value, "unit": "triplets/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "s16x2 (packed halfword integer SIMD; int32 for scores beyond 16 bits)", "data": "synthetic",
        "gcups": cells * world / (step_ms / 1e3) / 1e9,
        "gcups_poa_kernels_only": cells / poa_s / 1e9,
        "windows_per_sec": n * world / (step_ms / 1e3),
        "config": {"workload": workload_name, "step": "POA of every window (DP1 + DP2 phases) + per-read merge + tally + counter sum",
                   "windows_per_gpu": n, "cells_per_gpu": cells, "windows_from": wl["source"],
                   "l2": "inputs (%.0f MB per step) larger than the 126 MB L2, no flush" % (in_bytes / 1e6), "parity": parity},
        "e2e": {"value": e2e_val, "unit": "triplets/s", "h2d_bytes_per_step": wire[E2E_MODES[0]][0], "d2h_bytes_per_step": out_bytes,
                "ms_per_step": e2e_step_ms,
                "call": "elector_pipeline_run2: 2-bit packed letters + 16-bit window lengths in (packed once, outside the call), merged per-read MSA rows (what Donatello appends to msa.fa) as one byte per column (the three rows' characters base 6, ELECTOR_COLUMN_CHARS) + per-read counters + sums out; pinned host buffers",
                "host_link_gbs": (wire[E2E_MODES[0]][0] + out_bytes) / (e2e_step_ms / 1e3) / 1e9,
                "limiter": "kernels (%.2f ms resident) + the tail of the last chunk's results; the host link carries %.0f MB per call" % (step_ms, (wire[E2E_MODES[0]][0] + out_bytes) / 1e6),
                "modes": {m: {"ms_per_step": e2e_modes[m], "value": n_trip * world / (e2e_modes[m] / 1e3), "h2d_bytes_per_step": wire[m][0], "d2h_bytes_per_step": wire[m][1],
                              "host_link_gbs": (wire[m][0] + wire[m][1]) / (e2e_modes[m] / 1e3) / 1e9} for m in e2e_modes}},
        "gpu_launches": phase["launches"],
        "kernel_ms_per_step": {"sort1+poa_dp1_kernel": phase["p1"] / args.steps, "sort2+poa_dp2_kernel": (phase["tot"] - phase["p1"]) / args.steps,
                               "merge+tally": phase["tally_ms"] / args.steps},
        "clocks": clocks,
        "roofline": {"bound": "int32", "achieved": ach2, "peak": mixed.value, "unit": "TIOP/s",
                     "frac": ach2 / mixed.value if mixed.value else None,
                     "traffic": (traffic or {}).get("poa_dp2_kernel_bytes_per_launch_set"),
                     "kernel": "poa_dp2_kernel (all segment launches of one step, with its sort)",
                     "ops_per_cell": INT_OPS_PER_CELL, "cells_per_step": cells2,
                     "cells_swept_per_step": cells2,   # every window runs DP2 (the diagonal band of the linear kernels skips cells inside a window; not counted)
                     "issue": None if not issue else {
                         "warp_instructions_per_step": issue["phase2_warp_instructions_per_launch_set"],
                         "thread_instructions_per_cell": issue["phase2_warp_instructions_per_launch_set"] * 32 / cells2,
                         "ipc_active": issue["ipc_active_time_weighted"], "ipc_peak": 4.0,
                         "issue_slot_utilisation": issue["phase2_warp_instructions_per_launch_set"] / (p2_s * (clocks.get("sm_mhz") or 1965.0) * 1e6 * n_sm * 4),
                         "issue_slot_utilisation_note": "warp instructions of the launch set (ncu) / (4 issue slots x SMs x SM clock x the phase-2 time measured live)",
                         "alu_pipe_pct": issue["alu_pipe_pct_time_weighted"],
                         "source": "profiles/issue.json (ncu launch list of the same command, cold-cache and serialised)"},
                     "peak_alu_pipe_only": alu.value,
                     "peak_source": "measured on this device by elector_int32_peak (IMAD/IADD3/VIMNMX/LOP3 chains)",
                     "also": {"kernel": "poa_dp1_kernel", "achieved": ach1, "frac": ach1 / mixed.value if mixed.value else None,
                              "cells_per_step": cells1, "cells_swept_per_step": cells1_swept,
                              "note": "algorithmic cells (SURVEY.md 8d); %d of %d windows have cor == ref and skip DP1, the kernels sweep cells_swept_per_step" % (len(ident), n)}},
        "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / poa_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": alg_bytes / poa_s / 1e9 / hbm_peak, "traffic": (traffic or {}).get("poa_step_dram_bytes"),
                         "note": "algorithmic bytes = letters + offsets in, MSA rows + per-window results out; the path is integer-issue bound, not HBM bound"},
        "counters": {f: int(v) for f, v in zip(TALLY_FIELDS, sums_dev) if f in ("TP", "FP", "FN", "insU", "delU", "subsU", "insC", "delC", "subsC", "assessed")},
    }
    os.sched_setaffinity(0, full_affinity)   # the CPU baseline below uses every host core
    if numa_cpus:
        line["config"]["host_affinity"] = "rank threads bound to the %d CPUs next to their GPU (NVML)" % numa_cpus
    if rank == 0 and not args.no_cpu_baseline:
        kind = "reference" if have_ref else "port"
        k = args.cpu_triplets or int(min(n_trip, max(8, ncores * 26 * 10)))
        cb = cpu_reference_throughput(wl, k, ncores, kind)
        line["cpu_baseline"] = {"value": cb["triplets_per_s"], "unit": "triplets/s", "cores": ncores, "kind": kind,
                                "sample": "first %d triplets (%d windows), %.1f s, %d concurrent single-threaded poa processes (alignment only, no Donatello / computeStats)" %
                                          (k, cb["windows"], cb["seconds"], ncores) if kind == "reference" else
                                          "first %d triplets (%d windows), %.1f s, oracle with %d OpenMP threads" % (k, cb["windows"], cb["seconds"], ncores),
                                "gcups": cb["gcups"]}
    if rank == 0:
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, wl, d_rows, d_rowoff, d_stride, d_nring, d_s1, d_s2, d_cells, d_cnt, d_sums)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
