#!/usr/bin/env python3
"""Reads in, per-triplet counters out: a BASELINE.json config at its stated size (or N_READS triplets) held in host memory and run
through three arms in one process, alternating them, each REPEATS times after one warm-up call:
  loop      the per-chunk elector_reads_run loop of tools/config_bench.py (pageable buffers, one call per CHUNK triplets)
  pipe_one_device   elector_reads_pipeline_run on the context's device
  pipe_all_devices  elector_reads_pipeline_run on every visible device
  pinned    (--pinned) pipe_one_device with the input buffers registered (cudaHostRegister, portable) around the call; the
            registration is inside the timed region
--sweep 1,2,4 adds one pipe_one_device arm per forced chunk count (ELECTOR_PIPELINE_CHUNKS).  Every arm must give the same sums.  One JSON line
per arm: host clock (median and all repeats), device time (CUDA events of the three stages, summed over chunks), triplets/s, and the
GPU name and power limit (nvidia-smi, query only).
  python tools/reads_bench.py CONFIG [N_READS] [--repeats R] [--sweep LIST] [--pinned]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import elector_b200  # noqa: E402
import workloads  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("config", type=int)
ap.add_argument("n_reads", type=int, nargs="?", default=0)
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--sweep", default="")
ap.add_argument("--pinned", action="store_true")
args = ap.parse_args()
cfg = args.config
total = args.n_reads if args.n_reads > 0 else workloads.CONFIG_READS[cfg]
loop_chunk = {1: 10000, 2: 10000, 3: 2000, 4: 20000}[cfg]


def generate():
    """the triplets of the config, generated in slices in parallel and concatenated (reference / uncorrected / corrected)"""
    gen = workloads.ensure_gen()
    work = tempfile.mkdtemp(prefix="readsbench_")

    def part(first):
        pre = os.path.join(work, "r%d" % first)
        subprocess.check_call([gen, str(cfg), str(min(loop_chunk, total - first)), str(first), pre])
        got = []
        for k in ("ref", "unc", "cor"):
            h, let, off = workloads.parse_two_line_fasta(pre + "." + k + ".fa")
            os.remove(pre + "." + k + ".fa")
            got.append((h, let, off))
        return got
    with ThreadPoolExecutor(max(1, (os.cpu_count() or 2) - 1)) as ex:
        parts = list(ex.map(part, range(0, total, loop_chunk)))
    os.rmdir(work)
    out = []
    for k in range(3):
        lets = [p[k][1] for p in parts]
        offs, base = [np.zeros(1, np.int64)], 0
        for p in parts:
            offs.append(p[k][2][1:] + base)
            base += int(p[k][2][-1])
        out += [np.concatenate(lets), np.concatenate(offs)]
    hl = np.asarray([len(h) for p in parts for h in p[0][0]], np.int32)
    return tuple(out) + (hl,)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [line.strip() for line in q.stdout.splitlines() if line.strip()]


ref, ro, unc, uo, cor, co, hl = generate()
n = len(hl)
K = len(elector_b200.TALLY_FIELDS)
import torch  # noqa: E402  (device count and cudaHostRegister of the pinned arm)
n_dev = torch.cuda.device_count()


def loop(ctx):
    sums, ms, nw = np.zeros(K, np.int64), np.zeros(3), 0
    for t0 in range(0, n, loop_chunk):
        t1 = min(n, t0 + loop_chunk)
        got = ctx.reads_run(ref, ro[t0:t1 + 1], unc, uo[t0:t1 + 1], cor, co[t0:t1 + 1], hl[t0:t1], 0.1)
        sums += got["sums"]; ms += ctx.last_reads_ms(); nw += got["n_windows"]
    return sums, ms, nw


def pipe(devices):
    def run(ctx):
        got = ctx.reads_pipeline(ref, ro, unc, uo, cor, co, hl, 0.1, devices=devices)
        return got["sums"], np.asarray(ctx.last_reads_ms()), got["n_windows"]
    return run


def forced(chunks, devices):
    def run(ctx):
        os.environ["ELECTOR_PIPELINE_CHUNKS"] = str(chunks)
        try:
            return pipe(devices)(ctx)
        finally:
            del os.environ["ELECTOR_PIPELINE_CHUNKS"]
    return run


def pinned(ctx):
    rt = torch.cuda.cudart()
    bufs = [ref, ro, unc, uo, cor, co, hl]
    for b in bufs:
        assert int(rt.cudaHostRegister(b.ctypes.data, b.nbytes, 1)) == 0   # cudaHostRegisterPortable: every device reads them
    try:
        return pipe([0])(ctx)
    finally:
        for b in bufs:
            rt.cudaHostUnregister(b.ctypes.data)


arms = [("loop", loop), ("pipe_one_device", pipe([0])), ("pipe_all_devices", pipe(list(range(n_dev))))]
if args.pinned:
    arms.append(("pinned", pinned))
for c in [int(v) for v in args.sweep.split(",") if v]:
    arms.append(("pipe_one_device_chunks%d" % c, forced(c, [0])))
res = {name: dict(host=[], dev=None, sums=None, nw=None) for name, _ in arms}
with elector_b200.PoaContext(0) as ctx:
    for rep in range(args.repeats + 1):        # repeat 0 warms every arm up (scratch pools, worker contexts)
        for name, fn in arms:
            t0 = time.perf_counter()
            sums, ms, nw = fn(ctx)
            dt = (time.perf_counter() - t0) * 1e3
            r = res[name]
            if r["sums"] is None:
                r["sums"], r["nw"] = sums.copy(), nw
            assert np.array_equal(r["sums"], sums) and r["nw"] == nw, name
            if rep:
                r["host"].append(dt)
                r["dev"] = ms if r["dev"] is None else r["dev"] + ms
first = res[arms[0][0]]
info = gpu_info()
letters = int(ro[-1] + uo[-1] + co[-1])
for name, _ in arms:
    r = res[name]
    assert np.array_equal(r["sums"], first["sums"]), "arm %s gives other sums than %s" % (name, arms[0][0])
    host = float(np.median(r["host"]))
    dev = r["dev"] / args.repeats
    out = {"arm": name, "config": cfg, "workload": workloads.CONFIG_NAMES[cfg], "stated_size": workloads.CONFIG_READS[cfg], "triplets": n,
           "windows": int(r["nw"]), "letters": letters, "repeats": args.repeats, "host_clock_ms": round(host, 1),
           "host_clock_ms_all": [round(v, 1) for v in r["host"]],
           "device_ms": {"split_ms": round(dev[0], 2), "poa_ms": round(dev[1], 2), "merge_tally_ms": round(dev[2], 2)},
           "device_ms_total": round(float(dev.sum()), 2), "triplets_per_s_host_clock": round(n / host * 1e3),
           "triplets_per_s_device": round(n / float(dev.sum()) * 1e3), "visible_devices": n_dev,
           "loop_chunk_triplets": loop_chunk if name == "loop" else None, "gpus": info,
           "counters": {k: int(r["sums"][elector_b200.TALLY_FIELDS.index(k)]) for k in ("TP", "FP", "FN", "assessed")}}
    print(json.dumps(out), flush=True)
