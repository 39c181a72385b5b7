#!/usr/bin/env python3
"""Device timeline of the resident step that bench.py times (elector_poa_run_device, elector_merge_tally_device,
elector_tally_sum_device on config-1 windows already in HBM), under torch.profiler with CUDA activities.

  python tools/step_timeline.py [--out DIR] [--reads N] [--warmup W] [--steps K]      (DIR defaults to <tmp>/elector_step_timeline)
  python tools/step_timeline.py --trace DIR/step_timeline.pt.trace.json [--out DIR]    (summary of a saved trace; no GPU)

Writes DIR/step_timeline.pt.trace.json (the profiler trace) and DIR/summary.json / DIR/summary.txt:
  - every kernel of the last profiled step: name, stream, start and end (us from the step's first kernel);
  - device-idle time (no kernel running on any stream) per region of the step: before phase 1, during phase 1, between the
    phases, during phase 2, after phase 2; and after the last bulk launch of each phase until the next DP kernel;
  - the gap between the end of the last phase-1 bulk kernel and the start of the first phase-2 bulk kernel;
  - the duration of every sort and plan kernel;
medians over the profiled steps where a figure is per step.  Run it in a process of its own: the profiler slows the host,
so its step times are not bench.py's."""
import argparse
import ctypes
import json
import os
import statistics
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SORT_KERNELS = ("init_call_kernel", "bin1_count_kernel", "bin_scan_chunks_kernel", "bin_scan_totals_kernel", "bin_scatter_kernel",
                "plan_segments_kernel")


def short(name):
    """kernel name without its return type, namespace and parameter list (template arguments kept)"""
    n = name.replace("(anonymous namespace)::", "").replace("elector::", "").split("(")[0]
    return n[5:] if n.startswith("void ") else n


def dp_phase(name):
    if name.startswith("poa_dp1"):
        return 1
    if name.startswith("poa_dp2"):
        return 2
    return 0


def is_bulk(name):
    return dp_phase(name) and "coop" not in name


def idle_within(busy, t0, t1):
    """time in [t0, t1) covered by no interval of `busy` (sorted, merged)"""
    if t1 <= t0:
        return 0.0
    idle, cur = 0.0, t0
    for a, b in busy:
        if b <= cur:
            continue
        if a >= t1:
            break
        if a > cur:
            idle += a - cur
        cur = max(cur, b)
        if cur >= t1:
            break
    return idle + max(0.0, t1 - cur)


def merged(iv):
    out = []
    for a, b in sorted(iv):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def analyse_step(ks):
    """ks: kernels of one step (dicts name / stream / t0 / t1, us, absolute).  Figures of the step, times relative to its start."""
    s0 = min(k["t0"] for k in ks)
    s1 = max(k["t1"] for k in ks)
    busy = merged([(k["t0"], k["t1"]) for k in ks])
    p1 = [k for k in ks if dp_phase(k["name"]) == 1]
    p2 = [k for k in ks if dp_phase(k["name"]) == 2]
    r = {"step_us": s1 - s0, "idle_us": {}, "tail_idle_us": {}}
    p1s = min((k["t0"] for k in p1), default=None)
    p1e = max((k["t1"] for k in p1), default=None)
    p2s = min((k["t0"] for k in p2), default=None)
    p2e = max((k["t1"] for k in p2), default=None)
    if p1s is not None and p2s is not None:
        r["idle_us"] = {"before_phase1": idle_within(busy, s0, p1s), "during_phase1": idle_within(busy, p1s, p1e),
                        "between_phases": idle_within(busy, p1e, p2s) if p2s > p1e else 0.0,
                        "during_phase2": idle_within(busy, max(p2s, p1e), p2e), "after_phase2": idle_within(busy, p2e, s1)}
        r["phase1_us"] = [p1s - s0, p1e - s0]
        r["phase2_us"] = [p2s - s0, p2e - s0]
    b1 = [k for k in p1 if is_bulk(k["name"])]
    b2 = [k for k in p2 if is_bulk(k["name"])]
    dp = sorted(p1 + p2, key=lambda k: k["t0"])
    for tag, bl in (("phase1", b1), ("phase2", b2)):
        if not bl:
            continue
        last = max(bl, key=lambda k: k["t1"])
        nxt = min((k["t0"] for k in dp if k["t0"] >= last["t1"]), default=s1)
        r["tail_idle_us"]["after_last_bulk_" + tag] = idle_within(busy, last["t1"], nxt)
    if b1 and b2:
        r["gap_bulk1_end_to_bulk2_start_us"] = min(k["t0"] for k in b2) - max(k["t1"] for k in b1)
    r["sort_plan_us"] = {}
    for k in ks:
        base = k["name"].split("<")[0]
        if base in SORT_KERNELS:
            r["sort_plan_us"].setdefault(base, []).append(round(k["t1"] - k["t0"], 2))
    r["sort_plan_total_us"] = sum(sum(v) for v in r["sort_plan_us"].values())
    r["kernels"] = [{"name": k["name"], "stream": k["stream"], "start_us": round(k["t0"] - s0, 2), "end_us": round(k["t1"] - s0, 2)}
                    for k in sorted(ks, key=lambda k: k["t0"])]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "elector_step_timeline"))   # outside the tree: it may be read-only
    ap.add_argument("--config", type=int, default=1)
    ap.add_argument("--reads", type=int, default=10000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--trace", help="summarise this saved trace instead of running the step")
    args = ap.parse_args()
    if args.trace:
        return summarise(args.trace, args.out, None)
    import torch
    from torch.profiler import ProfilerActivity, profile
    import elector_b200
    import workloads
    from elector_b200 import TALLY_FIELDS

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    wl = workloads.make_windows(args.config, args.reads, 0)
    n_trip, n = len(wl["read_first"]) - 1, len(wl["ref_off"]) - 1
    ctx = elector_b200.PoaContext(device=0)
    lib = ctx._lib
    # the buffers and calls of bench.py's resident step
    hp = {k: torch.from_numpy(np.ascontiguousarray(wl[k])).pin_memory() for k in ("ref", "ref_off", "cor", "cor_off", "unc", "unc_off", "read_first")}
    hptr = {k: hp[k].numpy().ctypes.data for k in hp}
    dv = {k: hp[k].to(dev) for k in hp if k != "read_first"}
    bound = int(lib.elector_poa_rows_bound(n, hptr["ref_off"], hptr["cor_off"], hptr["unc_off"]))
    d_rows = torch.empty(bound, dtype=torch.uint8, device=dev)
    d_rowoff = torch.empty(n, dtype=torch.int64, device=dev)
    d_stride, d_nring, d_s1, d_s2 = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(4))
    d_cells = torch.empty(n, dtype=torch.int64, device=dev)
    d_used = torch.zeros(1, dtype=torch.int64, device=dev)
    d_cnt = torch.zeros(n_trip * len(TALLY_FIELDS), dtype=torch.int64, device=dev)
    d_sums = torch.zeros(len(TALLY_FIELDS), dtype=torch.int64, device=dev)
    h_used = torch.zeros(1, dtype=torch.int64).pin_memory()
    torch.cuda.synchronize()

    def step():
        ctx._check(lib.elector_poa_run_device(ctx._ctx, n, dv["ref"].data_ptr(), dv["ref_off"].data_ptr(), dv["cor"].data_ptr(),
                                              dv["cor_off"].data_ptr(), dv["unc"].data_ptr(), dv["unc_off"].data_ptr(),
                                              hptr["ref_off"], hptr["cor_off"], hptr["unc_off"],
                                              d_rows.data_ptr(), bound, d_rowoff.data_ptr(), d_stride.data_ptr(), d_nring.data_ptr(),
                                              d_s1.data_ptr(), d_s2.data_ptr(), d_cells.data_ptr(), d_used.data_ptr()))
        h_used.copy_(d_used)
        ctx._check(lib.elector_merge_tally_device(ctx._ctx, n_trip, hptr["read_first"], n, d_rows.data_ptr(), int(h_used.item()),
                                                  d_rowoff.data_ptr(), d_stride.data_ptr(), d_nring.data_ptr(), d_cnt.data_ptr()))
        d_sums.zero_()
        torch.cuda.current_stream().synchronize()
        ctx._check(lib.elector_tally_sum_device(ctx._ctx, n_trip, d_cnt.data_ptr(), d_sums.data_ptr()))
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    os.makedirs(args.out, exist_ok=True)
    trace = os.path.join(args.out, "step_timeline.pt.trace.json")
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
    prof.export_chrome_trace(trace)
    ctx.close()
    head = {"device": torch.cuda.get_device_name(0), "config": args.config, "reads": args.reads, "windows": n}
    try:
        import subprocess
        head["power_limit_clocks"] = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                                                     "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception:
        pass
    json.dump(head, open(os.path.join(args.out, "run.json"), "w"))
    summarise(trace, args.out, head)


def summarise(trace, out, head):
    """summary.json / summary.txt of a saved trace; head = what the run knew (device, config, windows), else DIR/run.json"""
    if head is None:
        head = json.load(open(os.path.join(os.path.dirname(os.path.abspath(trace)), "run.json")))
    os.makedirs(out, exist_ok=True)
    ev = json.load(open(trace))
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    ks = [{"name": short(e["name"]), "stream": e.get("args", {}).get("stream"), "t0": float(e["ts"]), "t1": float(e["ts"]) + float(e.get("dur", 0))}
          for e in ev if e.get("ph") == "X" and e.get("cat") == "kernel"]
    ks.sort(key=lambda k: k["t0"])
    # a step starts with init_call_kernel (run_device's first launch)
    starts = [i for i, k in enumerate(ks) if k["name"].startswith("init_call_kernel")]
    steps = [ks[a:b] for a, b in zip(starts, starts[1:] + [len(ks)])]
    per = [analyse_step(s) for s in steps]
    med = lambda xs: round(statistics.median(xs), 2) if xs else None   # noqa: E731
    summ = dict(head)
    summ.update({"steps": len(per),
            "step_us": med([p["step_us"] for p in per]),
            "idle_us": {k: med([p["idle_us"].get(k, 0.0) for p in per]) for k in per[-1]["idle_us"]},
            "tail_idle_us": {k: med([p["tail_idle_us"].get(k, 0.0) for p in per]) for k in per[-1]["tail_idle_us"]},
            "gap_bulk1_end_to_bulk2_start_us": med([p.get("gap_bulk1_end_to_bulk2_start_us", 0.0) for p in per]),
            "sort_plan_total_us": med([p["sort_plan_total_us"] for p in per]),
            "phase1_us": per[-1].get("phase1_us"), "phase2_us": per[-1].get("phase2_us"),
            "sort_plan_us_last_step": per[-1]["sort_plan_us"], "kernels_last_step": per[-1]["kernels"]})
    json.dump(summ, open(os.path.join(out, "summary.json"), "w"), indent=1)
    with open(os.path.join(out, "summary.txt"), "w") as f:
        f.write("%s  config %d, %d windows, median of %d profiled steps (profiler on: host gaps are longer than in bench.py)\n"
                % (summ["device"], summ["config"], summ["windows"], len(per)))
        f.write("%s\n" % summ.get("power_limit_clocks", ""))
        f.write("step (first to last kernel) %.1f us\n" % summ["step_us"])
        f.write("device idle (us): %s\n" % json.dumps(summ["idle_us"]))
        f.write("idle after the last bulk launch of a phase (us): %s\n" % json.dumps(summ["tail_idle_us"]))
        f.write("last phase-1 bulk end -> first phase-2 bulk start: %s us\n" % summ["gap_bulk1_end_to_bulk2_start_us"])
        f.write("sort + plan kernels, total %s us; last step: %s\n" % (summ["sort_plan_total_us"], json.dumps(summ["sort_plan_us_last_step"])))
        f.write("kernels of the last step (start, end in us from its first kernel; stream):\n")
        for k in summ["kernels_last_step"]:
            f.write("  %9.1f %9.1f  s%-4s %s\n" % (k["start_us"], k["end_us"], k["stream"], k["name"][:110]))
    print(open(os.path.join(out, "summary.txt")).read())


if __name__ == "__main__":
    main()
