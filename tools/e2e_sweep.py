#!/usr/bin/env python3
"""Host-clock time of elector_pipeline_run2 per wire format and chunk count (config 1, 10 000 reads).
  python tools/e2e_sweep.py [reads]"""
import ctypes, os, subprocess, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
if len(sys.argv) > 2 and sys.argv[2] == "child":
    import numpy as np, torch, workloads, elector_b200
    from elector_b200.poa import PipelineIoC, pack_letters
    wl = workloads.make_windows(1, int(sys.argv[1]))
    n, nr = len(wl["ref_off"]) - 1, len(wl["read_first"]) - 1
    ctx = elector_b200.PoaContext(0); lib = ctx._lib
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    keep = []
    pks = []
    for k in ("ref", "cor", "unc"):
        pk = pack_letters(wl[k]); t = pin(pk.bits); keep.append(t); pk.bits = t.numpy(); pks.append(pk)
    pc = [p.c_struct() for p in pks]
    offs = {k: pin(wl[k]) for k in ("ref_off", "cor_off", "unc_off", "read_first")}
    lens = [pin(np.diff(wl[k]).astype(np.int32)) for k in ("ref_off", "cor_off", "unc_off")]
    cap = int(lib.elector_merged_bound(n, nr, offs["ref_off"].data_ptr(), offs["cor_off"].data_ptr(), offs["unc_off"].data_ptr()))
    m = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(3)]
    moff, mlen = torch.empty(nr, dtype=torch.int64).pin_memory(), torch.empty(nr, dtype=torch.int32).pin_memory()
    cnt, sums = torch.empty(nr * 24, dtype=torch.int64).pin_memory(), torch.empty(24, dtype=torch.int64).pin_memory()
    ep, eb, ne = torch.empty(1 << 20, dtype=torch.int64).pin_memory(), torch.empty(1 << 20, dtype=torch.uint8).pin_memory(), torch.zeros(1, dtype=torch.int64)
    for mode in ("merged", "nibbles", "counters"):
        io = PipelineIoC(); io.n_windows, io.n_reads = n, nr
        io.pref, io.pcor, io.punc = (ctypes.addressof(c) for c in pc)
        io.ref_off, io.cor_off, io.unc_off, io.read_first = (offs[k].data_ptr() for k in ("ref_off", "cor_off", "unc_off", "read_first"))
        io.counters_out, io.sums_out = cnt.data_ptr(), sums.data_ptr()
        io.ref_len, io.cor_len, io.unc_len = (l.data_ptr() for l in lens)
        if mode != "counters":
            io.m_ref, io.m_cor, io.m_unc, io.m_cap, io.m_off, io.m_len = m[0].data_ptr(), m[1].data_ptr(), m[2].data_ptr(), cap, moff.data_ptr(), mlen.data_ptr()
            if mode == "nibbles":
                io.m_nibbles, io.m_esc_pos, io.m_esc_byte, io.m_esc_cap, io.m_n_esc = 1, ep.data_ptr(), eb.data_ptr(), 1 << 20, ne.data_ptr()
        ts = []
        for i in range(8):
            t0 = time.perf_counter(); ctx._check(lib.elector_pipeline_run2(ctx._ctx, ctypes.byref(io))); ts.append((time.perf_counter() - t0) * 1e3)
        print("%-9s chunks=%s workers=%s: %.2f ms (best of last 5: %.2f)" % (mode, os.environ.get("ELECTOR_PIPELINE_CHUNKS", "auto"), os.environ.get("ELECTOR_PIPELINE_WORKERS", "3"),
              sum(ts[3:]) / 5, min(ts[3:])), flush=True)
else:
    reads = sys.argv[1] if len(sys.argv) > 1 else "10000"
    for env in ({}, {"ELECTOR_PIPELINE_CHUNKS": "1"}, {"ELECTOR_PIPELINE_CHUNKS": "2"}, {"ELECTOR_PIPELINE_CHUNKS": "4"}):
        subprocess.call([sys.executable, __file__, reads, "child"], env=dict(os.environ, **env))
