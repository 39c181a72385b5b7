"""GPU: merge (Donatello) + tally (computeStats) kernels through the C-ABI against the
reference-generated goldens and the oracle.  The reads at the kernels' own edges (long reads, word and step edges of
the scanners, gap stretches, row offsets) are in tests/test_gpu_tally_edges.py."""
import gzip
import json
import os

import numpy as np
import pytest

from conftest import GOLD, parse_pir

pytestmark = pytest.mark.gpu
INT_FIELDS = ["TP", "FP", "FN", "cor", "uncor", "uncorCor", "uncorUncor", "insC", "delC", "subsC", "insU", "delU",
              "subsU", "lenRef", "lenCor", "lenUnc", "gapsLeft", "gapsRight", "missing", "extended", "ncols", "assessed"]


@pytest.fixture(scope="module")
def ctx():
    import elector_b200
    c = elector_b200.PoaContext(device=0)
    yield c
    c.close()


def load(name):
    return json.loads(gzip.open(os.path.join(GOLD, name)).read())


def check(fields, got_row, exp):
    got = dict(zip(fields, (int(v) for v in got_row)))
    if not exp["assessed"]:
        assert got["assessed"] == 0 and got["ncols"] == exp["ncols"]
        return
    for k in INT_FIELDS:
        assert got[k] == exp[k], (k, got[k], exp[k])
    assert round(got["GCref"] * 1.0 / got["lenRef"], 3) == exp["GCrateRef"]
    assert round(got["GCcor"] * 1.0 / got["lenCor"], 3) == exp["GCrateCor"]


def test_tally_equals_computestats_on_example_reads(ctx):
    from elector_b200 import TALLY_FIELDS
    ex = load("tally_example.json.gz")
    out = ctx.tally([e["R"] for e in ex], [e["C"] for e in ex], [e["U"] for e in ex])
    for e, row in zip(ex, out):
        check(TALLY_FIELDS, row, e["expect"])


def test_tally_equals_computestats_on_random_rows(ctx):
    from elector_b200 import TALLY_FIELDS
    from oracle import synth
    exp = load("tally_random.json.gz")
    rows = synth.random_msa_rows(3000, 21)
    out = ctx.tally([r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows])
    for e, row in zip(exp, out):
        check(TALLY_FIELDS, row, e)


def test_tally_vs_oracle_fresh_seed(ctx):
    from elector_b200 import TALLY_FIELDS
    from oracle import synth, tally_oracle as to
    rows = synth.random_msa_rows(4000, 777)
    out = ctx.tally([r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows])
    for (R, C, U), row in zip(rows, out):
        exp = to.tally_read(R, C, U)
        assert [int(v) for v in row] == [exp[k] for k in TALLY_FIELDS]


def test_merge_equals_donatello(ctx, golden_dir):
    """poa windows of 6 example reads -> merged rows identical to the reference Donatello's msa file"""
    from elector_b200 import windows_to_csr
    from conftest import read_fasta_simple
    recs = parse_pir(golden_dir + "/donatello.pir")
    exp = open(golden_dir + "/donatello.msa").read().split("\n")
    # rebuild the window inputs from the PIR rows themselves (a row without '.' is the sequence)
    refs = [r[1][0].replace(".", "") for r in recs]; cors = [r[1][1].replace(".", "") for r in recs]; uncs = [r[1][2].replace(".", "") for r in recs]
    res = ctx.run(refs, cors, uncs)
    for w, r in enumerate(recs):
        assert res.window_rows(w) == r[1]
    heads = [r[0][2] for r in recs]
    first = [0] + [i for i in range(1, len(heads)) if heads[i] != heads[i - 1]] + [len(heads)]
    merged = ctx.merge(res, first)
    got = []
    for k, (a, b, c) in enumerate(merged):
        h = heads[first[k]]
        h = h[:len(h) - 11] + " "
        got += [h, a, h, b, h, c]
    assert got == exp[:-1]


def test_device_chain_poa_merge_tally_vs_oracle():
    """elector_poa_run_device -> elector_merge_tally_device (everything resident on the device)
    equals oracle POA -> oracle merge -> oracle tally on a config-1 slice with N windows"""
    import torch
    import elector_b200
    import workloads
    from elector_b200 import TALLY_FIELDS
    from oracle import oracle, tally_oracle as to
    wl = workloads.make_windows(2, 40)          # config 2: trimmed / split reads, `N` windows
    n, n_reads = len(wl["ref_off"]) - 1, len(wl["read_first"]) - 1
    dev = torch.device("cuda", 0)
    with elector_b200.PoaContext(0) as c:
        lib = c._lib
        h = {k: np.ascontiguousarray(wl[k]) for k in ("ref", "ref_off", "cor", "cor_off", "unc", "unc_off", "read_first")}
        d = {k: torch.from_numpy(h[k]).to(dev) for k in ("ref", "ref_off", "cor", "cor_off", "unc", "unc_off")}
        bound = int(lib.elector_poa_rows_bound(n, h["ref_off"].ctypes.data, h["cor_off"].ctypes.data, h["unc_off"].ctypes.data))
        d_rows = torch.empty(bound, dtype=torch.uint8, device=dev)
        d_rowoff = torch.empty(n, dtype=torch.int64, device=dev)
        d_stride = torch.empty(n, dtype=torch.int32, device=dev)
        d_nring = torch.empty(n, dtype=torch.int32, device=dev)
        d_used = torch.zeros(1, dtype=torch.int64, device=dev)
        d_cnt = torch.zeros(n_reads * len(TALLY_FIELDS), dtype=torch.int64, device=dev)
        c._check(lib.elector_poa_run_device(c._ctx, n, d["ref"].data_ptr(), d["ref_off"].data_ptr(), d["cor"].data_ptr(), d["cor_off"].data_ptr(),
                                            d["unc"].data_ptr(), d["unc_off"].data_ptr(), h["ref_off"].ctypes.data, h["cor_off"].ctypes.data,
                                            h["unc_off"].ctypes.data, d_rows.data_ptr(), bound, d_rowoff.data_ptr(), d_stride.data_ptr(),
                                            d_nring.data_ptr(), None, None, None, d_used.data_ptr()))
        c._check(lib.elector_merge_tally_device(c._ctx, n_reads, h["read_first"].ctypes.data, n, d_rows.data_ptr(), int(d_used.item()),
                                                d_rowoff.data_ptr(), d_stride.data_ptr(), d_nring.data_ptr(), d_cnt.data_ptr()))
        got = d_cnt.cpu().numpy().reshape(n_reads, -1)
    o = oracle.batch(h["ref"], h["ref_off"], h["cor"], h["cor_off"], h["unc"], h["unc_off"], nthreads=os.cpu_count() or 1)
    rf = h["read_first"]
    for r in range(n_reads):
        rows = [oracle.window_rows(o, w) for w in range(rf[r], rf[r + 1])]
        R = "".join(x[0] for x in rows); C = "".join(x[1] for x in rows); U = "".join(x[2] for x in rows)
        keep = [i for i, ch in enumerate(C) if ch != "n"]
        R, C, U = ("".join(s[i] for i in keep) for s in (R, C, U))
        exp = to.tally_read(R, C, U)
        assert [int(v) for v in got[r]] == [exp[k] for k in TALLY_FIELDS], r


@pytest.mark.parametrize("chunks,workers", [("1", "1"), ("4", "3"), ("7", "2")])
def test_pipeline_call_equals_oracle_chain(chunks, workers, monkeypatch):
    """elector_pipeline_run (host buffers; one chunk, or several chunks on several worker contexts, copies overlapped,
    rows in two regions per chunk) equals oracle POA -> oracle merge -> oracle tally read by read; the sums equal the
    column sums"""
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", chunks)
    monkeypatch.setenv("ELECTOR_PIPELINE_WORKERS", workers)
    import elector_b200
    import workloads
    from elector_b200 import TALLY_FIELDS
    from oracle import oracle, tally_oracle as to
    wl = workloads.make_windows(2, 900)            # ~250k windows; trimmed / split reads
    with elector_b200.PoaContext(0) as c:
        res, counters, sums = c.pipeline_csr(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"], wl["read_first"])
        res2 = c.run_csr(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"])
    n, rf = len(wl["ref_off"]) - 1, wl["read_first"]
    assert np.array_equal(res.nring, res2.nring) and np.array_equal(res.score1, res2.score1) and np.array_equal(res.score2, res2.score2)
    ext = TALLY_FIELDS.index("extended")
    exp_sums = counters.sum(axis=0)
    exp_sums[ext] = counters[:, ext][counters[:, ext] >= 0].sum()
    assert np.array_equal(sums, exp_sums)
    k_reads = 60
    k = int(rf[k_reads])
    o = oracle.batch(wl["ref"], wl["ref_off"][:k + 1], wl["cor"], wl["cor_off"][:k + 1], wl["unc"], wl["unc_off"][:k + 1], nthreads=os.cpu_count() or 1)
    for r in list(range(k_reads)):
        rows = [oracle.window_rows(o, w) for w in range(rf[r], rf[r + 1])]
        for w in range(rf[r], rf[r + 1]):
            assert res.window_rows(w) == rows[w - rf[r]]
        R = "".join(x[0] for x in rows); C = "".join(x[1] for x in rows); U = "".join(x[2] for x in rows)
        keep = [i for i, ch in enumerate(C) if ch != "n"]
        R, C, U = ("".join(s[i] for i in keep) for s in (R, C, U))
        exp = to.tally_read(R, C, U)
        assert [int(v) for v in counters[r]] == [exp[f] for f in TALLY_FIELDS], r
    # the last read of the call (last chunk) against the oracle as well
    r = len(rf) - 2
    w0, w1 = int(rf[r]), int(rf[r + 1])
    sub = workloads.slice_windows(wl, r, r + 1)
    o = oracle.batch(sub["ref"], sub["ref_off"], sub["cor"], sub["cor_off"], sub["unc"], sub["unc_off"], nthreads=1)
    for w in range(w0, w1):
        assert res.window_rows(w) == oracle.window_rows(o, w - w0)


@pytest.mark.parametrize("cfg,reads", [(1, 60), (3, 10), (4, 240)])
def test_config_slices_pipeline_equals_oracle_chain(cfg, reads):
    """slices of BASELINE.json configs 1, 3 (50-100 kb reads: ~1 400 windows per read) and 4 (1-30 kb reads, log-uniform)
    through elector_pipeline_run: every window's rows and scores and every read's counters equal the oracle chain"""
    import elector_b200
    import workloads
    from elector_b200 import TALLY_FIELDS
    from oracle import oracle, tally_oracle as to
    wl = workloads.make_windows(cfg, reads)
    with elector_b200.PoaContext(0) as c:
        res, counters, sums = c.pipeline_csr(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"], wl["read_first"])
    o = oracle.batch(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"], nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"]) and np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    assert np.array_equal(res.cells, o["cells"])
    rf = wl["read_first"]
    for r in range(len(rf) - 1):
        rows = [oracle.window_rows(o, w) for w in range(rf[r], rf[r + 1])]
        for w in range(rf[r], rf[r + 1]):
            assert res.window_rows(w) == rows[w - rf[r]], (cfg, w)
        R = "".join(x[0] for x in rows); C = "".join(x[1] for x in rows); U = "".join(x[2] for x in rows)
        keep = [i for i, ch in enumerate(C) if ch != "n"]
        R, C, U = ("".join(s[i] for i in keep) for s in (R, C, U))
        exp = to.tally_read(R, C, U)
        assert [int(v) for v in counters[r]] == [exp[f] for f in TALLY_FIELDS], (cfg, r)


@pytest.mark.parametrize("packed,merged,chunks", [(True, "bytes", "1"), (True, "nibbles", "3"), (False, "nibbles", "2"), (True, "columns", "3"), (False, "columns", "1"), (True, None, "1")])
def test_compact_wire_format_equals_byte_path(packed, merged, chunks, monkeypatch):
    """elector_pipeline_run2: 2-bit letters + exceptions and 32-bit offsets in, merged rows as bytes or 4-bit columns (with
    escapes) or counters only out -- same windows, merged rows (= Donatello of the window rows) and counters as the byte
    path, on a config-2 slice (`N` placeholder windows: exceptions on the way in; out-of-code letters forced in: escapes)"""
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", chunks)
    import elector_b200
    import workloads
    wl = workloads.make_windows(2, 300)
    ref, cor, unc = wl["ref"].copy(), wl["cor"].copy(), wl["unc"].copy()
    # a few letters outside ACGT (IUPAC, lower case, 'u') and outside the 4-bit column code
    rng = np.random.default_rng(5)
    for arr, letters in ((ref, b"RYn"), (cor, b"acgtNu"), (unc, b"K?]")):
        idx = rng.integers(0, len(arr), 40)
        arr[idx] = np.frombuffer(letters, np.uint8)[rng.integers(0, len(letters), 40)]
    with elector_b200.PoaContext(0) as c:
        base_res, base_cnt, base_sums = c.pipeline_csr(ref, wl["ref_off"], cor, wl["cor_off"], unc, wl["unc_off"], wl["read_first"])
        base_merged = c.merge(base_res, wl["read_first"])
        out = c.pipeline_io(ref, wl["ref_off"], cor, wl["cor_off"], unc, wl["unc_off"], wl["read_first"], packed=packed, window_rows=False, merged=merged, lengths32=(chunks != "1"), lengths16=(merged == "columns"))
    assert np.array_equal(out["res"].nring, base_res.nring) and np.array_equal(out["res"].score2, base_res.score2)
    assert np.array_equal(out["counters"], base_cnt) and np.array_equal(out["sums"], base_sums)
    if merged:
        assert out["merged"] == base_merged
        if merged in ("nibbles", "columns"):
            assert out["n_esc"] > 0


@pytest.mark.gpu
def test_merge_copy_on_synthetic_rows(ctx):
    """merge_copy_kernel's paths on hand-made window rows (Donatello.cpp:50-84: concatenate a read's windows, drop the columns
    whose corrected row is 'n'): every destination alignment, windows of 1 .. 300 columns (the word path takes up to 124, the
    byte path the rest), windows with dropped columns, windows that are all 'n', reads of one window"""
    from elector_b200.poa import PoaResult
    rng = np.random.default_rng(17)
    n_win = 5000
    k = rng.integers(1, 70, n_win)
    k[rng.integers(0, n_win, 200)] = rng.integers(120, 301, 200)      # around and beyond the word path's limit
    k[rng.integers(0, n_win, 300)] = rng.integers(1, 5, 300)          # shorter than one word
    stride = (k + 3) & ~3
    off = np.concatenate([[0], np.cumsum(3 * stride)]).astype(np.int64)
    perm = rng.permutation(n_win)                                        # rows lie in the buffer in another order than the windows
    row_off = np.empty(n_win, np.int64)
    row_off[perm] = np.concatenate([[0], np.cumsum(3 * stride[perm])])[:-1]
    rows = np.zeros(int(off[-1]), np.uint8)
    letters = np.frombuffer(b".acgt", np.uint8)
    wins = []
    for w in range(n_win):
        r = [letters[rng.integers(0, 5, k[w])] for _ in range(3)]
        mode = rng.integers(0, 10)
        if mode == 0:
            r[1][:] = ord("n")                                          # a placeholder window: every column dropped
        elif mode == 1:
            r[1][rng.integers(0, k[w], max(1, k[w] // 5))] = ord("n")   # some columns dropped
        for s in range(3):
            rows[row_off[w] + s * stride[w]:row_off[w] + s * stride[w] + k[w]] = r[s]
        wins.append(r)
    cuts = np.unique(np.concatenate([[0, n_win], rng.integers(1, n_win, 400), np.arange(10, 40)]))
    res = PoaResult(rows, row_off, stride.astype(np.int32), k.astype(np.int32), np.zeros(n_win, np.int32), np.zeros(n_win, np.int32), np.zeros(n_win, np.int64))
    got = ctx.merge(res, cuts)
    for i in range(len(cuts) - 1):
        cat = [np.concatenate([wins[w][s] for w in range(cuts[i], cuts[i + 1])]) for s in range(3)]
        keep = cat[1] != ord("n")
        exp = tuple(c[keep].tobytes().decode("latin-1") for c in cat)
        assert got[i] == exp, i
