"""GPU: the pipelined reads-in call (elector_reads_pipeline_run, PoaContext.reads_pipeline) gives what one elector_reads_run over
the same triplets gives -- status, k_used, window count, read_first, counters, sums, the stretches elector_last_stretches returns
after reads_run, every triplet's merged rows -- however the call is cut into chunks, workers and devices; its errors; and the
README example through alignment.getPOA on two listed devices."""
import contextlib
import ctypes
import io
import os
import subprocess

import numpy as np
import pytest

from conftest import md5_file

pytestmark = pytest.mark.gpu

CASES = [(1, 300), (2, 400), (4, 600)]   # config 2: split and trimmed reads, N windows
THRESHOLDS = [0.1, 0.4, 0.9]             # 0.4 and 0.9 give status 1 triplets
SETTINGS = [(c, w, d) for c in (1, 3, 17) for w in (1, 3) for d in ([0], [0, 0])]


@pytest.fixture(scope="module")
def ctx():
    import elector_b200
    with elector_b200.PoaContext(0) as c:
        yield c


_READS = {}


def reads(tmp_path_factory, cfg, n):
    """(ref, ro, unc, uo, cor, co, header lengths) of n generated triplets of config cfg"""
    if (cfg, n) not in _READS:
        import workloads
        pre = str(tmp_path_factory.mktemp("reads") / "r")
        subprocess.check_call([workloads.ensure_gen(), str(cfg), str(n), "0", pre])
        hr, ref, ro = workloads.parse_two_line_fasta(pre + ".ref.fa")
        _, unc, uo = workloads.parse_two_line_fasta(pre + ".unc.fa")
        _, cor, co = workloads.parse_two_line_fasta(pre + ".cor.fa")
        _READS[(cfg, n)] = (ref, ro, unc, uo, cor, co, np.asarray([len(h) for h in hr], np.int32))
    return _READS[(cfg, n)]


def reference(ctx, r, thr, merged=True):
    """one elector_reads_run over all triplets, with the stretches of its tally"""
    got = ctx.reads_run(*r, thr, merged=merged)
    got["stretches"] = ctx.last_stretches(len(r[-1]))
    return got


def merged_rows(got, t):
    o, l = int(got["m_off"][t]), int(got["m_len"][t])
    return tuple(got[k][o:o + l].tobytes() for k in ("m_ref", "m_cor", "m_unc"))


def assert_same(got, want, merged=True):
    for k in ("status", "k_used", "read_first", "counters", "sums", "stretches"):
        assert np.array_equal(got[k], want[k]), k
    assert got["n_windows"] == want["n_windows"]
    if merged:
        assert np.array_equal(got["m_len"], want["m_len"])
        for t in range(len(want["status"])):
            assert merged_rows(got, t) == merged_rows(want, t), t


@pytest.mark.parametrize("thr", THRESHOLDS)
@pytest.mark.parametrize("cfg,n", CASES)
def test_pipeline_equals_reads_run(ctx, tmp_path_factory, monkeypatch, cfg, n, thr):
    r = reads(tmp_path_factory, cfg, n)
    want = reference(ctx, r, thr)
    for chunks, workers, devices in SETTINGS:
        monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", str(chunks))
        monkeypatch.setenv("ELECTOR_PIPELINE_WORKERS", str(workers))
        got = ctx.reads_pipeline(*r, thr, merged=True, devices=devices)
        assert_same(got, want)
        assert (got["m_off"] % 16 == 0).all()


def test_status_1_occurs(ctx, tmp_path_factory):
    seen = set()
    for cfg, n in CASES:
        for thr in THRESHOLDS:
            seen |= set(reference(ctx, reads(tmp_path_factory, cfg, n), thr, merged=False)["status"].tolist())
    assert {0, 1} <= seen


def test_unrelated_corrected_reads(ctx, tmp_path_factory, monkeypatch):
    """corrected reads that share nothing with their reference are not cut (status 2, wrongly_cor_reads)"""
    ref, ro, unc, uo, cor, co, hl = reads(tmp_path_factory, 1, 300)
    cor = cor.copy()
    rng = np.random.default_rng(5)
    for t in range(0, len(hl), 9):
        cor[co[t]:co[t + 1]] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(co[t + 1] - co[t]))]
    r = (ref, ro, unc, uo, cor, co, hl)
    want = reference(ctx, r, 0.1)
    assert (want["status"] == 2).any()
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "17")
    monkeypatch.setenv("ELECTOR_PIPELINE_WORKERS", "3")
    assert_same(ctx.reads_pipeline(*r, 0.1, merged=True, devices=[0, 0]), want)


def test_all_visible_devices(ctx, tmp_path_factory, monkeypatch):
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("one visible device")
    r = reads(tmp_path_factory, 2, 400)
    want = reference(ctx, r, 0.1)
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "9")
    assert_same(ctx.reads_pipeline(*r, 0.1, merged=True, devices=list(range(n_dev))), want)
    monkeypatch.delenv("ELECTOR_PIPELINE_CHUNKS")
    assert_same(ctx.reads_pipeline(*r, 0.1, merged=True, devices=list(range(n_dev))), want)


def test_counters_only(ctx, tmp_path_factory, monkeypatch):
    r = reads(tmp_path_factory, 2, 400)
    want = reference(ctx, r, 0.4, merged=False)
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "5")
    got = ctx.reads_pipeline(*r, 0.4, merged=False, devices=[0, 0])
    assert_same(got, want, merged=False)


def test_lowercase_n_runs_and_iupac_codes(ctx, tmp_path_factory, monkeypatch):
    """bytes the cutting codes case-sensitively or not at all, placed in reads on both sides of chunk edges"""
    ref, ro, unc, uo, cor, co, hl = reads(tmp_path_factory, 1, 300)
    ref, unc, cor = ref.copy(), unc.copy(), cor.copy()
    rng = np.random.default_rng(11)
    iupac = np.frombuffer(b"RYKMSWBDHVN", np.uint8)
    for t in range(len(hl)):
        for let, off in ((ref, ro), (unc, uo), (cor, co)):
            a, b = int(off[t]), int(off[t + 1])
            if b - a < 200:
                continue
            s = int(rng.integers(a, b - 150))
            if t % 4 == 0:
                let[s:s + 120] |= 0x20                       # lowercase
            elif t % 4 == 1:
                let[s:s + int(rng.integers(1, 80))] = ord("N")
            elif t % 4 == 2:
                pos = rng.integers(a, b, 6)
                let[pos] = iupac[rng.integers(0, len(iupac), 6)]
    r = (ref, ro, unc, uo, cor, co, hl)
    want = reference(ctx, r, 0.1)
    for chunks in ("17", "4"):
        monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", chunks)
        assert_same(ctx.reads_pipeline(*r, 0.1, merged=True, devices=[0, 0]), want)


def raw_call(ctx, r, m_cap, sentinel=7):
    """elector_reads_pipeline_run with every output prefilled -> (rc, outputs)"""
    from elector_b200.poa import ReadsIoC
    ref, ro, unc, uo, cor, co, hl = r
    n = len(hl)
    out = dict(status=np.full(n, sentinel, np.int32), k_used=np.full(n, sentinel, np.int32), read_first=np.full(n + 1, sentinel, np.int64),
               n_windows=np.full(1, sentinel, np.int64), counters=np.full((n, 24), sentinel, np.int64), sums=np.full(24, sentinel, np.int64),
               stretches=np.full((n, 17), sentinel, np.int32), m_ref=np.full(max(m_cap, 1), sentinel, np.uint8),
               m_cor=np.full(max(m_cap, 1), sentinel, np.uint8), m_unc=np.full(max(m_cap, 1), sentinel, np.uint8),
               m_off=np.full(n, sentinel, np.int64), m_len=np.full(n, sentinel, np.int32))
    io = ReadsIoC()
    io.n_triplets = n
    io.ref, io.unc, io.cor, io.ref_off, io.unc_off, io.cor_off = (a.ctypes.data for a in (ref, unc, cor, ro, uo, co))
    io.header_len, io.threshold = hl.ctypes.data, 0.1
    for f, k in (("status", "status"), ("k_used", "k_used"), ("read_first", "read_first"), ("n_windows", "n_windows"), ("counters_out", "counters"),
                 ("sums_out", "sums"), ("stretches_out", "stretches"), ("m_ref", "m_ref"), ("m_cor", "m_cor"), ("m_unc", "m_unc"),
                 ("m_off", "m_off"), ("m_len", "m_len")):
        setattr(io, f, out[k].ctypes.data)
    io.m_cap = m_cap
    rc = ctx._lib.elector_reads_pipeline_run(ctx._ctx, ctypes.byref(io))
    return rc, out


def test_capacity_one_byte_short_writes_nothing(ctx, tmp_path_factory):
    from elector_b200.poa import reads_merged_bound
    r = reads(tmp_path_factory, 1, 300)
    bound = reads_merged_bound(r[1], r[3], r[5])
    rc, out = raw_call(ctx, r, bound - 1)
    assert rc == -7 and "capacity" in ctx._lib.elector_last_error(ctx._ctx).decode()
    for k, a in out.items():
        assert (a == 7).all(), k
    rc, out = raw_call(ctx, r, bound)
    assert rc == 0
    assert np.array_equal(out["counters"], reference(ctx, r, 0.1, merged=False)["counters"])


def test_null_inputs(ctx, tmp_path_factory):
    from elector_b200.poa import ReadsIoC
    lib = ctx._lib
    assert lib.elector_reads_pipeline_run(ctx._ctx, None) == -1
    r = reads(tmp_path_factory, 1, 300)
    io = ReadsIoC()
    io.n_triplets = len(r[-1])
    io.unc, io.cor, io.ref_off, io.unc_off, io.cor_off, io.header_len = (a.ctypes.data for a in (r[2], r[4], r[1], r[3], r[5], r[6]))
    assert lib.elector_reads_pipeline_run(ctx._ctx, ctypes.byref(io)) == -1          # ref NULL
    assert "null" in lib.elector_last_error(ctx._ctx).decode()
    io.ref = r[0].ctypes.data
    m = np.zeros(16, np.uint8)
    io.m_ref, io.m_cap = m.ctypes.data, 16
    assert lib.elector_reads_pipeline_run(ctx._ctx, ctypes.byref(io)) == -1          # merged rows without m_cor / m_unc / m_off / m_len
    io.m_ref, io.m_cap = None, 0
    io.n_devices = 2
    assert lib.elector_reads_pipeline_run(ctx._ctx, ctypes.byref(io)) == -1          # devices NULL with n_devices > 0
    assert lib.elector_reads_pipeline_run(None, ctypes.byref(io)) == -1


def test_device_that_does_not_exist(ctx, tmp_path_factory):
    import elector_b200
    r = reads(tmp_path_factory, 1, 300)
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.reads_pipeline(*r, 0.1, devices=[0, 4096])
    assert e.value.code == -1 and "device 4096" in str(e.value)
    want = reference(ctx, r, 0.1)          # the context still works
    assert_same(ctx.reads_pipeline(*r, 0.1, merged=True), want)


def test_failed_chunk_in_the_worker_pool(ctx, tmp_path_factory, monkeypatch):
    """a chunk that fails inside the worker pool of either pipelined call, while other workers run theirs, gives the call its own
    error; a clean call on the same context afterwards gives what it gave before the failure"""
    import elector_b200
    import workloads
    # elector_pipeline_run2: four chunks on three workers; the first window of the last read (last chunk) has no corrected letters
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "4")
    monkeypatch.setenv("ELECTOR_PIPELINE_WORKERS", "3")
    wl = workloads.make_windows(2, 900)
    clean = (wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"], wl["read_first"])
    w = int(wl["read_first"][-2])
    co = np.array(wl["cor_off"], dtype=np.int64)
    cor = np.concatenate([wl["cor"][:co[w]], wl["cor"][co[w + 1]:]])
    co[w + 1:] -= co[w + 1] - co[w]
    want = ctx.pipeline_io(*clean)
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.pipeline_io(wl["ref"], wl["ref_off"], cor, co, wl["unc"], wl["unc_off"], wl["read_first"])
    assert e.value.code == -1 and "empty sequence" in str(e.value)
    got = ctx.pipeline_io(*clean)
    for k in ("nring", "score1", "score2", "cells"):
        assert np.array_equal(getattr(got["res"], k), getattr(want["res"], k)), k
    assert np.array_equal(got["counters"], want["counters"]) and np.array_equal(got["sums"], want["sums"])
    assert got["merged"] == want["merged"]
    # elector_reads_pipeline_run: five chunks on two listed devices; the last triplet (last chunk) has an empty reference read
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "5")
    monkeypatch.delenv("ELECTOR_PIPELINE_WORKERS")
    r = reads(tmp_path_factory, 1, 300)
    ro = r[1].copy()
    ro[-1] = ro[-2]
    want = ctx.reads_pipeline(*r, 0.1, merged=True, devices=[0, 0])
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.reads_pipeline(r[0], ro, *r[2:], 0.1, merged=True, devices=[0, 0])
    assert e.value.code == -1 and "empty reference read" in str(e.value)
    assert_same(ctx.reads_pipeline(*r, 0.1, merged=True, devices=[0, 0]), want)


def test_no_triplets(ctx):
    z8, z64 = np.zeros(0, np.uint8), np.zeros(1, np.int64)
    got = ctx.reads_pipeline(z8, z64, z8, z64, z8, z64, np.zeros(0, np.int32), 0.1, merged=True, devices=[0, 0])
    assert got["n_windows"] == 0 and not got["sums"].any()
    rc, out = raw_call(ctx, (z8, z64, z8, z64, z8, z64, np.zeros(0, np.int32)), 0)
    assert rc == 0 and not out["sums"].any() and out["n_windows"][0] == 0


def test_readme_example_on_two_listed_devices(example_chain, tmp_path, monkeypatch):
    from elector_b200 import alignment, computeStats
    from test_report import check_against_golden
    monkeypatch.setenv("ELECTOR_DEVICES", "0,0")
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "4")
    g, work = example_chain["gold"], example_chain["work"]
    out = str(tmp_path / "out")
    os.makedirs(out)
    assert alignment.getPOA(work + "/cor.fa", work + "/ref.fa", work + "/unc.fa", 4, out, 0.1) == (g["small_reads"], g["wrongly_cor_reads"])
    assert md5_file(out + "/msa.fa") == g["msa_md5"]
    log, buf = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(buf):
        ret = computeStats.outputRecallPrecision(work + "/cor.fa", out, log, g["small_reads"], g["wrongly_cor_reads"], 5, 0.1, "read_size_distribution.txt", {},
                                                 0, 0, None, compensated_sum=True)
    check_against_golden({"log": log.getvalue(), "stdout": buf.getvalue(), "assessed_reads": ret[0], "trimmed_or_split": ret[17], "extended_reads": int(ret[12]),
                          "size_distribution_complete": 1}, out, g)
    assert ret[:6] == (459, 4454164, 0.9938972, 0.995006, 0.9938413, 1 - 0.9938413)
    assert ret[15] == [159839, 160207, 154842] and ret[16] == [8119, 8161, 12148] and ret[18] == 0.9925
