"""GPU: the window cutting on the device (SURVEY.md 8f-1):
  - the `masterSplitter` drop-in (elector_b200/bin/masterSplitter, alignment.py:99's command line) on the README example against
    the UNMODIFIED masterSplitter: md5 of every shard file == tests/golden/example_full.json.gz;
  - the same executable on synthetic reads of configs 1-4, several rounds through progress.txt, against the compiled reference
    (oracle/_ref/masterSplitter, only where oracle/build_ref.sh has built it) and against the serial CPU build of the project's
    own cutting code (tests/emul/split_emul: the same source, run one job after the other, so that check holds the parallel
    device run to the serial one, not to the reference);
  - elector_reads_run (reads in, windows never leave the device) == splitter -> elector_pipeline_run on the same reads, with
    the same two splitters."""
import os
import subprocess

import numpy as np
import pytest

from conftest import load_example_golden, md5_file
from test_split_emul import REF_SPLITTER, compare_dirs, run_splitter

pytestmark = pytest.mark.gpu


def drop_in():
    from elector_b200.lib import splitter_binary_path
    exe = splitter_binary_path()
    assert os.path.exists(exe), "elector_b200/bin/masterSplitter not built (__graft_entry__.build())"
    return exe


def test_dropin_cuts_the_example_like_the_reference(tmp_path):
    from oracle import example_prep as ep
    src, work, out = str(tmp_path / "src"), str(tmp_path / "work"), str(tmp_path / "out")
    os.makedirs(src); os.makedirs(work)
    ep.unpack(src)
    ep.sort_and_duplicate(src, work)
    rc = run_splitter(drop_in(), [work + "/ref.fa", work + "/unc.fa", work + "/cor.fa"], out)
    g = load_example_golden()
    assert rc == 0
    for i in range(200):
        if str(i) in g["splitter"]:
            for q in (1, 2, 3):
                assert md5_file("%s/out%d%d" % (out, q, i)) == g["splitter"][str(i)]["out%d" % q], (q, i)
        else:
            assert os.path.getsize("%s/out3%d" % (out, i)) == 0
    assert int(open(out + "/small_reads.txt").read()) == g["small_reads"]
    assert int(open(out + "/wrongly_cor_reads.txt").read()) == g["wrongly_cor_reads"]


SYNTHETIC_CUTS = [(1, 400, 10000, "0.1"), (2, 600, 10000, "0.1"), (3, 24, 10000, "0.1"), (4, 1500, 10000, "0.1"),
                  (2, 300, 110, "0.4"), (4, 400, 150, "0.9")]


def dropin_cuts_like(exe, tmp_path, cfg, reads, amount, thr):
    import workloads
    pre = str(tmp_path / "r")
    subprocess.check_call([workloads.ensure_gen(), str(cfg), str(reads), "0", pre])
    files = [pre + ".ref.fa", pre + ".unc.fa", pre + ".cor.fa"]
    a, b = str(tmp_path / "cpu"), str(tmp_path / "gpu")
    for rnd in range(8):
        ra = run_splitter(exe, files, a, amount, thr)
        rb = run_splitter(drop_in(), files, b, amount, thr)
        assert ra == rb, rnd
        compare_dirs(a, b)
        if ra == 0:
            break
    else:
        raise AssertionError("more rounds than expected")


@pytest.mark.skipif(not os.path.exists(REF_SPLITTER), reason="oracle/_ref/masterSplitter not built")
@pytest.mark.parametrize("cfg,reads,amount,thr", SYNTHETIC_CUTS)
def test_dropin_equals_compiled_reference_on_synthetic_reads(tmp_path, cfg, reads, amount, thr):
    dropin_cuts_like(REF_SPLITTER, tmp_path, cfg, reads, amount, thr)


@pytest.mark.parametrize("cfg,reads,amount,thr", SYNTHETIC_CUTS)
def test_dropin_equals_serial_cpu_cutting_on_synthetic_reads(tmp_path, split_emul_bin, cfg, reads, amount, thr):
    dropin_cuts_like(split_emul_bin, tmp_path, cfg, reads, amount, thr)


@pytest.mark.skipif(not os.path.exists(REF_SPLITTER), reason="oracle/_ref/masterSplitter not built")
@pytest.mark.parametrize("cfg,reads", [(1, 300), (2, 400)])
def test_reads_run_equals_reference_splitter_then_pipeline(tmp_path, cfg, reads):
    reads_run_equals_splitter_then_pipeline(REF_SPLITTER, tmp_path, cfg, reads)


@pytest.mark.parametrize("cfg,reads", [(1, 300), (2, 400)])
def test_reads_run_equals_serial_cpu_cutting_then_pipeline(tmp_path, split_emul_bin, cfg, reads):
    reads_run_equals_splitter_then_pipeline(split_emul_bin, tmp_path, cfg, reads)


def reads_run_equals_splitter_then_pipeline(exe, tmp_path, cfg, reads):
    """the chained call: per-triplet counters, merged rows and window counts equal what the splitter's windows give
    through elector_pipeline_run (itself held to the reference poa / Donatello / computeStats by the other GPU tests)"""
    import elector_b200
    import workloads
    pre = str(tmp_path / "r")
    subprocess.check_call([workloads.ensure_gen(), str(cfg), str(reads), "0", pre])
    hr, ref, ro = workloads.parse_two_line_fasta(pre + ".ref.fa")
    _, unc, uo = workloads.parse_two_line_fasta(pre + ".unc.fa")
    _, cor, co = workloads.parse_two_line_fasta(pre + ".cor.fa")
    n = len(hr)
    out = str(tmp_path / "cut")
    assert run_splitter(exe, [pre + ".ref.fa", pre + ".unc.fa", pre + ".cor.fa"], out, 10000, "0.1") == 0
    heads, parts = [], {q: ([], [np.zeros(1, np.int64)], 0) for q in (1, 2, 3)}
    for i in range(200):
        if os.path.getsize("%s/out3%d" % (out, i)) == 0:
            continue
        for q in (1, 2, 3):
            h, s, o = workloads.parse_two_line_fasta("%s/out%d%d" % (out, q, i))
            segs, offs, tot = parts[q]
            segs.append(s); offs.append(o[1:] + tot)
            parts[q] = (segs, offs, tot + int(o[-1]))
            if q == 1:
                heads += h
    w = {q: (np.concatenate(parts[q][0]), np.concatenate(parts[q][1])) for q in (1, 2, 3)}
    first = [0] + [k for k in range(1, len(heads)) if heads[k] != heads[k - 1]] + [len(heads)]
    assert len(first) == n + 1
    with elector_b200.PoaContext(0) as ctx:
        got = ctx.reads_run(ref, ro, unc, uo, cor, co, [len(h) for h in hr], 0.1, merged=True)
        res, counters, sums = ctx.pipeline_csr(w[1][0], w[1][1], w[3][0], w[3][1], w[2][0], w[2][1], first)
        merged = ctx.merge(res, first)
    assert got["n_windows"] == len(heads)
    assert np.array_equal(got["read_first"], np.asarray(first))
    assert np.array_equal(got["counters"], counters)
    assert np.array_equal(got["sums"], sums)
    for t in range(n):
        o, l = int(got["m_off"][t]), int(got["m_len"][t])
        rows = tuple(got[k][o:o + l].tobytes().decode() for k in ("m_ref", "m_cor", "m_unc"))
        assert rows == tuple(merged[t]), t
