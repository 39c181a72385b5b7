"""CPU: the window-cutting DEVICE code (elector_b200/csrc/split_kernel.cuh, host/device dual) run serially by
tests/emul/split_emul.cu with the reference's own file handling around it, against
  - the md5 of every shard file the UNMODIFIED masterSplitter wrote for the README example (tests/golden/example_full.json.gz), and
  - the compiled reference itself (oracle/_ref/masterSplitter) on synthetic reads of configs 1-4 (trimmed / split corrected
    reads of config 2 take the late-start / early-end branches, Master_Splitter.cpp:268-277,295-301)."""
import os
import subprocess

import pytest

from conftest import ROOT, load_example_golden, md5_file

REF_SPLITTER = os.path.join(ROOT, "oracle", "_ref", "masterSplitter")


def run_splitter(exe, files, out, amount=10000, threshold="0.1", nfiles=200):
    os.makedirs(out, exist_ok=True)
    return subprocess.call([exe] + list(files) + [out + "/out1", out + "/out2", out + "/out3", "7", str(nfiles), str(amount), str(threshold), out],
                           stdout=subprocess.DEVNULL)


def compare_dirs(a, b, nfiles=200):
    for i in range(nfiles):
        for q in (1, 2, 3):
            fa, fb = "%s/out%d%d" % (a, q, i), "%s/out%d%d" % (b, q, i)
            assert open(fa, "rb").read() == open(fb, "rb").read(), (q, i)
    for f in ("small_reads.txt", "wrongly_cor_reads.txt"):
        assert open(os.path.join(a, f)).read() == open(os.path.join(b, f)).read(), f
    pa, pb = os.path.join(a, "progress.txt"), os.path.join(b, "progress.txt")
    assert os.path.exists(pa) == os.path.exists(pb)
    if os.path.exists(pa):
        assert open(pa).read() == open(pb).read()


def test_emulated_cutting_of_the_example_equals_reference_md5(split_emul_bin, tmp_path):
    from oracle import example_prep as ep
    src, work, out = str(tmp_path / "src"), str(tmp_path / "work"), str(tmp_path / "out")
    os.makedirs(src); os.makedirs(work)
    ep.unpack(src)
    ep.sort_and_duplicate(src, work)
    rc = run_splitter(split_emul_bin, [work + "/ref.fa", work + "/unc.fa", work + "/cor.fa"], out)
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


@pytest.mark.parametrize("mode", ["SPLIT_EMUL_TIGHT", "SPLIT_EMUL_PACKED"])
def test_emulated_cutting_with_the_fullest_table_and_with_packed_letters(split_emul_bin, tmp_path, mode, monkeypatch):
    """the two shapes the kernel runs in that the default emulation does not: the smallest table it accepts, and reads taken from the
    letters packed once per call (split_prepack_kernel) -- config 2 has N placeholders, trimmed and split reads (sub-strings at odd offsets);
    held to the compiled reference where oracle/build_ref.sh has built it, else to the default emulation (other table size, letters
    read unpacked)"""
    import workloads
    pre = str(tmp_path / "r")
    subprocess.check_call([workloads.ensure_gen(), "2", "120", "0", pre])
    files = [pre + ".ref.fa", pre + ".unc.fa", pre + ".cor.fa"]
    a, b = str(tmp_path / "ref"), str(tmp_path / "emu")
    assert run_splitter(REF_SPLITTER if os.path.exists(REF_SPLITTER) else split_emul_bin, files, a) == 0
    monkeypatch.setenv(mode, "1")
    assert run_splitter(split_emul_bin, files, b) == 0
    compare_dirs(a, b)


@pytest.mark.skipif(not os.path.exists(REF_SPLITTER), reason="oracle/_ref/masterSplitter not built")
@pytest.mark.parametrize("cfg,reads,amount,thr", [(1, 60, 10000, "0.1"), (2, 150, 10000, "0.1"), (3, 6, 10000, "0.1"), (4, 200, 10000, "0.1"),
                                                  (2, 150, 60, "0.4"), (4, 120, 50, "0.9")])
def test_emulated_cutting_equals_compiled_reference_on_synthetic_reads(split_emul_bin, tmp_path, cfg, reads, amount, thr):
    """amount < reads: several rounds through progress.txt with the reference's exit code 1 (alignment.py:98-100 loops on it)"""
    import workloads
    pre = str(tmp_path / "r")
    subprocess.check_call([workloads.ensure_gen(), str(cfg), str(reads), "0", pre])
    files = [pre + ".ref.fa", pre + ".unc.fa", pre + ".cor.fa"]
    a, b = str(tmp_path / "ref"), str(tmp_path / "emu")
    for rnd in range(6):
        ra = run_splitter(REF_SPLITTER, files, a, amount, thr)
        rb = run_splitter(split_emul_bin, files, b, amount, thr)
        assert ra == rb, rnd
        compare_dirs(a, b)
        if ra == 0:
            break
    else:
        raise AssertionError("more rounds than expected")
