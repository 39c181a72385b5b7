"""CPU: the oracle (oracle/poa_oracle.c) against outputs of the compiled reference."""
import hashlib
import os
import subprocess

import pytest

from conftest import GOLDEN_SETS, ROOT


@pytest.mark.parametrize("name", GOLDEN_SETS)
def test_oracle_pir_equals_reference(golden_dir, name, tmp_path):
    from oracle import oracle
    d = golden_dir
    out = str(tmp_path / "o.pir")
    rc = oracle.poa_files(d + "/blosum80.mat", "%s/%s.ref.fa" % (d, name), "%s/%s.cor.fa" % (d, name),
                          "%s/%s.unc.fa" % (d, name), out)
    assert rc == 0
    assert open(out, "rb").read() == open("%s/%s.pir" % (d, name), "rb").read()


@pytest.mark.parametrize("name", GOLDEN_SETS)
def test_oracle_scores_and_maps_equal_reference(golden_dir, name, tmp_path):
    """both align_lpo_po scores and the four x_to_y / y_to_x maps (align_lpo_po2.c:486,158-165)"""
    from oracle import oracle
    d = golden_dir
    out = str(tmp_path / "o.dump")
    assert oracle.dump_files(d + "/blosum80.mat", "%s/%s.ref.fa" % (d, name), "%s/%s.cor.fa" % (d, name),
                             "%s/%s.unc.fa" % (d, name), out) == 0
    assert open(out).read() == open("%s/%s.dump" % (d, name)).read()


def test_oracle_batch_matches_file_driver(golden_dir):
    from conftest import parse_pir, read_fasta_simple
    from elector_b200 import windows_to_csr
    from oracle import oracle
    d = golden_dir
    refs = [s for _, s in read_fasta_simple(d + "/hard.ref.fa")]
    cors = [s for _, s in read_fasta_simple(d + "/hard.cor.fa")]
    uncs = [s for _, s in read_fasta_simple(d + "/hard.unc.fa")]
    r, ro = windows_to_csr(refs); c, co = windows_to_csr(cors); u, uo = windows_to_csr(uncs)
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=4)
    gold = parse_pir(d + "/hard.pir")
    for w in range(len(refs)):
        assert oracle.window_rows(o, w) == gold[w][1]


def test_oracle_cli_flags(golden_dir, tmp_path):
    """oracle CLI has the reference's five flags and ignores the others (main.c:85-113)"""
    from oracle import oracle
    oracle.build()
    d = golden_dir
    out = str(tmp_path / "cli.pir")
    rc = subprocess.call([os.path.join(ROOT, "oracle", "poa_oracle_cli"), "-pir", out, "-preserve_seqorder",
                          "-corrected_reads_fasta", d + "/edge.cor.fa", "-reference_reads_fasta", d + "/edge.ref.fa",
                          "-uncorrected_reads_fasta", d + "/edge.unc.fa", "-preserve_seqorder", "-threads", "1",
                          "-pathMatrix", d + "/blosum80.mat"], stdout=subprocess.DEVNULL)
    assert rc == 0
    assert open(out, "rb").read() == open(d + "/edge.pir", "rb").read()


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "poa")), reason="compiled reference not present")
def test_live_reference_agrees_with_golden_and_generated_matrix(golden_dir, tmp_path):
    """when oracle/_ref/poa exists: it reproduces the committed golden with OUR generated matrix file"""
    d = golden_dir
    out = str(tmp_path / "ref.pir")
    rc = subprocess.call([os.path.join(ROOT, "oracle", "_ref", "poa"), "-pir", out, "-corrected_reads_fasta", d + "/hard.cor.fa",
                          "-reference_reads_fasta", d + "/hard.ref.fa", "-uncorrected_reads_fasta", d + "/hard.unc.fa",
                          "-pathMatrix", d + "/blosum80.mat"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert rc == 0
    assert hashlib.md5(open(out, "rb").read()).hexdigest() == hashlib.md5(open(d + "/hard.pir", "rb").read()).hexdigest()


def test_oracle_long_windows_equal_reference(golden_dir, tmp_path):
    """golden set `long` (oracle/make_golden_long.py): a 3 300-letter window, a 33 500-letter window on one FASTA line
    longer than the reference's 32 KiB line buffer (fasta_format.c:20), wrapped lines with blanks, a window after them"""
    from conftest import parse_dump
    from oracle import oracle
    d = golden_dir
    out, dump = str(tmp_path / "o.pir"), str(tmp_path / "o.dump")
    assert oracle.poa_files(d + "/blosum80.mat", d + "/long.ref.fa", d + "/long.cor.fa", d + "/long.unc.fa", out) == 0
    assert open(out, "rb").read() == open(d + "/long.pir", "rb").read()


def test_edge_windows_sit_on_their_edges():
    """oracle/synth.edge_windows: every window has the lengths, len(P1) (from the oracle: (cells - lr lc) / lu) and cor-is-ref
    its tag states, and every edge the scheduler tests need is present -- the set cannot drift off its edges unnoticed"""
    import numpy as np
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    k = synth.kernel_constants()
    S, Q4, NMAX = k["kSmallMax"], 4 * k["kN1q"], k["kMaxNodes"]
    wins = synth.edge_windows()
    assert wins[-1][0] == "toolarge sum=%d" % (NMAX + 1) and len(wins[-1][1]) + len(wins[-1][2]) == NMAX + 1
    wins = wins[:-1]
    r, ro = windows_to_csr([w[1] for w in wins]); c, co = windows_to_csr([w[2] for w in wins]); u, uo = windows_to_csr([w[3] for w in wins])
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=os.cpu_count() or 1)
    n1 = (o["cells"] - np.diff(ro) * np.diff(co)) // np.diff(uo)
    for i, (tag, ref, cor, unc) in enumerate(wins):
        got = synth.window_measures(ref, cor, unc, int(n1[i]))
        for key, val in synth.parse_tag(tag)[1].items():
            assert got[key] == val, (tag, key, got[key])
    tags = {w[0] for w in wins}
    need = ["p1 lr=%d lc=%d" % (lr, lc) for lc in (1, 8, 9, 64, 65, 128, 129, S, S + 1) for lr in (50, S)]
    need += ["p1 lr=%d lc=%d" % (lr, lc) for lr in (1, 2, S - 1, S, S + 1) for lc in (50, 1)]
    need += ["p1big mx=%d %s=%d" % (mx, side, mx) for mx in (2 * S, 2 * S + 1, 4 * S, 4 * S + 1, 8 * S, 8 * S + 1) for side in ("lr", "lc")]
    need += ["p2 lu=%d" % lu for lu in (1, 8, 9, 32, 33, 64, 65, 128, 129, S, S + 1)]
    need += ["p2 lu=%d n1=500" % lu for lu in (1, 8, 9, 32, 33, 64, 65, 128, 129, S, S + 1)]
    need += ["p2q n1=%d lu=%d" % (n, lu) for n in (Q4 - 2, Q4 - 1, Q4, Q4 + 1) for lu in (8, 128, 129, S)]
    need += ["id lr=%d lu=%d id=1" % (lr, lu) for lr in (1, 8, 9, 128, 129, S - 1, S, S + 1) for lu in (1, 128, 129, S, S + 1)]
    need += ["idd lr=60 d=%d id=1" % d for d in (-40, -7, -6, -3, -2, 1, 2, 5, 6, 9, 10, 40)]
    B = synth.band_span_limit(10, k)
    need += ["band1 sum=%d" % s for s in (B, B + 1)] + ["band2 span2=%d id=1" % s for s in (B, B + 1)]
    need += ["asym lr=%d lc=1" % lr for lr in (S, S + 1, 3000)] + ["asym lr=1 lc=300", "asym lu=1 n1=500"]
    need += ["asym lr=%d lu=%d" % (lr, 4 * lr) for lr in (60, 100)]
    need += ["cap lr=%d lc=534 lu=64 sum=%d" % (NMAX - 534, NMAX), "cap lr=534 lc=%d lu=64 sum=%d" % (NMAX - 534, NMAX),
             "cap lr=50 lc=50 lu=%d" % k["kMaxWindowLen"]]
    assert not [t for t in need if t not in tags]
    # the ones whose point is the small tier: both sequences of the len(P1) windows below 4 kN1q fit it
    for i, (tag, ref, cor, unc) in enumerate(wins):
        if tag.startswith("p2q") and n1[i] < Q4:
            assert max(len(ref), len(cor)) <= S, tag
