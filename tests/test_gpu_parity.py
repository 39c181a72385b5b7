"""GPU: the CUDA path through the C-ABI against the reference goldens and the oracle."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_SETS, ROOT, parse_dump, parse_pir, read_fasta_simple

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(golden_dir):
    import elector_b200
    c = elector_b200.PoaContext(device=0, matrix_path=golden_dir + "/blosum80.mat")
    yield c
    c.close()


def csr_of(d, name):
    from elector_b200 import windows_to_csr
    return [windows_to_csr([s for _, s in read_fasta_simple("%s/%s.%s.fa" % (d, name, k))]) for k in ("ref", "cor", "unc")]


@pytest.mark.parametrize("name", GOLDEN_SETS)
def test_files_api_pir_is_byte_identical_to_reference(ctx, golden_dir, name, tmp_path):
    d = golden_dir
    out = str(tmp_path / "o.pir")
    ctx.files("%s/%s.ref.fa" % (d, name), "%s/%s.cor.fa" % (d, name), "%s/%s.unc.fa" % (d, name), out)
    assert open(out, "rb").read() == open("%s/%s.pir" % (d, name), "rb").read()


@pytest.mark.parametrize("name", GOLDEN_SETS)
def test_scores_rows_and_cells_equal_reference(ctx, golden_dir, name):
    """best_score of both align_lpo_po calls, len(P1), every MSA row"""
    d = golden_dir
    (r, ro), (c, co), (u, uo) = csr_of(d, name)
    res = ctx.run_csr(r, ro, c, co, u, uo)
    gold, pir = parse_dump("%s/%s.dump" % (d, name)), parse_pir("%s/%s.pir" % (d, name))
    assert len(gold) == len(res.nring)
    lr, lc, lu = np.diff(ro), np.diff(co), np.diff(uo)
    for w, g in enumerate(gold):
        assert (int(res.score1[w]), int(res.score2[w])) == (g["s1"], g["s2"])
        assert int(res.cells[w]) == int(lr[w] * lc[w] + g["n1"] * lu[w])
        assert res.window_rows(w) == pir[w][1]


def test_cli_dropin(golden_dir, tmp_path):
    """the poa executable with alignment.py's exact command line (alignment.py:60)"""
    from elector_b200.lib import poa_binary_path
    d = golden_dir
    out = str(tmp_path / "smsa0")
    p = subprocess.run([poa_binary_path(), "-pir", out, "-preserve_seqorder", "-corrected_reads_fasta", d + "/hard.cor.fa",
                        "-reference_reads_fasta", d + "/hard.ref.fa", "-uncorrected_reads_fasta", d + "/hard.unc.fa",
                        "-preserve_seqorder", "-threads", "1", "-pathMatrix", d + "/blosum80.mat"], capture_output=True)
    assert p.returncode == 0 and p.stderr == b""
    assert open(out, "rb").read() == open(d + "/hard.pir", "rb").read()
    assert p.stdout == b"0 1 2 \n" * 3000          # buildup_lpo.c:545


def test_random_windows_vs_oracle(ctx):
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    wins = synth.hard_windows(20000, seed=1234)
    r, ro = windows_to_csr([w[1] for w in wins]); c, co = windows_to_csr([w[2] for w in wins]); u, uo = windows_to_csr([w[3] for w in wins])
    res = ctx.run_csr(r, ro, c, co, u, uo)
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"])
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    assert np.array_equal(res.cells, o["cells"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), w


def test_large_tier_vs_oracle(ctx):
    """windows beyond the shared-memory tier (rows > 256) and int16-unsafe totals"""
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    rng = synth.SplitMix64(99)
    wins = []
    for L in (257, 300, 511, 700, 1100, 1900, 3300):
        ref = "".join("ACGT"[rng.below(4)] for _ in range(L))
        wins.append((ref, synth.mutate(rng, ref, 0.03, "ACGT"), synth.mutate(rng, ref, 0.12, "ACGT")))
    wins.append((wins[3][0], "N", wins[3][2]))                       # placeholder against a long window
    wins.append((wins[2][0], wins[2][1][:40], wins[2][2]))           # trimmed corrected
    r, ro = windows_to_csr([w[0] for w in wins]); c, co = windows_to_csr([w[1] for w in wins]); u, uo = windows_to_csr([w[2] for w in wins])
    res = ctx.run_csr(r, ro, c, co, u, uo)
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), w


def test_long_windows_warp_cooperative_vs_oracle():
    """windows of 120..600 letters (the segments the warp-cooperative kernels of poa_coop.cuh run, one and several
    256-row passes, odd and even lane counts, a partial group at the end of every segment with an odd count) against
    the oracle"""
    import elector_b200
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    rng = synth.SplitMix64(2025)
    wins = []
    for i in range(1203):
        L = 120 + rng.below(200) if i % 4 else 257 + rng.below(350)
        ab = ["ACGT", "AC", "ACGTN"][rng.below(3)]
        ref = "".join(ab[rng.below(len(ab))] for _ in range(L))
        cor = ref if i % 3 == 0 else (synth.mutate(rng, ref, [0.01, 0.05, 0.3][rng.below(3)], ab) or "A")
        if i % 17 == 0:
            cor = cor[len(cor) // 2:] or "N"
        if i % 29 == 0:
            cor = "N"
        unc = synth.mutate(rng, ref, [0.1, 0.2][rng.below(2)], ab) or "A"
        wins.append((ref, cor, unc))
    r, ro = windows_to_csr([w[0] for w in wins]); c, co = windows_to_csr([w[1] for w in wins]); u, uo = windows_to_csr([w[2] for w in wins])
    with elector_b200.PoaContext(0) as c2:
        res = c2.run_csr(r, ro, c, co, u, uo)
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"])
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), w


@pytest.mark.parametrize("band_w", ["0", "1", "3", "12"])
def test_band_dp_is_exact_whatever_the_width(band_w, monkeypatch):
    """the diagonal band of the packed linear kernels (DESIGN.md 4.4): windows that fail the exactness test are run again
    without the band by the same launch (per-warp retry queue); results equal the oracle at any half-width, 0 = band off"""
    import elector_b200
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    wins = synth.hard_windows(6000, seed=77)
    rng = synth.SplitMix64(78)
    for i in range(3000):                      # plus windows of the bulk's shape: cor == ref or nearly, unc at 10-20 %
        L = 20 + rng.below(110)
        ref = "".join("ACGT"[rng.below(4)] for _ in range(L))
        cor = ref if i % 2 else (synth.mutate(rng, ref, 0.02, "ACGT") or "A")
        wins.append(("b%d" % i, ref, cor, synth.mutate(rng, ref, [0.1, 0.2, 0.4][i % 3], "ACGT") or "A"))
    r, ro = windows_to_csr([w[1] for w in wins]); c, co = windows_to_csr([w[2] for w in wins]); u, uo = windows_to_csr([w[3] for w in wins])
    monkeypatch.setenv("ELECTOR_BAND_W", band_w)
    with elector_b200.PoaContext(0) as c2:
        res = c2.run_csr(r, ro, c, co, u, uo)
    o = oracle.batch(r, ro, c, co, u, uo, nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"])
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), w


def test_generic_matrix_vs_oracle(golden_dir, tmp_path):
    """non-uniform substitution scores and other gap penalties (table path of the kernel)"""
    import elector_b200
    from oracle import oracle, synth
    d = golden_dir
    mp = str(tmp_path / "m.mat")
    open(mp, "w").write(synth.matrix_text("table"))
    out, oout = str(tmp_path / "g.pir"), str(tmp_path / "o.pir")
    with elector_b200.PoaContext(0, mp) as c2:
        c2.files(d + "/hard.ref.fa", d + "/hard.cor.fa", d + "/hard.unc.fa", out)
    assert oracle.poa_files(mp, d + "/hard.ref.fa", d + "/hard.cor.fa", d + "/hard.unc.fa", oout) == 0
    assert open(out, "rb").read() == open(oout, "rb").read()


def matrix_sweep_params():
    from oracle import synth
    # the matrices whose small windows run packed, at the default band and at the narrowest
    return [pytest.param(m[0], b, id=m[0] + ("-band" + b if b else "")) for m in synth.MATRICES for b in ([None, "1"] if m[4][3] else [None])]


@pytest.mark.parametrize("mid,band_w", matrix_sweep_params())
def test_matrix_sweep_vs_oracle(tmp_path, mid, band_w, monkeypatch):
    """every matrix of oracle/synth.MATRICES: the packed class at its edges, INT32 compare-select (a positive match, one step
    outside the packed class, packed_ok beyond the small-window limit), the substitution table; on hard, bubble and the
    small edge windows, every output vs the oracle"""
    import elector_b200
    from elector_b200 import windows_to_csr
    from oracle import oracle, synth
    mp = str(tmp_path / "m.mat")
    open(mp, "w").write(synth.matrix_text(mid))
    if band_w is not None:
        monkeypatch.setenv("ELECTOR_BAND_W", band_w)
    S = synth.kernel_constants()["kSmallMax"]
    ma = next(m for m in synth.MATRICES if m[0] == mid)[4][2]
    wins = synth.hard_windows(3000) + synth.bubble_windows() + [w for w in synth.edge_windows(maxabs=ma) if max(map(len, w[1:])) <= S]
    r, ro = windows_to_csr([w[1] for w in wins]); c, co = windows_to_csr([w[2] for w in wins]); u, uo = windows_to_csr([w[3] for w in wins])
    with elector_b200.PoaContext(0, mp) as c2:
        res = c2.run_csr(r, ro, c, co, u, uo)
    o = oracle.batch(r, ro, c, co, u, uo, m=oracle.matrix(mp), nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"]) and np.array_equal(res.cells, o["cells"])
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), wins[w][0]


def test_errors(ctx, golden_dir, tmp_path):
    import elector_b200
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.run(["ACGT", "ACGT"], ["ACGT", ""], ["ACGT", "ACGT"])   # empty sequence: undefined in the reference
    assert e.value.code == -1
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.files(golden_dir + "/edge.ref.fa", str(tmp_path / "missing.fa"), golden_dir + "/edge.unc.fa", str(tmp_path / "o.pir"))
    assert e.value.code == -5
    # ragged record counts: common prefix aligned, error reported (reference: crash, SURVEY.md appendix A)
    rag = tmp_path / "short.cor.fa"
    rag.write_text("".join(open(golden_dir + "/edge.cor.fa").readlines()[:10]))
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.files(golden_dir + "/edge.ref.fa", str(rag), golden_dir + "/edge.unc.fa", str(tmp_path / "o.pir"))
    assert e.value.code == -5
    assert open(tmp_path / "o.pir").read() == "".join(open(golden_dir + "/edge.pir").readlines()[:30])
    res = ctx.run([], [], [])
    assert len(res.nring) == 0


def test_full_size_properties():
    """BASELINE.json configs[1]-shaped workload (a 600-triplet slice, ~117k windows): size-independent
    properties -- every MSA row spells its input sequence, results do not depend on batch composition
    or order, runs are deterministic -- plus a sampled comparison with the oracle."""
    import elector_b200
    import workloads
    from oracle import oracle
    wl = workloads.make_windows(1, 600)
    n = len(wl["ref_off"]) - 1
    with elector_b200.PoaContext(0) as c:
        res = c.run_csr(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"])
        res2 = c.run_csr(wl["ref"], wl["ref_off"], wl["cor"], wl["cor_off"], wl["unc"], wl["unc_off"])
        # reversed window order
        def rev(seq, off):
            lens = np.diff(off)[::-1]
            o2 = np.zeros(n + 1, np.int64); o2[1:] = np.cumsum(lens)
            parts = [seq[off[w]:off[w + 1]] for w in range(n - 1, -1, -1)]
            return np.concatenate(parts), o2
        rr, rro = rev(wl["ref"], wl["ref_off"]); cc, cco = rev(wl["cor"], wl["cor_off"]); uu, uuo = rev(wl["unc"], wl["unc_off"])
        res3 = c.run_csr(rr, rro, cc, cco, uu, uuo)
    assert np.array_equal(res.nring, res2.nring) and np.array_equal(res.score2, res2.score2)
    assert np.array_equal(res.nring, res3.nring[::-1]) and np.array_equal(res.score1, res3.score1[::-1])
    lower = np.arange(256, dtype=np.uint8); lower[65:91] += 32
    for w in range(0, n, 7):
        rows = res.window_rows(w)
        for s, key in enumerate(("ref", "cor", "unc")):
            seq = lower[wl[key][wl[key + "_off"][w]:wl[key + "_off"][w + 1]]].tobytes().decode()
            assert rows[s].replace(".", "") == seq
        assert rows == res3.window_rows(n - 1 - w)
    k = 20000
    o = oracle.batch(wl["ref"], wl["ref_off"][:k + 1], wl["cor"], wl["cor_off"][:k + 1], wl["unc"], wl["unc_off"][:k + 1], nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring[:k], o["nring"]) and np.array_equal(res.cells[:k], o["cells"])
    assert np.array_equal(res.score1[:k], o["score1"]) and np.array_equal(res.score2[:k], o["score2"])
    for w in range(k):
        assert res.window_rows(w) == oracle.window_rows(o, w)


def test_long_windows_equal_reference(ctx, golden_dir, tmp_path):
    """golden set `long` (reference-generated, oracle/make_golden_long.py): the 3 300-letter window runs the INT32 tier
    (scores beyond 16 bits), the 33 500-letter one is longer than a 32 KiB FASTA line buffer and than the former
    32 000-letter cap; PIR bytes, both DP scores and len(P1) equal the reference's"""
    d = golden_dir
    out = str(tmp_path / "o.pir")
    ctx.files(d + "/long.ref.fa", d + "/long.cor.fa", d + "/long.unc.fa", out)
    assert open(out, "rb").read() == open(d + "/long.pir", "rb").read()
    recs = [[s for _, s in read_fasta_simple("%s/long.%s.fa" % (d, k))] for k in ("ref", "cor", "unc")]
    gold = parse_dump(d + "/long.dump")
    res = ctx.run(recs[0], recs[1], recs[2])
    for w, g in enumerate(gold):
        assert (int(res.score1[w]), int(res.score2[w])) == (g["s1"], g["s2"]), w
        assert int(res.cells[w]) == len(recs[0][w]) * len(recs[1][w]) + g["n1"] * len(recs[2][w])


def test_window_beyond_the_cap_is_refused_not_approximated(ctx):
    """len(ref) + len(cor) > 65 534 (16-bit node indices): ELECTOR_ETOOLARGE with the reason, never a wrong answer"""
    import elector_b200
    with pytest.raises(elector_b200.ElectorError) as e:
        ctx.run(["A" * 40000], ["A" * 30000], ["ACGT"])
    assert e.value.code == -6 and "65534" in str(e.value)
