"""CPU: the per-window DEVICE code (elector_b200/csrc/poa_kernel.cuh) compiled as host code
and run by tests/emul/poa_emul.cu, against the reference goldens.  This checks the kernel's
restructuring (8-row register bands, two frontier sets, 2-bit moves + ordinals, fused
emit) without a GPU; the GPU tests then check the real launch path."""
import subprocess

import pytest

from conftest import GOLDEN_SETS, parse_dump, read_fasta_simple
from oracle import synth


@pytest.mark.parametrize("mode", ["int32", "packed", "dual-general", "coop"])
@pytest.mark.parametrize("name", GOLDEN_SETS)
def test_emulated_kernel_equals_reference(golden_dir, emul_bin, name, mode, tmp_path):
    """mode packed: the 16-bit packed kernels wherever the library would use them (Phase1P, Phase2L for windows whose P1 is
    linear, the dual-frontier Phase2D of poa_dual.cuh for the rest); dual-general: Phase2D for every window; coop: both DPs
    of every window through the warp-cooperative wavefront of poa_coop.cuh (32 lanes of 8 rows, emulated lane by lane).
    The emulator also checks that the number of MSA columns announced before the fusion equals the number emitted."""
    d = golden_dir
    pir, sc = str(tmp_path / "e.pir"), str(tmp_path / "e.scores")
    cmd = [emul_bin, d + "/blosum80.mat", "%s/%s.ref.fa" % (d, name), "%s/%s.cor.fa" % (d, name),
           "%s/%s.unc.fa" % (d, name), pir, sc] + ([mode] if mode != "int32" else [])
    assert subprocess.call(cmd) == 0
    assert open(pir, "rb").read() == open("%s/%s.pir" % (d, name), "rb").read()
    gold = parse_dump("%s/%s.dump" % (d, name))
    got = [tuple(int(v) for v in line.split()) for line in open(sc)]
    assert len(got) == len(gold)
    for g, e in zip(gold, got):
        assert (g["s1"], g["s2"], g["n1"]) == e[:3]


@pytest.mark.parametrize("band_w", ["1", "3", "6", "16"])
@pytest.mark.parametrize("name", ["hard", "example_tail"])
def test_emulated_band_dp_is_exact(golden_dir, emul_bin, name, band_w, tmp_path, monkeypatch):
    """the diagonal-band DP of the packed linear kernels with its exactness test (poa_packed.cuh): whatever the half-width,
    a window either passes the test and equals the reference, or is run again without the band"""
    monkeypatch.setenv("ELECTOR_BAND_W", band_w)
    d = golden_dir
    pir, sc = str(tmp_path / "e.pir"), str(tmp_path / "e.scores")
    cmd = [emul_bin, d + "/blosum80.mat", "%s/%s.ref.fa" % (d, name), "%s/%s.cor.fa" % (d, name), "%s/%s.unc.fa" % (d, name), pir, sc, "packed"]
    assert subprocess.call(cmd) == 0
    assert open(pir, "rb").read() == open("%s/%s.pir" % (d, name), "rb").read()
    gold = parse_dump("%s/%s.dump" % (d, name))
    got = [tuple(int(v) for v in line.split()) for line in open(sc)]
    assert [(g["s1"], g["s2"], g["n1"]) for g in gold] == [e[:3] for e in got]


MATRIX_IDS = [m[0] for m in synth.MATRICES]


@pytest.fixture(scope="module")
def sweep(golden_dir, tmp_path_factory):
    """inputs of the matrix sweep: the golden set `hard`, bubble windows for the dual-frontier kernel and the small windows of
    the edge set (every sequence <= kSmallMax: the packed kernels' size classes), as FASTA files; the oracle's PIR per
    matrix, computed once"""
    d = str(tmp_path_factory.mktemp("sweep"))
    S = synth.kernel_constants()["kSmallMax"]
    hard = list(zip(*[[s for _, s in read_fasta_simple("%s/hard.%s.fa" % (golden_dir, key))] for key in ("ref", "cor", "unc")]))
    wins = [("h%d" % i,) + w for i, w in enumerate(hard)] + synth.bubble_windows(2000)
    wins += [w for w in synth.edge_windows() if max(map(len, w[1:])) <= S]
    synth.write_windows([("w%d" % i,) + w[1:] for i, w in enumerate(wins)], d + "/in")
    return {"dir": d, "oracle": {}}


def sweep_matrix(sweep, mid):
    from oracle import oracle
    mp = "%s/%s.mat" % (sweep["dir"], mid)
    if mid not in sweep["oracle"]:
        open(mp, "w").write(synth.matrix_text(mid))
        opir = "%s/%s.oracle.pir" % (sweep["dir"], mid)
        assert oracle.poa_files(mp, *["%s/in.%s.fa" % (sweep["dir"], k) for k in ("ref", "cor", "unc")], opir) == 0
        sweep["oracle"][mid] = open(opir, "rb").read()
    return mp, sweep["oracle"][mid]


def test_emulated_kernel_generic_matrix(golden_dir, emul_bin, tmp_path):
    """non-uniform substitution scores + other gap penalties: table path vs the oracle"""
    from oracle import oracle
    d = golden_dir
    mp = str(tmp_path / "m.mat")
    open(mp, "w").write(synth.matrix_text("table"))
    pir, opir = str(tmp_path / "e.pir"), str(tmp_path / "o.pir")
    assert subprocess.call([emul_bin, mp, d + "/hard.ref.fa", d + "/hard.cor.fa", d + "/hard.unc.fa", pir]) == 0
    assert oracle.poa_files(mp, d + "/hard.ref.fa", d + "/hard.cor.fa", d + "/hard.unc.fa", opir) == 0
    assert open(pir, "rb").read() == open(opir, "rb").read()


@pytest.mark.parametrize("mode", ["int32", "packed", "dual-general", "coop"])
@pytest.mark.parametrize("mid", MATRIX_IDS)
def test_emulated_kernel_matrix_sweep(sweep, emul_bin, mid, mode, tmp_path):
    """every matrix of oracle/synth.MATRICES (the packed class at its edges, INT32 compare-select, the substitution table)
    through every kernel family, on hard, bubble and small edge windows, vs the oracle"""
    mp, want = sweep_matrix(sweep, mid)
    pir = str(tmp_path / "e.pir")
    ins = ["%s/in.%s.fa" % (sweep["dir"], k) for k in ("ref", "cor", "unc")]
    assert subprocess.call([emul_bin, mp] + ins + [pir] + (["-", mode] if mode != "int32" else []), stderr=subprocess.DEVNULL) == 0
    assert open(pir, "rb").read() == want


@pytest.mark.parametrize("mid", MATRIX_IDS)
def test_matrix_lands_in_its_class(golden_dir, emul_bin, mid, tmp_path):
    """ScoringSetup::analyse puts each matrix of the sweep into the class oracle/synth.MATRICES names for it (packed_ok,
    generic_sub, maxabs, small windows packed): no matrix can drift into another kernel family unnoticed"""
    mp = str(tmp_path / "m.mat")
    open(mp, "w").write(synth.matrix_text(mid))
    d = golden_dir
    p = subprocess.run([emul_bin, mp, d + "/edge.ref.fa", d + "/edge.cor.fa", d + "/edge.unc.fa", str(tmp_path / "e.pir")],
                       capture_output=True, text=True)
    assert p.returncode == 0
    line = [l for l in p.stderr.splitlines() if l.startswith("matrix class:")]
    assert len(line) == 1
    t = line[0].split()
    got = tuple(int(t[t.index(key) + 1]) for key in ("packed_ok", "generic_sub", "maxabs", "small_packed"))
    assert got == next(m[4] for m in synth.MATRICES if m[0] == mid)


def test_emulated_kernel_rejects_unsupported_matrix(golden_dir, emul_bin, tmp_path):
    from elector_b200.matrix import default_matrix_text
    mp = str(tmp_path / "m.mat")
    open(mp, "w").write(default_matrix_text(gaps=(10, 5, 1)))  # decaying extension penalty
    d = golden_dir
    rc = subprocess.call([emul_bin, mp, d + "/edge.ref.fa", d + "/edge.cor.fa", d + "/edge.unc.fa", str(tmp_path / "x.pir")],
                         stderr=subprocess.DEVNULL)
    assert rc == 3


@pytest.mark.parametrize("mode", ["int32", "packed", "dual-general", "coop"])
def test_emulated_kernel_long_windows(golden_dir, emul_bin, mode, tmp_path):
    """many bands, 8- and 16-row last bands, long placeholder / trimmed windows, vs the oracle"""
    from oracle import oracle, synth
    rng = synth.SplitMix64(4242)
    wins = []
    for L in (15, 16, 17, 24, 25, 31, 32, 33, 40, 41, 129, 257, 300, 511, 700, 1100):
        ref = "".join("ACGT"[rng.below(4)] for _ in range(L))
        wins.append((ref, synth.mutate(rng, ref, 0.03, "ACGT") or "A", synth.mutate(rng, ref, 0.12, "ACGT") or "A"))
        wins.append((ref, synth.mutate(rng, ref, 0.3, "AC") or "A", synth.mutate(rng, ref, 0.3, "AC") or "A"))
    wins.append((wins[-2][0], "N", wins[-2][2]))
    wins.append((wins[-3][0], wins[-3][1][:40], wins[-3][2]))
    wins.append(("ACGT" * 30, "ACGT" * 30, "A"))
    paths = []
    for k, key in enumerate(("ref", "cor", "unc")):
        p = str(tmp_path / (key + ".fa"))
        with open(p, "w") as f:
            for i, w in enumerate(wins):
                f.write(">w%d\n%s\n" % (i, w[k]))
        paths.append(p)
    pir, opir = str(tmp_path / "e.pir"), str(tmp_path / "o.pir")
    mp = golden_dir + "/blosum80.mat"
    assert subprocess.call([emul_bin, mp, paths[0], paths[1], paths[2], pir] + (["-", mode] if mode != "int32" else [])) == 0
    assert oracle.poa_files(mp, paths[0], paths[1], paths[2], opir) == 0
    assert open(pir, "rb").read() == open(opir, "rb").read()


@pytest.mark.parametrize("mode", ["packed", "dual-general"])
def test_emulated_dual_kernel_on_bubble_windows(golden_dir, emul_bin, mode, tmp_path):
    """the skewed two-set dual kernel (poa_dual.cuh) on ELECTOR-like windows: a corrected sequence with a few differences (bubbles
    that open and close at every position of a band, in the low and in the high half, back to back, at the first and at the last
    node; late starts and early ends of either sequence) against a noisier uncorrected one, lengths around the band sizes"""
    from oracle import oracle, synth
    synth.write_windows(synth.bubble_windows(6000, seed=20261018), str(tmp_path / "in"))
    paths = [str(tmp_path / ("in.%s.fa" % key)) for key in ("ref", "cor", "unc")]
    pir, opir = str(tmp_path / "e.pir"), str(tmp_path / "o.pir")
    mp = golden_dir + "/blosum80.mat"
    assert subprocess.call([emul_bin, mp, paths[0], paths[1], paths[2], pir, "-", mode], stderr=subprocess.DEVNULL) == 0
    assert oracle.poa_files(mp, paths[0], paths[1], paths[2], opir) == 0
    assert open(pir, "rb").read() == open(opir, "rb").read()
