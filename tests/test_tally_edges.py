"""CPU: oracle/synth.tally_edge_reads sits on the edges of the tally kernel (tally_kernel.cuh) -- every read has the shape its
tag states (lengths, border gaps, extension, dot runs, cr, gap stretches: synth.tally_measures, from the oracle), and every
edge tests/test_gpu_tally_edges.py relies on is in the set, so a later edit of the generator cannot quietly leave one."""
import pytest


@pytest.fixture(scope="module")
def reads():
    from oracle import synth
    return synth.tally_edge_reads()


def test_tally_edge_reads_sit_on_their_edges(reads):
    from oracle import synth
    for tag, R, C, U in reads:
        assert len(R) == len(C) == len(U) and "n" not in C, tag
        assert not synth.tally_tag_mismatches(tag, R, C, U), (tag, synth.tally_tag_mismatches(tag, R, C, U))


def test_tally_edge_reads_cover_every_edge(reads):
    from oracle import synth
    k = synth.tally_constants()
    T, T2, S = k["T_THRESH"], k["T_THRESH2"], k["kSmemCols"]
    tags = {t for t, _, _, _ in reads}
    names = {t.split()[0] for t in tags}
    lengths = {len(R) for _, R, _, _ in reads}
    assert {10, 11, 15, 16, 17, 31, 32, 33, 1023, 1024, 1025, 2049, S - 1, S, S + 1, 65537} <= lengths
    assert max(lengths) >= 150000
    assert {"bordl:n%d" % n for n in (T - 1, T, T2 - 1, T2, T2 + 1)} <= names
    assert {"bordr:n%d" % n for n in (T - 1, T, T2 - 1, T2, T2 + 1)} <= names
    assert {"bordsepl:sep%d" % s for s in (T, T + 1)} | {"bordsepr:sep%d" % s for s in (T, T + 1)} | {"bordw", "bordmin", "borde"} <= names
    assert {"crunr:a%d" % a for a in (31, 32, 1023, 1024, 2047, 2048)} <= names
    assert {"crunl:b%d" % b for b in (31, 32, 1023, 1024, 2047, 2048)} <= names
    assert {"crunk:n%d" % n for n in (1, 2, T - 1, T, T + 1)} | {"crunstep"} <= names
    assert {"cr:n%d" % n for n in (T2 - 1, T2, T2 + 1)} | {"crsr:k0", "crsr:k1", "crsr:k1dot", "crs0:k0", "crs0:k1", "crpre", "crrb"} <= names
    assert {"slotl:a%d" % a for a in (T2, T2 + 1)} | {"slotr:d%d" % d for d in (T2, T2 + 1)} | {"slotp:g%d" % g for g in (T, T + 1)} <= names
    assert {"cls", "keys3"} | {"mask:i%d" % i for i in range(16)} <= names
    # each shape on several backgrounds
    assert all(sum(t == u for u, _, _, _ in reads) >= 3 for t in tags)
    # mask ends at every offset inside a 16-column group: gapsLeft, L - gapsRight and both ends of the keys
    m = [synth.tally_measures(R, C, U) for t, R, C, U in reads if t.startswith("mask:")]
    assert {int(x["gl"]) % 16 for x in m} == set(range(16)) and {(int(x["L"]) - int(x["gr"])) % 16 for x in m} == set(range(16))
    ends = [[int(v) for v in key.split("-")] for x in m for key in x["keys"].split(",")]
    assert {a % 16 for a, b in ends if a} == set(range(16)) and {b % 16 for a, b in ends} == set(range(16))


def test_no_read_has_more_than_three_gap_stretches(reads):
    """the bound of synth.tally_edge_reads' docstring: the set reaches 3 keys, overlapping ones included, and no more"""
    from oracle import synth, tally_oracle as to
    nk = {tag: len(to.gap_stretch_keys(C, R)) for tag, R, C, U in reads}
    assert max(nk.values()) == 3 < synth.tally_constants()["kMaxStretchKeys"]
    assert [t for t in nk if t.startswith("keys3")] and all(nk[t] == 3 for t in nk if t.startswith("keys3"))
