"""GPU: windows at the edges of the device scheduler (oracle/synth.edge_windows) -- sort bins and big tiers of both phases,
the cor-is-ref shortcut and the d-classes of the linear bins, the band span limit, lopsided shapes, the 16-bit node cap --
each alone in a call (its segment holds one window) and as letter variants mixed into config-1 windows (partial groups,
bulk and side streams), under the launcher's settings that change which kernel a window meets, against the oracle."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VARIANTS = 33      # a full warp and a partial group of every edge shape


def csr(wins):
    from elector_b200 import windows_to_csr
    return [a for k in (1, 2, 3) for a in windows_to_csr([w[k] for w in wins])]


@pytest.fixture(scope="module")
def edges():
    """the edge windows, the mixed call (edge variants shuffled into ~5 000 config-1 windows) and the oracle's results for the
    mixed call and for the cap windows, which run alone only: a segment's scratch is sized by its longest len(P1) times its
    longest uncorrected sequence, so one call holding both the 65 000-node windows and the 65 534-letter uncorrected one is
    refused (ELECTOR_ETOOLARGE, ~76 GB of scratch) -- a limit of the launcher, not an edge of the kernels."""
    import workloads
    from oracle import oracle, synth
    wins = synth.edge_windows()
    too_large = [w for w in wins if w[0].startswith("toolarge")]
    wins = [w for w in wins if not w[0].startswith("toolarge")]
    wl = workloads.make_windows(1, 26)
    mix = [("c%d" % i,) + tuple(wl[k][wl[k + "_off"][i]:wl[k + "_off"][i + 1]].tobytes().decode() for k in ("ref", "cor", "unc"))
           for i in range(len(wl["ref_off"]) - 1)]
    caps = [w for w in wins if w[0].startswith("cap")]
    for i, w in enumerate(wins):
        if w not in caps:
            mix += synth.letter_variants(("e%d %s" % (i, w[0]),) + w[1:], VARIANTS, seed=i)   # tags may repeat, names do not
    order = np.random.default_rng(11).permutation(len(mix))
    mix = [mix[i] for i in order]
    where = {w[0]: i for i, w in enumerate(mix)}
    alone = [len(mix) + caps.index(w) if w in caps else where["e%d %s v0" % (i, w[0])] for i, w in enumerate(wins)]   # w in the oracle results
    o = oracle.batch(*csr(mix + caps), nthreads=os.cpu_count() or 1)
    return dict(wins=wins, too_large=too_large, mix=mix, alone=alone, oracle=o)


def assert_window(res, i, o, j, what):
    got = (int(res.nring[i]), int(res.score1[i]), int(res.score2[i]), int(res.cells[i]), res.window_rows(i))
    from oracle import oracle
    want = (int(o["nring"][j]), int(o["score1"][j]), int(o["score2"][j]), int(o["cells"][j]), oracle.window_rows(o, j))
    assert got == want, what


SETTINGS = {
    "default": {},
    "band0": {"ELECTOR_BAND_W": "0"},
    "band1": {"ELECTOR_BAND_W": "1"},
}


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_edge_windows_alone_and_mixed_vs_oracle(edges, setting, monkeypatch):
    import elector_b200
    for k, v in SETTINGS[setting].items():
        monkeypatch.setenv(k, v)
    o = edges["oracle"]
    with elector_b200.PoaContext(0) as c:
        for w, j in zip(edges["wins"], edges["alone"]):
            assert_window(c.run_csr(*csr([w])), 0, o, j, w[0])
        res = c.run_csr(*csr(edges["mix"]))
    for i, w in enumerate(edges["mix"]):
        assert_window(res, i, o, i, w[0])


def test_edge_windows_through_the_pipeline(edges, monkeypatch):
    """the pipelined call (three chunks, one read per window) computes for every window the rows and scores of run_csr"""
    import elector_b200
    monkeypatch.setenv("ELECTOR_PIPELINE_CHUNKS", "3")
    args = csr(edges["mix"])
    with elector_b200.PoaContext(0) as c:
        want = c.run_csr(*args)
        got, _, _ = c.pipeline_csr(*args, np.arange(len(edges["mix"]) + 1, dtype=np.int64))
    for a in ("nring", "score1", "score2", "cells"):
        assert np.array_equal(getattr(got, a), getattr(want, a)), a
    for i in range(len(edges["mix"])):
        assert got.window_rows(i) == want.window_rows(i), edges["mix"][i][0]


def test_one_node_beyond_the_cap_is_refused(edges):
    """len(ref) + len(cor) == kMaxNodes + 1: ELECTOR_ETOOLARGE (the windows at kMaxNodes exactly run above)"""
    import elector_b200
    (w,) = edges["too_large"]
    with elector_b200.PoaContext(0) as c:
        with pytest.raises(elector_b200.ElectorError) as e:
            c.run_csr(*csr([w]))
        assert e.value.code == -6
        with pytest.raises(elector_b200.ElectorError) as e:            # the cor-heavy orientation
            c.run_csr(*csr([(w[0], w[2], w[1], w[3])]))
        assert e.value.code == -6
