"""GPU: the device sorts and the launch order of one call against the oracle -- every window in one phase-1 bin and one
phase-2 bin (a whole tile of the scatter on one key), only windows whose cor is ref (empty phase 1 and general view), no such
window (empty linear view), and the edge windows mixed into config-1 windows, three calls on one context."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def csr(wins):
    from elector_b200 import windows_to_csr
    return [a for k in (1, 2, 3) for a in windows_to_csr([w[k] for w in wins])]


def check(ctx, wins):
    from oracle import oracle
    args = csr(wins)
    res = ctx.run_csr(*args)
    o = oracle.batch(*args, nthreads=os.cpu_count() or 1)
    assert np.array_equal(res.nring, o["nring"])
    assert np.array_equal(res.score1, o["score1"]) and np.array_equal(res.score2, o["score2"])
    assert np.array_equal(res.cells, o["cells"])
    for w in range(len(wins)):
        assert res.window_rows(w) == oracle.window_rows(o, w), "MSA rows differ at window %d" % w


def config1(n):
    import workloads
    wl = workloads.make_windows(1, 26)
    return [("c%d" % i,) + tuple(wl[k][wl[k + "_off"][i]:wl[k + "_off"][i + 1]].tobytes().decode() for k in ("ref", "cor", "unc"))
            for i in range(min(n, len(wl["ref_off"]) - 1))]


@pytest.fixture(scope="module")
def ctx():
    import elector_b200
    with elector_b200.PoaContext(device=0) as c:
        yield c


def test_hot_bin(ctx):
    """5 000 windows of one shape (lengths equal, one substitution at the same place): one bin in each phase"""
    rng = np.random.default_rng(3)
    ref = "".join(rng.choice(list("ACGT"), 80))
    cor = ref[:40] + ("A" if ref[40] != "A" else "C") + ref[41:]
    wins = []
    for i in range(5000):
        unc = list(ref)
        unc[int(rng.integers(0, 80))] = "ACGT"[int(rng.integers(0, 4))]
        wins.append(("h%d" % i, ref, cor, "".join(unc)))
    check(ctx, wins)


def test_only_cor_is_ref(ctx):
    wins = [w for w in config1(6000) if w[1] == w[2]]
    assert len(wins) > 1000
    check(ctx, wins)


def test_no_cor_is_ref(ctx):
    wins = [w for w in config1(6000) if w[1] != w[2]]
    assert len(wins) > 500
    check(ctx, wins)


def test_edges_mixed_three_calls(ctx):
    from oracle import synth
    edges = [w for w in synth.edge_windows() if not w[0].startswith(("toolarge", "cap"))]
    base = config1(4000)
    for call in range(3):
        rng = np.random.default_rng(100 + call)
        mix = base + edges
        mix = [mix[i] for i in rng.permutation(len(mix))]
        check(ctx, mix)
