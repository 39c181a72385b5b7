"""GPU: the merge (merge_plan_kernel, merge_copy_kernel) and the tally (tally_read_kernel) on the reads of
oracle/synth.tally_edge_reads -- lengths around 16-column groups, 32-column words, 1 024-column steps and the shared-memory
bitmasks, border gaps, runs of the corrected and reference rows at word and step edges, cr at its threshold, stretches
within T_THRESH2 of a border, pending merges, overlapping keys -- read by read against oracle/tally_oracle.py: all 24
counters exactly, and the gap stretches the report (report_host.hpp, ReportRecords::mask) rebuilds its masks from."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
OFFSETS = (0, 1, 8, 15)   # byte offset of a read's rows mod 16: 0 takes the 16-byte vector path, the others the byte path


def expect(R, C, U):
    from elector_b200 import TALLY_FIELDS
    from oracle import tally_oracle as to
    t = to.tally_read(R, C, U)
    keys = sorted(to.gap_stretch_keys(C, R)) if t["assessed"] else []
    return [t[k] for k in TALLY_FIELDS], keys


@pytest.fixture(scope="module")
def corpus():
    """the edge reads with their oracle counters and stretches, and fillers of 1 .. 16 columns (checked as well)"""
    from oracle import synth
    reads = [(tag, R, C, U) for tag, R, C, U in synth.tally_edge_reads()]
    rng = synth.SplitMix64(99)
    fillers = [("filler", *("".join(x) for x in synth.msa_background(rng, f))) for f in range(1, 17)]
    return dict(reads=[(r, expect(*r[1:])) for r in reads], fillers=[(f, expect(*f[1:])) for f in fillers],
                S=synth.tally_constants()["kSmemCols"])


@pytest.fixture(scope="module")
def ctx():
    import elector_b200
    c = elector_b200.PoaContext(device=0)
    yield c
    c.close()


def layout(corpus, offset):
    """every edge read at a byte offset = `offset` mod 16, a filler read in front of each to set it"""
    items, at = [], 0
    for r in corpus["reads"]:
        f = (offset - at - 1) % 16 + 1
        items += [corpus["fillers"][f - 1], r]
        at += f + len(r[0][1])
    return items


def tally_and_compare(ctx, items):
    """elector_tally_run on the reads of `items` in one call; returns the mismatches against the oracle and the stretch counts"""
    from elector_b200 import TALLY_FIELDS
    out = ctx.tally([r[1] for r, _ in items], [r[2] for r, _ in items], [r[3] for r, _ in items])
    st = ctx.last_stretches(len(items))
    bad = []
    for i, ((tag, R, C, U), (cnt, keys)) in enumerate(zip([r for r, _ in items], [e for _, e in items])):
        got = [int(v) for v in out[i]]
        if got != cnt:
            bad.append((i, tag, len(R), {f: (g, e) for f, g, e in zip(TALLY_FIELDS, got, cnt) if g != e}))
        n = int(st[i, 0])
        gk = sorted((int(st[i, 1 + 2 * k]), int(st[i, 2 + 2 * k])) for k in range(min(n, 8)))
        if n != len(keys) or gk != keys:
            bad.append((i, tag, len(R), "stretches", gk, keys))
    return bad, st[:, 0]


@pytest.mark.parametrize("offset", OFFSETS)
def test_tally_edge_reads_at_every_row_offset(ctx, corpus, offset):
    """elector_tally_run: every edge read (and its filler) at this offset: counters and stretches equal the oracle's"""
    bad, _ = tally_and_compare(ctx, layout(corpus, offset))
    assert not bad, bad[:5]


def test_tally_long_reads_side_by_side(ctx, corpus):
    """reads longer than kSmemCols next to each other at unaligned offsets (their bitmasks in adjacent global plane ranges),
    then short reads, in one launch"""
    S = corpus["S"]
    long_ = [r for r in corpus["reads"] if len(r[0][1]) > S]
    short = [r for r in corpus["reads"] if len(r[0][1]) <= S]
    assert len(long_) >= 6
    items = [corpus["fillers"][0]] + long_ + short[::3] + long_[::-1]
    bad, _ = tally_and_compare(ctx, items)
    assert not bad, bad[:5]


def test_stretch_count_stays_within_the_bound(ctx, corpus):
    """no read can have more than 3 gap stretches (synth.tally_edge_reads): the device finds the oracle's count on every read,
    reaches 3 and never sets the overflow flag (elector_tally_run would fail with ELECTOR_EUNSUPPORTED)"""
    from oracle import synth
    items = layout(corpus, 0)
    bad, nk = tally_and_compare(ctx, items)
    assert not bad, bad[:5]
    assert [len(e[1]) for _, e in items] == nk.tolist()
    assert nk.max() == 3 < synth.tally_constants()["kMaxStretchKeys"]


def windows_of(rng, rows, n_frac=0.0, n_windows=0):
    """cuts the merged rows (R, C, U) into windows of 1 .. 300 columns; n_frac of the columns of a window come back as
    placeholders ('n' in the corrected row) and n_windows windows of placeholders only go in between: the merge drops both"""
    R, C, U = (np.frombuffer(s.encode("latin-1"), np.uint8) for s in rows)
    L, cuts = len(R), [0]
    while cuts[-1] < L:
        cuts.append(min(L, cuts[-1] + int(rng.integers(1, 301))))
    junk = np.frombuffer(b".acgtNRY", np.uint8)
    wins = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        w = [R[a:b], C[a:b], U[a:b]]
        if n_frac:
            k = b - a
            m = int(rng.binomial(k, n_frac))
            where = np.sort(rng.integers(0, k + 1, m))
            w = [np.insert(x, where, junk[rng.integers(0, len(junk), m)]) for x in w]
            w[1][where + np.arange(m)] = ord("n")
        wins.append(w)
    for _ in range(n_windows):
        k = int(rng.integers(1, 200))
        w = [junk[rng.integers(0, len(junk), k)] for _ in range(3)]
        w[1][:] = ord("n")
        wins.insert(int(rng.integers(0, len(wins) + 1)), w)
    return wins


@pytest.fixture(scope="module")
def merged_input(corpus):
    """the edge reads cut into windows (with and without placeholder columns), plus reads that are 0, 1, 10 and 11 columns
    after the drop, laid out as a PoaResult (rows 4-byte aligned and padded, in another order than the windows)"""
    from elector_b200.poa import PoaResult
    from oracle import synth
    rng = np.random.default_rng(23)
    items = list(corpus["reads"])
    srng = synth.SplitMix64(5)
    for L in (0, 1, 10, 11):
        rows = tuple("".join(x) for x in synth.msa_background(srng, L))
        items.append((("drop L=%d" % L, *rows), expect(*rows)))
    wins, first = [], [0]
    for i, ((tag, R, C, U), _) in enumerate(items):
        w = windows_of(rng, (R, C, U), n_frac=[0.0, 0.02, 0.3][i % 3], n_windows=int(i % 4 == 0 or len(R) <= 11) * int(rng.integers(1, 4)))
        wins += w
        first.append(len(wins))
    k = np.array([len(w[0]) for w in wins], np.int64)
    stride = (k + 3) & ~3
    perm = rng.permutation(len(wins))
    row_off = np.empty(len(wins), np.int64)
    row_off[perm] = np.concatenate([[0], np.cumsum(3 * stride[perm])])[:-1]
    rows = np.zeros(int(3 * stride.sum()), np.uint8)
    for w, x in enumerate(wins):
        for s in range(3):
            rows[row_off[w] + s * stride[w]:row_off[w] + s * stride[w] + k[w]] = x[s]
    res = PoaResult(rows, row_off, stride.astype(np.int32), k.astype(np.int32), np.zeros(len(wins), np.int32),
                    np.zeros(len(wins), np.int32), np.zeros(len(wins), np.int64))
    return dict(items=items, res=res, read_first=np.array(first, np.int64))


def test_merge_returns_the_edge_reads(ctx, merged_input):
    """elector_merge_run: the windows of every read (more than 32 for the long ones: merge_plan_kernel takes 32 per step)
    concatenate to the read's rows once the placeholder columns are dropped"""
    m = merged_input
    assert np.diff(m["read_first"]).max() > 32
    got = ctx.merge(m["res"], m["read_first"])
    bad = [(i, r[0]) for i, ((r, _), g) in enumerate(zip(m["items"], got)) if g != r[1:]]
    assert not bad, bad[:5]


def test_merge_tally_device_and_sums_on_edge_reads(ctx, merged_input):
    """elector_merge_tally_device (the merged rows' lengths from the merge, bitmask planes sized by the merged capacity) gives
    the oracle's counters on every read; elector_tally_sum_device over them gives the column sums, `extended` over the
    reads that have one"""
    import torch
    from elector_b200 import TALLY_FIELDS
    m = merged_input
    res, rf = m["res"], m["read_first"]
    n_reads, n_win = len(rf) - 1, len(res.nring)
    dev = torch.device("cuda", 0)
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(res, k))).to(dev) for k in ("rows", "row_off", "row_stride", "nring")}
    d_cnt = torch.zeros(n_reads * len(TALLY_FIELDS), dtype=torch.int64, device=dev)
    ctx._check(ctx._lib.elector_merge_tally_device(ctx._ctx, n_reads, rf.ctypes.data, n_win, d["rows"].data_ptr(), len(res.rows),
                                                   d["row_off"].data_ptr(), d["row_stride"].data_ptr(), d["nring"].data_ptr(), d_cnt.data_ptr()))
    got = d_cnt.cpu().numpy().reshape(n_reads, -1)
    exp = np.array([e[0] for _, e in m["items"]], np.int64)
    bad = [(i, m["items"][i][0][0], {f: (int(g), int(e)) for f, g, e in zip(TALLY_FIELDS, got[i], exp[i]) if g != e})
           for i in range(n_reads) if not np.array_equal(got[i], exp[i])]
    assert not bad, bad[:5]
    d_sums = torch.zeros(len(TALLY_FIELDS), dtype=torch.int64, device=dev)
    ctx._check(ctx._lib.elector_tally_sum_device(ctx._ctx, n_reads, d_cnt.data_ptr(), d_sums.data_ptr()))
    ext = TALLY_FIELDS.index("extended")
    want = exp.sum(axis=0)
    want[ext] = exp[:, ext][exp[:, ext] >= 0].sum()
    assert np.array_equal(d_sums.cpu().numpy(), want)


def test_report_from_device_stretches_equals_report_from_oracle(ctx, corpus, tmp_path):
    """elector_report_write from the device's counters and stretches and from the oracle's: byte-identical files, log and
    printed text.  Split reads (consecutive records with one header) end on a fragment with stretches, where
    ReportRecords::mask rebuilds the columns no fragment keeps from them"""
    import elector_b200
    items = [r for r in corpus["reads"] if len(r[0][1]) > 10]
    heads, i, nsplit = [], 0, 0
    while i < len(items):
        if i + 2 < len(items) and items[i + 2][1][1] and nsplit < 40:   # the third record has stretches: a read in three fragments
            heads += ["split%d " % i] * 3
            i += 3
            nsplit += 1
        else:
            heads.append("read%d " % i)
            i += 1
    assert nsplit >= 20
    rows = [r for r, _ in items]
    cnt_dev = ctx.tally([r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows])
    st_dev = ctx.last_stretches(len(rows))
    cnt_or = np.array([e[0] for _, e in items], np.int64)
    st_or = np.zeros_like(st_dev)
    for k, (_, keys) in enumerate(e for _, e in items):
        st_or[k, 0] = len(keys)
        for j, (a, b) in enumerate(keys):
            st_or[k, 1 + 2 * j], st_or[k, 2 + 2 * j] = a, b
    out = {}
    for name, cnt, st in (("device", cnt_dev, st_dev), ("oracle", cnt_or, st_or)):
        d = tmp_path / name
        d.mkdir()
        res = elector_b200.report_write(heads, cnt, st, [r[1] for r in rows], [r[2] for r in rows], out_dir=str(d))
        out[name] = (res["log"], res["stdout"], (d / "per_read_metrics.txt").read_bytes(), (d / "read_size_distribution.txt").read_bytes())
        assert res["split_reads"] == nsplit
    assert out["device"] == out["oracle"]
