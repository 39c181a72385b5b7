"""Bench / test infrastructure: synthetic workloads of the BASELINE.json configs.

reads (tools/gen_reads.c, seeded)  ->  windows (the UNCHANGED reference splitter,
oracle/_ref/masterSplitter, run as parallel instances over read slices exactly like
elector/alignment.py:99 runs it: `... 7 200 10000 <minfrac> <outdir>`)  ->  CSR arrays.
The timed regions of bench.py start from these arrays in host memory (SURVEY.md 8d).
Nothing here reads /root/reference: the splitter binary travels in oracle/_ref.  If it
is absent the windows are synthesised directly with the splitter's observed length
distribution and the workload name says so.
"""
import os
import shutil
import subprocess
import tempfile
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
SPLITTER = os.path.join(ROOT, "oracle", "_ref", "masterSplitter")
GEN = os.path.join(ROOT, "tools", "gen_reads")
# per user: a directory another user created first is not writable
CACHE = os.environ.get("ELECTOR_CACHE", os.path.join(tempfile.gettempdir(), "elector_b200_cache_%d" % os.getuid()))

CONFIG_NAMES = {
    1: "synthetic 10k triplets, 10 kb reads, 10% raw / 1% corrected error",
    2: "synthetic 100k triplets, 15 kb ONT-like reads at 12% error, split/trimmed corrected reads",
    3: "synthetic 20k triplets, 50-100 kb ultra-long reads",
    4: "synthetic 1M triplets of mixed 1-30 kb reads",
}
CONFIG_READS = {1: 10000, 2: 100000, 3: 20000, 4: 1000000}


_GEN_LOCK = threading.Lock()


def ensure_gen():
    """builds tools/gen_reads once (threads of make_windows call this concurrently)"""
    src = os.path.join(ROOT, "tools", "gen_reads.c")
    with _GEN_LOCK:
        if not os.path.exists(GEN) or os.path.getmtime(GEN) < os.path.getmtime(src):
            tmp = "%s.tmp%d" % (GEN, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-o", tmp, src, "-lm"])
            os.replace(tmp, GEN)
    return GEN


def parse_two_line_fasta(path):
    """2-lines-per-record FASTA -> (headers list[bytes], uint8 letters, int64 offsets[n+1])"""
    raw = np.fromfile(path, dtype=np.uint8)
    if raw.size == 0:
        return [], np.zeros(0, np.uint8), np.zeros(1, np.int64)
    nl = np.flatnonzero(raw == 10)
    starts = np.concatenate(([0], nl[:-1] + 1))
    hs, he = starts[0::2], nl[0::2]
    ss, se = starts[1::2], nl[1::2]
    lens = (se - ss).astype(np.int64)
    off = np.zeros(len(lens) + 1, np.int64)
    off[1:] = np.cumsum(lens)
    # gather sequence bytes: mask out header lines and newlines
    keep = np.zeros(raw.size, dtype=bool)
    idx = np.repeat(ss - off[:-1], lens) + np.arange(off[-1])
    keep[idx] = True
    seq = raw[keep]
    b = raw.tobytes()
    headers = [b[a:e] for a, e in zip(hs.tolist(), he.tolist())]
    return headers, seq, off


def _split_slice(args):
    cfg, first, count, minfrac = args
    work = tempfile.mkdtemp(prefix="elsplit_")
    try:
        pre = os.path.join(work, "r")
        subprocess.check_call([ensure_gen(), str(cfg), str(count), str(first), pre])
        out = os.path.join(work, "out")
        os.makedirs(out)
        rc = subprocess.call([SPLITTER, pre + ".ref.fa", pre + ".unc.fa", pre + ".cor.fa", out + "/out1", out + "/out2",
                              out + "/out3", "7", "200", "10000", str(minfrac), out], stdout=subprocess.DEVNULL)
        if rc != 0:
            raise RuntimeError("masterSplitter returned %d (slice larger than one round?)" % rc)
        parts = []
        for i in range(200):
            p3 = "%s/out3%d" % (out, i)
            if not os.path.exists(p3) or os.path.getsize(p3) == 0:
                continue
            h, r, ro = parse_two_line_fasta("%s/out1%d" % (out, i))
            _, u, uo = parse_two_line_fasta("%s/out2%d" % (out, i))
            _, c, co = parse_two_line_fasta(p3)
            assert len(ro) == len(uo) == len(co)
            parts.append((h, r, ro, c, co, u, uo))
        return parts
    finally:
        shutil.rmtree(work, ignore_errors=True)


def _concat(parts):
    heads, segs = [], {k: [] for k in "rcu"}
    offs = {k: [np.zeros(1, np.int64)] for k in "rcu"}
    tot = {k: 0 for k in "rcu"}
    for h, r, ro, c, co, u, uo in parts:
        heads += h
        for k, s, o in (("r", r, ro), ("c", c, co), ("u", u, uo)):
            segs[k].append(s)
            offs[k].append(o[1:] + tot[k])
            tot[k] += int(o[-1])
    cat = {k: (np.concatenate(segs[k]) if segs[k] else np.zeros(0, np.uint8)) for k in "rcu"}
    off = {k: np.concatenate(offs[k]) for k in "rcu"}
    # windows of one read are consecutive and share the header (Master_Splitter.cpp:283-285)
    first = [0]
    for i in range(1, len(heads)):
        if heads[i] != heads[i - 1]:
            first.append(i)
    first.append(len(heads))
    return dict(ref=cat["r"], ref_off=off["r"], cor=cat["c"], cor_off=off["c"], unc=cat["u"], unc_off=off["u"],
                read_first=np.asarray(first, np.int64))


def _direct_windows(cfg, n_reads, first_read):
    """fallback without the splitter binary: windows drawn with the observed length distribution"""
    rng = np.random.default_rng(1000 * cfg + first_read)
    per_read = {1: 195, 2: 286, 3: 1387, 4: 160}[cfg]
    n = n_reads * per_read
    lens = np.clip(rng.gamma(9.0, 5.7, n).astype(np.int64), 20, 480)
    ref_off = np.zeros(n + 1, np.int64); ref_off[1:] = np.cumsum(lens)
    ref = rng.integers(0, 4, ref_off[-1], dtype=np.uint8)

    def mutate(rate):
        # substitutions + deletions only (keeps the generator vectorised)
        r = rng.random(ref.size)
        sub = r < rate * 0.5
        dele = (r >= rate * 0.5) & (r < rate)
        x = np.where(sub, (ref + 1 + rng.integers(0, 3, ref.size, dtype=np.uint8)) % 4, ref).astype(np.uint8)
        win = np.repeat(np.arange(n), lens)
        first_of = np.zeros(ref.size, bool); first_of[ref_off[:-1]] = True
        keep = ~dele | first_of
        l2 = np.bincount(win[keep], minlength=n).astype(np.int64)
        off = np.zeros(n + 1, np.int64); off[1:] = np.cumsum(l2)
        return x[keep], off

    lut = np.frombuffer(b"ACGT", np.uint8)
    unc, unc_off = mutate(0.10)
    cor, cor_off = mutate(0.01)
    rf = np.arange(0, n + 1, per_read, dtype=np.int64)
    return dict(ref=lut[ref], ref_off=ref_off, cor=lut[cor], cor_off=cor_off, unc=lut[unc], unc_off=unc_off, read_first=rf)


def make_windows(cfg, n_reads, first_read=0, procs=None, minfrac=0.1, cache=True):
    """Returns dict(ref, ref_off, cor, cor_off, unc, unc_off, read_first, source)."""
    os.makedirs(CACHE, exist_ok=True)
    have_splitter = os.path.exists(SPLITTER)
    key = os.path.join(CACHE, "cfg%d_n%d_f%d_%s.npz" % (cfg, n_reads, first_read, "split" if have_splitter else "direct"))
    if cache and os.path.exists(key):
        z = np.load(key)
        d = {k: z[k] for k in z.files}
        d["source"] = "reference masterSplitter" if have_splitter else "direct synthesis (splitter binary absent)"
        return d
    if have_splitter:
        procs = procs or max(1, (os.cpu_count() or 2) - 1)
        per = max(8, min(2000, (n_reads + procs * 4 - 1) // (procs * 4)))
        jobs = [(cfg, first_read + s, min(per, n_reads - s), minfrac) for s in range(0, n_reads, per)]
        with ThreadPoolExecutor(max_workers=procs) as ex:
            res = list(ex.map(_split_slice, jobs))
        d = _concat([p for parts in res for p in parts])
    else:
        d = _direct_windows(cfg, n_reads, first_read)
    if cache:
        tmp = key + ".tmp%d.npz" % os.getpid()
        np.savez(tmp, **d)
        os.replace(tmp, key)
    d["source"] = "reference masterSplitter" if have_splitter else "direct synthesis (splitter binary absent)"
    return d


from elector_b200.shard import shard_reads, slice_windows  # noqa: E402,F401  (host logic of SURVEY.md 8e lives in the package)
