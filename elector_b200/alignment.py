"""Batched, in-process replacement of elector/alignment.py:getPOA (SURVEY.md 8f-3).

The reference runs, per round of 10 001 triplets: one `masterSplitter` process (alignment.py:98-100), up to 200 `poa` processes through
a multiprocessing.Pool (fpoa, :59-63, :117-119), 200 `Donatello` processes (:120-124) and two `rm` shells over ~800 temporary files.
`getPOA` here has the reference's signature, return value and output file (`<outDir>/msa.fa` or `msa_<soft>.fa`, same bytes), and is one
C-ABI call per batch of triplets on a context that stays alive between calls (elector_reads_pipeline_run: the windows never leave the
device; the library cuts the call into chunks that run on worker contexts of one or more devices: ELECTOR_DEVICES="0,1,..", else the
context's device ELECTOR_DEVICE); no process is started and no temporary file is written.  The per-read counters of the last call are kept for computeStats.py's
replacement (elector_b200/computeStats.py), which then needs no tally pass over msa.fa at all."""
import os

import numpy as np

from .poa import PoaContext

_CTX = None
BATCH_TRIPLETS = 200000    # triplets per call: bounds the host buffers of the merged rows (3 x the letters of a batch); the device side is chunked by the library
LAST = None                # what the last getPOA left for the report: dict(headers, counters, stretches, msa_path)


def context(device=None):
    """the persistent context of this process (one CUDA context, scratch pools kept across calls)"""
    global _CTX
    if _CTX is None:
        _CTX = PoaContext(int(os.environ.get("ELECTOR_DEVICE", "0")) if device is None else device)
    return _CTX


def devices():
    """the devices of the reads-in call: ELECTOR_DEVICES="0,1,..", else None (the context's own device)"""
    e = os.environ.get("ELECTOR_DEVICES", "").strip()
    return [int(d) for d in e.split(",") if d.strip()] if e else None


def read_two_line_fasta(path):
    """the splitter's reading of its inputs (Master_Splitter.cpp:405-412: one header line, one sequence line per record)
    -> (headers list[bytes] with '>', uint8 letters, int64 offsets[n + 1])"""
    raw = np.fromfile(path, dtype=np.uint8)
    if raw.size == 0:
        return [], np.zeros(0, np.uint8), np.zeros(1, np.int64)
    if raw[-1] != 10:
        raw = np.concatenate((raw, np.asarray([10], np.uint8)))
    nl = np.flatnonzero(raw == 10)
    if len(nl) % 2:
        nl = nl[:-1]                     # a header without a sequence line at the end of the file
    starts = np.concatenate(([0], nl[:-1] + 1))
    hs, he, ss, se = starts[0::2], nl[0::2], starts[1::2], nl[1::2]
    lens = (se - ss).astype(np.int64)
    off = np.zeros(len(lens) + 1, np.int64)
    off[1:] = np.cumsum(lens)
    keep = np.zeros(raw.size, dtype=bool)
    if off[-1]:
        keep[np.repeat(ss - off[:-1], lens) + np.arange(off[-1])] = True
    b = raw.tobytes()
    return [b[a:e] for a, e in zip(hs.tolist(), he.tolist())], raw[keep], off


def pir_header(h):
    """the header line `poa` writes for a record whose FASTA header line is h (fasta_format.c:35-37, lpo_format.c:407-421)"""
    t = h[1:].split(None, 1)
    name = t[0] if t else ""
    title = t[1].rstrip() if len(t) > 1 and t[1].strip() else "untitled"
    return ">" + name + " " + title


def getPOA(corrected, reference, uncorrected, threads, outDir, SIZE_CORRECTED_READ_THRESHOLD, soft=None):
    """alignment.py:66-131 (oldMode False).  `threads` is accepted and ignored: the devices run every window of a batch at once."""
    global LAST
    ctx = context()
    merge_out = outDir + ("/msa_" + soft + ".fa" if soft is not None else "/msa.fa")
    hr, ref, ro = read_two_line_fasta(reference)
    _, unc, uo = read_two_line_fasta(uncorrected)
    _, cor, co = read_two_line_fasta(corrected)
    n = min(len(ro), len(uo), len(co)) - 1
    # records whose reference read has at most 2 letters are not triplets (Master_Splitter.cpp:414)
    keep = np.flatnonzero((ro[1:n + 1] - ro[:n]) > 2)
    small_reads = wrongly_cor_reads = 0
    heads, counters, stretches = [], [], []
    with open(merge_out, "ab") as out:                       # Donatello appends (Donatello.cpp:48)
        for b0 in range(0, len(keep), BATCH_TRIPLETS):
            idx = keep[b0:b0 + BATCH_TRIPLETS]

            def gather(let, off):
                lens = off[idx + 1] - off[idx]
                o = np.zeros(len(idx) + 1, np.int64)
                o[1:] = np.cumsum(lens)
                if idx[-1] - idx[0] + 1 == len(idx):                   # a contiguous range: no copy
                    return let[off[idx[0]]:off[idx[-1] + 1]], o
                pos = np.repeat(off[idx] - o[:-1], lens) + np.arange(o[-1])
                return let[pos], o
            (r, r_o), (u, u_o), (c, c_o) = gather(ref, ro), gather(unc, uo), gather(cor, co)
            got = ctx.reads_pipeline(r, r_o, u, u_o, c, c_o, [len(hr[t]) for t in idx], float(SIZE_CORRECTED_READ_THRESHOLD), merged=True,
                                     devices=devices())
            st = got["stretches"]
            small_reads += int((got["status"] == 1).sum())
            wrongly_cor_reads += int((got["status"] == 2).sum())
            chunks = []
            for k, t in enumerate(idx):
                o, l = int(got["m_off"][k]), int(got["m_len"][k])
                if l <= 1:                                   # Donatello.cpp:70
                    continue
                h = pir_header(hr[t].decode("latin-1"))
                h = (h[:len(h) - 11] + " \n").encode("latin-1")   # Donatello.cpp:72-74
                for key in ("m_ref", "m_cor", "m_unc"):
                    chunks += [h, got[key][o:o + l].tobytes(), b"\n"]
                heads.append(h[1:-1].decode("latin-1"))
                counters.append(got["counters"][k])
                stretches.append(st[k])
            out.write(b"".join(chunks))
    LAST = dict(headers=heads, counters=np.asarray(counters, np.int64).reshape(-1, 24), stretches=np.asarray(stretches, np.int32).reshape(-1, 17),
                msa_path=os.path.abspath(merge_out))
    return small_reads, wrongly_cor_reads
