"""Host-side mirror of the `poa` boundary over the C-ABI (include/elector_poa.h).

The reference's interface for this path is the `poa` command line (main.c:85-113) and
its PIR output (lpo_format.c:398-426); `PoaContext.files()` is that call in-process,
`PoaContext.run()` is the same computation on in-memory windows, `PoaContext.tally()`
the integer part of computeStats.py's per-read tally.  numpy is used for the host
buffers only; all arithmetic happens in the CUDA library.
"""
import ctypes
from dataclasses import dataclass

import numpy as np

from .lib import load_library

TALLY_FIELDS = ["TP", "FP", "FN", "cor", "uncor", "uncorCor", "uncorUncor", "insC", "delC", "subsC",
                "insU", "delU", "subsU", "GCref", "GCcor", "lenRef", "lenCor", "lenUnc", "gapsLeft",
                "gapsRight", "missing", "extended", "ncols", "assessed"]


NIBBLE_CHARS = ".acgtnA"   # ELECTOR_NIBBLE_CHARS: 4-bit column codes of the merged rows; 15 = listed in the escape arrays


class PackedC(ctypes.Structure):     # struct elector_packed
    _fields_ = [("bits", ctypes.c_void_p), ("n_letters", ctypes.c_int64), ("exc_pos", ctypes.c_void_p),
                ("exc_byte", ctypes.c_void_p), ("n_exc", ctypes.c_int64)]


class PipelineIoC(ctypes.Structure):  # struct elector_pipeline_io
    _fields_ = [("n_windows", ctypes.c_int64), ("n_reads", ctypes.c_int64),
                ("ref", ctypes.c_void_p), ("cor", ctypes.c_void_p), ("unc", ctypes.c_void_p),
                ("pref", ctypes.c_void_p), ("pcor", ctypes.c_void_p), ("punc", ctypes.c_void_p),
                ("ref_off", ctypes.c_void_p), ("cor_off", ctypes.c_void_p), ("unc_off", ctypes.c_void_p), ("read_first", ctypes.c_void_p),
                ("ref_len", ctypes.c_void_p), ("cor_len", ctypes.c_void_p), ("unc_len", ctypes.c_void_p),
                ("rows_out", ctypes.c_void_p), ("rows_cap", ctypes.c_int64), ("row_off", ctypes.c_void_p), ("row_stride", ctypes.c_void_p),
                ("nring", ctypes.c_void_p), ("score1", ctypes.c_void_p), ("score2", ctypes.c_void_p), ("cells", ctypes.c_void_p),
                ("m_ref", ctypes.c_void_p), ("m_cor", ctypes.c_void_p), ("m_unc", ctypes.c_void_p), ("m_cap", ctypes.c_int64), ("m_nibbles", ctypes.c_int),
                ("m_off", ctypes.c_void_p), ("m_len", ctypes.c_void_p),
                ("m_esc_pos", ctypes.c_void_p), ("m_esc_byte", ctypes.c_void_p), ("m_esc_cap", ctypes.c_int64), ("m_n_esc", ctypes.c_void_p),
                ("counters_out", ctypes.c_void_p), ("sums_out", ctypes.c_void_p),
                ("ref_len16", ctypes.c_void_p), ("cor_len16", ctypes.c_void_p), ("unc_len16", ctypes.c_void_p)]


class ReadsIoC(ctypes.Structure):     # struct elector_reads_io
    _fields_ = [("n_triplets", ctypes.c_int64),
                ("ref", ctypes.c_void_p), ("unc", ctypes.c_void_p), ("cor", ctypes.c_void_p),
                ("ref_off", ctypes.c_void_p), ("unc_off", ctypes.c_void_p), ("cor_off", ctypes.c_void_p),
                ("header_len", ctypes.c_void_p), ("threshold", ctypes.c_double),
                ("devices", ctypes.c_void_p), ("n_devices", ctypes.c_int),
                ("status", ctypes.c_void_p), ("k_used", ctypes.c_void_p),
                ("read_first", ctypes.c_void_p), ("n_windows", ctypes.c_void_p),
                ("counters_out", ctypes.c_void_p), ("sums_out", ctypes.c_void_p),
                ("stretches_out", ctypes.c_void_p),
                ("m_ref", ctypes.c_void_p), ("m_cor", ctypes.c_void_p), ("m_unc", ctypes.c_void_p),
                ("m_off", ctypes.c_void_p), ("m_len", ctypes.c_void_p), ("m_cap", ctypes.c_int64)]


def reads_merged_bound(ref_off, unc_off, cor_off):
    """bytes per merged-row buffer that elector_reads_pipeline_run needs: letters of the call + 32 per triplet, rounded up to 16"""
    n = len(ref_off) - 1
    letters = sum(int(o[n] - o[0]) for o in (ref_off, unc_off, cor_off))
    return (letters + 32 * n + 15) & ~15


@dataclass
class PackedLetters:
    """2 bits per letter + the exceptions (elector_pack_letters)"""
    bits: np.ndarray
    n_letters: int
    exc_pos: np.ndarray
    exc_byte: np.ndarray

    def c_struct(self):
        return PackedC(self.bits.ctypes.data, self.n_letters, self.exc_pos.ctypes.data, self.exc_byte.ctypes.data, len(self.exc_pos))


def pack_letters(letters):
    """uint8 array of FASTA letters -> PackedLetters"""
    lib = load_library()
    letters = np.ascontiguousarray(letters, dtype=np.uint8)
    n = len(letters)
    bits = np.zeros((n + 3) // 4 + 8, np.uint8)
    cap = 1024
    while True:
        pos, byt = np.zeros(cap, np.int64), np.zeros(cap, np.uint8)
        ne = int(lib.elector_pack_letters(letters.ctypes.data, n, bits.ctypes.data, pos.ctypes.data, byt.ctypes.data, cap))
        if ne <= cap:
            return PackedLetters(bits, n, pos[:ne].copy(), byt[:ne].copy())
        cap = ne + 16


class ElectorError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("elector error %d: %s" % (code, msg))
        self.code = code


def windows_to_csr(seqs):
    """list of str/bytes -> (uint8 array of all letters, int64 offsets[n+1])"""
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs])
    cat = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if bs else np.zeros(0, np.uint8)
    return cat, off


@dataclass
class PoaResult:
    rows: np.ndarray        # uint8 buffer holding every row
    row_off: np.ndarray     # int64[n]
    row_stride: np.ndarray  # int32[n]
    nring: np.ndarray       # int32[n]
    score1: np.ndarray
    score2: np.ndarray
    cells: np.ndarray       # int64[n]

    def window_rows(self, w):
        o, st, k = int(self.row_off[w]), int(self.row_stride[w]), int(self.nring[w])
        return tuple(self.rows[o + s * st:o + s * st + k].tobytes().decode("latin-1") for s in range(3))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


class PoaContext:
    """One context per device per thread (like one `poa` process)."""

    def __init__(self, device=0, matrix_path=None):
        self._lib = load_library()
        self._ctx = ctypes.c_void_p()
        mp = matrix_path.encode() if matrix_path else None
        rc = self._lib.elector_poa_init(int(device), mp, ctypes.byref(self._ctx))
        if rc != 0:
            msg = self._lib.elector_last_error(None).decode()
            self._ctx = None
            raise ElectorError(rc, msg)

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.elector_poa_free(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise ElectorError(rc, self._lib.elector_last_error(self._ctx).decode())

    def run_csr(self, ref, ref_off, cor, cor_off, unc, unc_off, rows=None):
        n = len(ref_off) - 1
        ref_off, cor_off, unc_off = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, cor_off, unc_off))
        ref, cor, unc = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, cor, unc))
        bound = self._lib.elector_poa_rows_bound(n, _p(ref_off), _p(cor_off), _p(unc_off)) if n else 0
        if rows is None or len(rows) < bound:
            rows = np.empty(max(bound, 1), dtype=np.uint8)
        res = PoaResult(rows, np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32),
                        np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int64))
        self._check(self._lib.elector_poa_run(self._ctx, n, _p(ref), _p(ref_off), _p(cor), _p(cor_off), _p(unc),
                                              _p(unc_off), _p(res.rows), len(res.rows), _p(res.row_off),
                                              _p(res.row_stride), _p(res.nring), _p(res.score1), _p(res.score2),
                                              _p(res.cells)))
        return res

    def run(self, refs, cors, uncs):
        """refs/cors/uncs: equal-length lists of window sequences (str or bytes)."""
        r, ro = windows_to_csr(refs)
        c, co = windows_to_csr(cors)
        u, uo = windows_to_csr(uncs)
        return self.run_csr(r, ro, c, co, u, uo)

    def pipeline_csr(self, ref, ref_off, cor, cor_off, unc, unc_off, read_first):
        """alignment.py's Pool(fpoa) + Donatello + the integer part of computeStats in one call
        (elector_pipeline_run).  Returns (PoaResult, counters int64[n_reads, K], sums int64[K])."""
        n = len(ref_off) - 1
        ref_off, cor_off, unc_off, read_first = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, cor_off, unc_off, read_first))
        ref, cor, unc = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, cor, unc))
        n_reads = len(read_first) - 1
        bound = self._lib.elector_poa_rows_bound(n, _p(ref_off), _p(cor_off), _p(unc_off)) if n else 0
        res = PoaResult(np.empty(max(bound, 1), dtype=np.uint8), np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32),
                        np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int64))
        counters = np.zeros((n_reads, len(TALLY_FIELDS)), dtype=np.int64)
        sums = np.zeros(len(TALLY_FIELDS), dtype=np.int64)
        self._check(self._lib.elector_pipeline_run(self._ctx, n, _p(ref), _p(ref_off), _p(cor), _p(cor_off), _p(unc), _p(unc_off),
                                                   n_reads, _p(read_first), _p(res.rows), len(res.rows), _p(res.row_off),
                                                   _p(res.row_stride), _p(res.nring), _p(res.score1), _p(res.score2), _p(res.cells),
                                                   _p(counters), _p(sums)))
        return res, counters, sums

    def pipeline_io(self, ref, ref_off, cor, cor_off, unc, unc_off, read_first, packed=False, window_rows=False, merged="bytes", lengths32=False, lengths16=False):
        """elector_pipeline_run2: letters as bytes or 2-bit packed (PackedLetters or packed=True to pack here), outputs chosen by
        the caller: window_rows (PoaResult), merged = "bytes" | "nibbles" | None, always the counters and sums.
        Returns dict(res, merged (list of (R, C, U) strings or None), counters, sums, m_len)."""
        lib = self._lib
        n = len(ref_off) - 1
        ref_off, cor_off, unc_off, read_first = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, cor_off, unc_off, read_first))
        n_reads = len(read_first) - 1
        io = PipelineIoC()
        io.n_windows, io.n_reads = n, n_reads
        keep = []
        if packed:
            pk = [s if isinstance(s, PackedLetters) else pack_letters(s) for s in (ref, cor, unc)]
            cs = [p.c_struct() for p in pk]
            keep += pk + cs
            io.pref, io.pcor, io.punc = (ctypes.addressof(c) for c in cs)
            if lengths16:
                lens = [np.ascontiguousarray(np.diff(o), dtype=np.uint16) for o in (ref_off, cor_off, unc_off)]
                keep += lens
                io.ref_len16, io.cor_len16, io.unc_len16 = (l.ctypes.data for l in lens)
            elif lengths32:
                lens = [np.ascontiguousarray(np.diff(o), dtype=np.int32) for o in (ref_off, cor_off, unc_off)]
                keep += lens
                io.ref_len, io.cor_len, io.unc_len = (l.ctypes.data for l in lens)
        else:
            ref, cor, unc = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, cor, unc))
            keep += [ref, cor, unc]
            io.ref, io.cor, io.unc = ref.ctypes.data, cor.ctypes.data, unc.ctypes.data
        io.ref_off, io.cor_off, io.unc_off, io.read_first = ref_off.ctypes.data, cor_off.ctypes.data, unc_off.ctypes.data, read_first.ctypes.data
        res = PoaResult(np.zeros(1, np.uint8), np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32),
                        np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int64))
        if window_rows:
            bound = lib.elector_poa_rows_bound(n, _p(ref_off), _p(cor_off), _p(unc_off)) if n else 0
            res.rows = np.empty(max(bound, 1), dtype=np.uint8)
            io.rows_out, io.rows_cap, io.row_off, io.row_stride = res.rows.ctypes.data, len(res.rows), res.row_off.ctypes.data, res.row_stride.ctypes.data
        io.nring, io.score1, io.score2, io.cells = res.nring.ctypes.data, res.score1.ctypes.data, res.score2.ctypes.data, res.cells.ctypes.data
        counters = np.zeros((n_reads, len(TALLY_FIELDS)), dtype=np.int64)
        sums = np.zeros(len(TALLY_FIELDS), dtype=np.int64)
        io.counters_out, io.sums_out = counters.ctypes.data, sums.ctypes.data
        m = m_off = m_len = esc_pos = esc_byte = None
        n_esc = np.zeros(1, np.int64)
        if merged:
            cap = int(lib.elector_merged_bound(n, n_reads, _p(ref_off), _p(cor_off), _p(unc_off)))
            nib = merged in ("nibbles", "columns")
            m = [np.zeros(cap // 2 + 16 if merged == "nibbles" else cap, np.uint8) for _ in range(3)]
            m_off, m_len = np.zeros(n_reads, np.int64), np.zeros(n_reads, np.int32)
            io.m_ref, io.m_cor, io.m_unc, io.m_cap, io.m_nibbles = m[0].ctypes.data, m[1].ctypes.data, m[2].ctypes.data, cap, {"nibbles": 1, "columns": 2}.get(merged, 0)
            io.m_off, io.m_len = m_off.ctypes.data, m_len.ctypes.data
            if nib:
                esc_pos, esc_byte = np.zeros(65536, np.int64), np.zeros(65536, np.uint8)
                io.m_esc_pos, io.m_esc_byte, io.m_esc_cap, io.m_n_esc = esc_pos.ctypes.data, esc_byte.ctypes.data, len(esc_pos), n_esc.ctypes.data
        self._check(lib.elector_pipeline_run2(self._ctx, ctypes.byref(io)))
        rows = None
        if merged == "bytes":
            rows = [tuple(m[s][m_off[r]:m_off[r] + m_len[r]].tobytes().decode("latin-1") for s in range(3)) for r in range(n_reads)]
        elif merged == "nibbles":
            lut = np.frombuffer((NIBBLE_CHARS + "?" * (16 - len(NIBBLE_CHARS))).encode(), np.uint8)
            full = []
            for s in range(3):
                b = np.empty(2 * len(m[s]), np.uint8)
                b[0::2] = lut[m[s] & 15]
                b[1::2] = lut[m[s] >> 4]
                full.append(b)
            for k in range(int(n_esc[0])):
                full[int(esc_pos[k] % 3)][int(esc_pos[k] // 3)] = esc_byte[k]
            rows = [tuple(full[s][m_off[r]:m_off[r] + m_len[r]].tobytes().decode("latin-1") for s in range(3)) for r in range(n_reads)]
        elif merged == "columns":   # one byte per column: elector_unpack_columns + the escape list
            full = [np.empty(cap, np.uint8) for _ in range(3)]
            lib.elector_unpack_columns(ctypes.c_void_p(m[0].ctypes.data), ctypes.c_int64(cap), *(ctypes.c_void_p(f.ctypes.data) for f in full))
            for k in range(int(n_esc[0])):
                full[int(esc_pos[k] % 3)][int(esc_pos[k] // 3)] = esc_byte[k]
            rows = [tuple(full[s][m_off[r]:m_off[r] + m_len[r]].tobytes().decode("latin-1") for s in range(3)) for r in range(n_reads)]
        return dict(res=res, merged=rows, counters=counters, sums=sums, m_len=m_len, n_esc=int(n_esc[0]))

    def split_csr(self, ref, ref_off, unc, unc_off, cor, cor_off, header_len, threshold=0.1):
        """One masterSplitter round on in-memory reads (elector_split_run; Master_Splitter.cpp:352-472 minus the files): the
        windows of every triplet as CSR letter arrays, in triplet order.  -> dict(status, k_used, read_first, ref, ref_off,
        unc, unc_off, cor, cor_off)"""
        n = len(ref_off) - 1
        ref_off, unc_off, cor_off = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, unc_off, cor_off))
        ref, unc, cor = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, unc, cor))
        header_len = np.ascontiguousarray(header_len, dtype=np.int32)
        caps = [ctypes.c_int64() for _ in range(4)]
        self._check(self._lib.elector_split_bounds(n, _p(ref_off), _p(unc_off), _p(cor_off), *[ctypes.cast(ctypes.byref(c), ctypes.c_void_p) for c in caps]))
        wcap, rcap, ucap, ccap = (int(c.value) for c in caps)
        status, k_used = np.zeros(n, np.int32), np.zeros(n, np.int32)
        read_first = np.zeros(n + 1, np.int64)
        wo = [np.zeros(wcap + 1, np.int64) for _ in range(3)]
        wl = [np.empty(max(cap, 1), np.uint8) for cap in (rcap, ucap, ccap)]
        nw = ctypes.c_int64()
        self._check(self._lib.elector_split_run(self._ctx, n, _p(ref), _p(ref_off), _p(unc), _p(unc_off), _p(cor), _p(cor_off), _p(header_len),
                                                float(threshold), _p(status), _p(k_used), _p(read_first), wcap, _p(wo[0]), _p(wo[1]), _p(wo[2]),
                                                _p(wl[0]), rcap, _p(wl[1]), ucap, _p(wl[2]), ccap, ctypes.cast(ctypes.byref(nw), ctypes.c_void_p)))
        nw = int(nw.value)
        out = dict(status=status, k_used=k_used, read_first=read_first, n_windows=nw)
        for name, o, l in zip(("ref", "unc", "cor"), wo, wl):
            out[name + "_off"] = o[:nw + 1]
            out[name] = l[:int(o[nw])] if nw else l[:0]
        return out

    def reads_run(self, ref, ref_off, unc, unc_off, cor, cor_off, header_len, threshold=0.1, merged=False):
        """alignment.py:98-129 from the reads on (elector_reads_run): window cutting, alignment, per-triplet merge and tally in one
        call; the windows stay on the device.  -> dict(status, k_used, read_first, n_windows, counters, sums[, merged rows])"""
        n = len(ref_off) - 1
        ref_off, unc_off, cor_off = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, unc_off, cor_off))
        ref, unc, cor = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, unc, cor))
        header_len = np.ascontiguousarray(header_len, dtype=np.int32)
        status, k_used = np.zeros(n, np.int32), np.zeros(n, np.int32)
        read_first = np.zeros(n + 1, np.int64)
        counters = np.zeros((n, len(TALLY_FIELDS)), dtype=np.int64)
        sums = np.zeros(len(TALLY_FIELDS), dtype=np.int64)
        nw = ctypes.c_int64()
        m_cap = int(ref_off[n] - ref_off[0] + unc_off[n] - unc_off[0] + cor_off[n] - cor_off[0]) + 32 * n + 64 if merged else 0
        m = [np.empty(max(m_cap, 1), np.uint8) for _ in range(3)] if merged else [None] * 3
        m_off, m_len = (np.zeros(n, np.int64), np.zeros(n, np.int32)) if merged else (None, None)
        self._check(self._lib.elector_reads_run(self._ctx, n, _p(ref), _p(ref_off), _p(unc), _p(unc_off), _p(cor), _p(cor_off), _p(header_len),
                                                float(threshold), _p(status), _p(k_used), _p(read_first), ctypes.cast(ctypes.byref(nw), ctypes.c_void_p),
                                                _p(counters), _p(sums), _p(m[0]), _p(m[1]), _p(m[2]), m_cap, _p(m_off), _p(m_len)))
        out = dict(status=status, k_used=k_used, read_first=read_first, n_windows=int(nw.value), counters=counters, sums=sums)
        if merged:
            out.update(m_ref=m[0], m_cor=m[1], m_unc=m[2], m_off=m_off, m_len=m_len)
        return out

    def reads_pipeline(self, ref, ref_off, unc, unc_off, cor, cor_off, header_len, threshold=0.1, merged=False, devices=None, m_cap=None):
        """reads_run for any number of triplets (elector_reads_pipeline_run): the call is cut into chunks of whole triplets that run on
        worker contexts of `devices` (None: this context's device; a device may be listed more than once).  -> the dict of reads_run
        plus "stretches" (int32[n, 17], what last_stretches gives after reads_run).  m_cap: merged-row capacity (default: the bound)."""
        n = len(ref_off) - 1
        ref_off, unc_off, cor_off = (np.ascontiguousarray(o, dtype=np.int64) for o in (ref_off, unc_off, cor_off))
        ref, unc, cor = (np.ascontiguousarray(s, dtype=np.uint8) for s in (ref, unc, cor))
        header_len = np.ascontiguousarray(header_len, dtype=np.int32)
        status, k_used = np.zeros(n, np.int32), np.zeros(n, np.int32)
        read_first = np.zeros(n + 1, np.int64)
        counters = np.zeros((n, len(TALLY_FIELDS)), dtype=np.int64)
        sums = np.zeros(len(TALLY_FIELDS), dtype=np.int64)
        stretches = np.zeros((n, 17), dtype=np.int32)
        nw = np.zeros(1, np.int64)
        io = ReadsIoC()
        io.n_triplets = n
        io.ref, io.unc, io.cor = ref.ctypes.data, unc.ctypes.data, cor.ctypes.data
        io.ref_off, io.unc_off, io.cor_off = ref_off.ctypes.data, unc_off.ctypes.data, cor_off.ctypes.data
        io.header_len, io.threshold = header_len.ctypes.data, float(threshold)
        dev = np.ascontiguousarray(devices if devices is not None else [], dtype=np.intc)
        io.devices, io.n_devices = (dev.ctypes.data if len(dev) else None), len(dev)
        io.status, io.k_used, io.read_first, io.n_windows = status.ctypes.data, k_used.ctypes.data, read_first.ctypes.data, nw.ctypes.data
        io.counters_out, io.sums_out, io.stretches_out = counters.ctypes.data, sums.ctypes.data, stretches.ctypes.data
        if merged:
            cap = reads_merged_bound(ref_off, unc_off, cor_off) if m_cap is None else int(m_cap)
            m = [np.zeros(max(cap, 1), np.uint8) for _ in range(3)]
            m_off, m_len = np.zeros(n, np.int64), np.zeros(n, np.int32)
            io.m_ref, io.m_cor, io.m_unc = (b.ctypes.data for b in m)
            io.m_off, io.m_len, io.m_cap = m_off.ctypes.data, m_len.ctypes.data, cap
        self._check(self._lib.elector_reads_pipeline_run(self._ctx, ctypes.byref(io)))
        out = dict(status=status, k_used=k_used, read_first=read_first, n_windows=int(nw[0]), counters=counters, sums=sums, stretches=stretches)
        if merged:
            out.update(m_ref=m[0], m_cor=m[1], m_unc=m[2], m_off=m_off, m_len=m_len)
        return out

    def last_reads_ms(self):
        a, b, c = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
        self._lib.elector_last_reads_ms(self._ctx, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        return a.value, b.value, c.value

    def files(self, ref_fasta, cor_fasta, unc_fasta, pir_out, print_perm=False):
        """The body of one `poa` process (main.c:241-287)."""
        self._check(self._lib.elector_poa_files(self._ctx, ref_fasta.encode(), cor_fasta.encode(), unc_fasta.encode(),
                                                pir_out.encode(), int(bool(print_perm))))

    def tally(self, rows_ref, rows_cor, rows_unc):
        """Per-read integer counters (computeStats.py) for merged MSA rows; returns int64[n, K]."""
        r, off = windows_to_csr(rows_ref)
        c, off_c = windows_to_csr(rows_cor)
        u, off_u = windows_to_csr(rows_unc)
        if not (np.array_equal(off, off_c) and np.array_equal(off, off_u)):
            raise ValueError("the three rows of a read must have equal length")
        n = len(off) - 1
        out = np.zeros((n, len(TALLY_FIELDS)), dtype=np.int64)
        self._check(self._lib.elector_tally_run(self._ctx, n, _p(r), _p(c), _p(u), _p(off), _p(out)))
        return out

    def last_stretches(self, n_reads):
        """Border gap stretches of the reads of the last tally on this context: int32[n, 17] (count, then first / last column pairs)."""
        out = np.zeros((n_reads, 17), dtype=np.int32)
        self._check(self._lib.elector_last_stretches(self._ctx, n_reads, _p(out)))
        return out

    def merge(self, res, read_first):
        """Donatello's per-read merge of a PoaResult (Donatello.cpp:50-84); returns list of (R, C, U) strings."""
        read_first = np.ascontiguousarray(read_first, dtype=np.int64)
        n_reads, n_win = len(read_first) - 1, len(res.nring)
        used = int((res.row_off + 3 * res.row_stride.astype(np.int64)).max()) if n_win else 0
        cap = int(res.nring.sum()) + 16 * n_reads + 16
        m = [np.zeros(cap, np.uint8) for _ in range(3)]
        m_off, m_len = np.zeros(n_reads, np.int64), np.zeros(n_reads, np.int32)
        self._check(self._lib.elector_merge_run(self._ctx, n_reads, _p(read_first), n_win, _p(res.rows), used, _p(res.row_off),
                                                _p(res.row_stride), _p(res.nring), _p(m[0]), _p(m[1]), _p(m[2]), cap,
                                                _p(m_off), _p(m_len)))
        return [tuple(m[s][m_off[r]:m_off[r] + m_len[r]].tobytes().decode("latin-1") for s in range(3)) for r in range(n_reads)]

    def last_kernel_ms(self):
        ms, k = ctypes.c_float(0), ctypes.c_int(0)
        self._lib.elector_last_kernel_ms(self._ctx, ctypes.byref(ms), ctypes.byref(k))
        return ms.value, k.value
