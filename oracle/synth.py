"""TEST INFRASTRUCTURE ONLY -- deterministic synthetic inputs for the POA path.

Two generators:
  * hard_windows(): adversarial window triplets (tiny alphabets => many score ties,
    high error rates, trimmed ends, `N` / `AAA` placeholders as the reference
    splitter emits them (src/split/Master_Splitter.cpp:139-154,417-423), IUPAC and
    other out-of-alphabet letters, mixed case, lengths 1..~500).
  * reads(): read-level triplets for the BASELINE.json configs (SURVEY.md 8d):
    reference = i.i.d. uniform ACGT, raw = reference with error events, corrected =
    the same events each kept with probability p_keep.
PRNG: splitmix64, so the streams are reproducible in C as well.
"""
import math
import os
import re

MASK = (1 << 64) - 1


class SplitMix64:
    def __init__(self, seed):
        self.s = seed & MASK

    def next(self):
        self.s = (self.s + 0x9E3779B97F4A7C15) & MASK
        z = self.s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK
        return z ^ (z >> 31)

    def below(self, n):
        return self.next() % n

    def unit(self):
        return (self.next() >> 11) / float(1 << 53)


def mutate(rng, seq, rate, alphabet, ins=1, dele=1, sub=1):
    out = []
    tot = ins + dele + sub
    for ch in seq:
        if rng.unit() < rate:
            k = rng.below(tot)
            if k < ins:
                out.append(alphabet[rng.below(len(alphabet))])
                out.append(ch)
            elif k < ins + dele:
                pass
            else:
                out.append(alphabet[rng.below(len(alphabet))])
        else:
            out.append(ch)
    return "".join(out)


def hard_windows(n, seed=7):
    """returns list of (name, ref, cor, unc)"""
    rng = SplitMix64(seed)
    wins = []
    alphabets = ["ACGT", "AC", "A", "ACGTN", "acgt", "ACG"]
    for i in range(n):
        ab = alphabets[rng.below(len(alphabets))]
        mode = rng.below(12)
        if mode == 0:
            L = 1 + rng.below(6)
        elif mode == 1:
            L = 100 + rng.below(400)
        else:
            L = 8 + rng.below(90)
        ref = "".join(ab[rng.below(len(ab))] for _ in range(L))
        er_u = [0.01, 0.1, 0.2, 0.3][rng.below(4)]
        er_c = [0.0, 0.01, 0.05, 0.3][rng.below(4)]
        unc = mutate(rng, ref, er_u, ab) or ab[0]
        cor = mutate(rng, ref, er_c, ab) or ab[0]
        t = rng.below(16)
        if t == 0:
            cor = "N"
        elif t == 1:
            cor = cor[: max(1, len(cor) // 3)]
        elif t == 2:
            cor = cor[len(cor) // 2:] or "N"
        elif t == 3:
            ref, cor, unc = "AAA", "AAA", "AAA"
        elif t == 4:
            unc = unc[: max(1, len(unc) // 4)]
        elif t == 5:  # out-of-alphabet letters and mixed case
            extra = "RYKMSWBDHVN?]-x"
            l = list(cor)
            for _ in range(1 + rng.below(4)):
                l[rng.below(len(l))] = extra[rng.below(len(extra))]
            cor = "".join(l)
            unc = "".join(c.lower() if rng.below(2) else c for c in unc)
        elif t == 6:  # unrelated sequences
            cor = "".join(ab[rng.below(len(ab))] for _ in range(1 + rng.below(60)))
        elif t == 7:
            unc = "".join(ab[rng.below(len(ab))] for _ in range(1 + rng.below(60)))
        wins.append(("w%d" % i, ref, cor, unc))
    return wins


def write_windows(wins, prefix, titles=False):
    """writes prefix.ref.fa / .cor.fa / .unc.fa in the shard format of the splitter"""
    with open(prefix + ".ref.fa", "w") as fr, open(prefix + ".cor.fa", "w") as fc, open(prefix + ".unc.fa", "w") as fu:
        for k, (name, r, c, u) in enumerate(wins):
            h = ">" + name + (" some title %d" % k if titles and k % 3 == 0 else "")
            fr.write(h + "\n" + r + "\n")
            fc.write(h + "\n" + c + "\n")
            fu.write(h + "\n" + u + "\n")


def reads(n, length_fn, seed, raw_rate=0.10, keep=0.1, ratios=(1, 1, 1), homopolymer_del_bias=False):
    """read-level triplets: yields (name, ref, raw, corrected)."""
    rng = SplitMix64(seed)
    ab = "ACGT"
    ins, dele, sub = ratios
    tot = ins + dele + sub
    for i in range(n):
        L = length_fn(rng)
        ref = [ab[rng.next() & 3] for _ in range(L)]
        raw = []
        cor = []
        prev = ""
        for ch in ref:
            rate = raw_rate
            if homopolymer_del_bias and ch == prev:
                rate = min(0.9, raw_rate * 1.5)
            prev = ch
            if rng.unit() < rate:
                k = rng.below(tot)
                kept = rng.unit() < keep
                if k < ins:
                    b = ab[rng.next() & 3]
                    raw.append(b); raw.append(ch)
                    if kept:
                        cor.append(b)
                    cor.append(ch)
                elif k < ins + dele:
                    if not kept:
                        cor.append(ch)
                else:
                    b = ab[rng.next() & 3]
                    raw.append(b)
                    cor.append(b if kept else ch)
            else:
                raw.append(ch)
                cor.append(ch)
        yield ("read_%d" % i, "".join(ref), "".join(raw), "".join(cor))


def loguniform(lo, hi):
    return lambda rng: int(math.exp(math.log(lo) + rng.unit() * (math.log(hi) - math.log(lo))))


def random_msa_rows(n, seed=21):
    """gap-rich random 3-row MSAs (ref, corrected, uncorrected) for the tally: long '.' runs at the
    borders (trimmed / extended reads), gap stretches inside, 'n' never present (Donatello drops
    those columns).  Returns list of (R, C, U) strings of equal length."""
    rng = SplitMix64(seed)
    out = []
    for _ in range(n):
        L = 11 + rng.below(400) if rng.below(8) else 1 + rng.below(14)
        rows = []
        base = [("acgt")[rng.below(4)] for _ in range(L)]
        for k in range(3):
            row = []
            p_gap = [0.02, 0.05, 0.15][rng.below(3)]
            p_mut = [0.0, 0.02, 0.2][rng.below(3)]
            i = 0
            while i < L:
                if rng.unit() < p_gap / 4:
                    run = 1 + rng.below([3, 8, 30, 60][rng.below(4)])
                    row.extend("." * min(run, L - i))
                    i += min(run, L - i)
                else:
                    row.append("acgt"[rng.below(4)] if rng.unit() < p_mut else base[i])
                    i += 1
            # border effects
            t = rng.below(10)
            if t == 0:
                g = min(L, 3 + rng.below(40)); row[:g] = "." * g
            elif t == 1:
                g = min(L, 3 + rng.below(40)); row[L - g:] = "." * g
            elif t == 2:
                g = min(L // 2, 3 + rng.below(30)); row[:g] = "." * g; row[L - g:] = "." * g
            row = row[:L]
            if all(ch == "." for ch in row):  # the reference divides by the non-gap length
                row[rng.below(L)] = base[0]
            rows.append("".join(row))
        out.append((rows[0], rows[1], rows[2]))
    return out


def bubble_windows(n=6000, seed=20261018):
    """ELECTOR-like windows for the dual-frontier kernel (poa_dual.cuh): a corrected sequence with a few differences (bubbles
    that open and close at every position of a band, in the low and in the high half, back to back, at the first and at the
    last node; late starts and early ends of either sequence) against a noisier uncorrected one, lengths around the band
    sizes.  Returns list of (name, ref, cor, unc)."""
    rng = SplitMix64(seed)
    wins = []
    for i in range(n):
        L = [7, 8, 9, 15, 16, 17, 23, 24, 25, 31, 32, 33, 40, 48, 50, 55, 64, 65, 80, 100, 127][rng.below(21)]
        ref = "".join("ACGT"[rng.below(4)] for _ in range(L))
        cor = mutate(rng, ref, [0.01, 0.02, 0.05, 0.1, 0.2][rng.below(5)], "ACGT")
        t = rng.below(8)
        if t == 0:
            cor = cor[1 + rng.below(3):]                      # cor starts late: INITIAL node with the virtual link first
        elif t == 1:
            cor = cor[:max(1, len(cor) - 1 - rng.below(3))]   # cor ends early: several FINAL nodes
        elif t == 2:
            cor = "ACGT"[rng.below(4)] * (1 + rng.below(3)) + cor   # cor starts with an insertion
        unc = mutate(rng, ref, [0.05, 0.1, 0.2][rng.below(3)], "ACGT")
        wins.append(("b%d" % i, ref, cor or "A", unc or "C"))
    return wins


# ---- matrices beyond the shipped one ---------------------------------------------------------------------------------
# The shipped blosum80.mat has |mismatch| = open = 2 ext = 10, so a kernel that confuses these constants still computes the
# right numbers with it.  These matrices break the coincidences and walk the edges of the classes ScoringSetup::analyse
# (elector_b200/csrc/host_setup.hpp) tells apart.  Each entry: id, match, mismatch, GAP-PENALTIES (truncation 10, decay 5 as
# shipped; None: the non-uniform table matrix), and the class analyse must find: (packed_ok, generic_sub, maxabs,
# small_packed = the small windows run the 16-bit packed kernels).
MATRICES = [
    ("ties", 0, -1, (1, 1, 1), (1, 0, 1, 1)),         # ties everywhere; band span capped at kBandMaxSpan
    ("q3", 0, -3, (9, 6, 6), (1, 0, 9, 1)),           # |mismatch| < ext < open
    ("mis16", 0, -16, (8, 8, 8), (1, 0, 16, 1)),      # the min.u16x2 edge: a mismatch ties with an insertion plus a deletion
    ("max20", 0, -16, (20, 16, 16), (1, 0, 20, 1)),   # largest maxabs whose small windows stay packed (20 * 772 <= 16000)
    ("max21", 0, -7, (21, 21, 21), (1, 0, 21, 0)),    # packed class, but 21 * 772 > 16000: every window on the INT32 kernels
    ("pos2", 2, -3, (5, 2, 2), (0, 0, 5, 0)),         # uniform with a positive match: INT32 compare-select
    ("mis17", 0, -17, (10, 5, 5), (0, 0, 17, 0)),     # one step outside the packed class
    ("table", None, None, None, (0, 1, 7, 0)),        # non-uniform substitution table, other gap lengths
]


def matrix_text(mid):
    """the matrix file of MATRICES entry `mid`, in the reference's format"""
    from elector_b200.matrix import ALPHABET, default_matrix_text
    _, match, mismatch, gaps, _ = next(m for m in MATRICES if m[0] == mid)
    if gaps is not None:
        return default_matrix_text(match=match, mismatch=mismatch, gaps=gaps, trunc=10, decay=5)
    lines = ["GAP-TRUNCATION-LENGTH=4", "GAP-DECAY-LENGTH=0", "GAP-PENALTIES=7 3 3", "  " + " ".join(ALPHABET)]
    for i, a in enumerate(ALPHABET):
        lines.append(a + " " + " ".join(str(4 if i == j else -((i * 7 + j * 3) % 5) - 1) for j in range(len(ALPHABET))))
    return "\n".join(lines) + "\n"


# ---- windows at the edges of the device scheduler ---------------------------------------------------------------------
_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "elector_b200", "csrc")


def kernel_constants():
    """the size-class constants of the kernels, read from their headers, so that the edges follow the code"""
    out = {}
    for f in ("poa_kernel.cuh", "bin_kernel.cuh", "poa_packed.cuh"):
        for name, val in re.findall(r"constexpr int (k\w+) = (\d+);", open(os.path.join(_CSRC, f)).read()):
            out[name] = int(val)
    return out


def band_span_limit(maxabs, k=None):
    """poa_kernel.cuh band_span_limit: the diagonal band runs only for groups with len_x + len_y <= this"""
    k = k or kernel_constants()
    return min(k["kBandMaxScore"] // max(maxabs, 1) - 4, k["kBandMaxSpan"])


def window_measures(ref, cor, unc, n1=None):
    """what an edge tag may state about a window: lr, lc, lu, mx = max(lr, lc), sum = lr + lc, d = lu - lr, id = (cor is
    ref), and with len(P1) given n1 and span2 = n1 + lu"""
    m = dict(lr=len(ref), lc=len(cor), lu=len(unc), mx=max(len(ref), len(cor)), sum=len(ref) + len(cor),
             d=len(unc) - len(ref), id=int(ref == cor))
    if n1 is not None:
        m.update(n1=n1, span2=n1 + len(unc))
    return m


def parse_tag(tag):
    """'group k=v k=v' -> (group, {k: v})"""
    g, *kv = tag.split()
    return g, {k: int(v) for k, v in (x.split("=") for x in kv)}


def edge_windows(seed=5, maxabs=10):
    """Windows at the edges of the decisions only the device path makes: the phase-1 and phase-2 sort bins and big tiers
    (bin_kernel.cuh bin1_of, poa_kernel.cuh bin2_of), the cor-is-ref shortcut of the size sort and the d-classes of the
    linear bins, the band span limit of a matrix with this maxabs, lopsided shapes and the 16-bit node cap.  Returns a list
    of (tag, ref, cor, unc); a tag is 'group k=v ...' with the measures (window_measures) the window is built to have.  The
    last window, group 'toolarge', is one node beyond the cap: the library refuses it."""
    k = kernel_constants()
    S, Q4, NMAX = k["kSmallMax"], 4 * k["kN1q"], k["kMaxNodes"]
    rng = SplitMix64(seed)

    def rand(L, ab="ACGT"):
        return "".join(ab[rng.below(len(ab))] for _ in range(L))

    def fit(s, L, ab="ACGT"):          # exactly L letters
        s = s[:L]
        return s + rand(L - len(s), ab)

    def near(s, L, rate=0.03):         # L letters that align to s with a few differences
        return fit(mutate(rng, s, rate, "ACGT"), L)

    out = []

    def add(tag, ref, cor, unc):
        out.append((tag, ref, cor, unc))

    # phase 1: columns (cor) in 8-row half-bands, rows (ref) in len/2 quanta, big tiers beyond S
    for lc in (1, 8, 9, 64, 65, 128, 129, S, S + 1):
        for lr in (50, S):
            ref = rand(lr)
            add("p1 lr=%d lc=%d" % (lr, lc), ref, near(ref, lc), near(ref, lr, 0.1))
    for lr in (1, 2, S - 1, S, S + 1):
        for lc in (50, 1):
            ref = rand(lr)
            add("p1 lr=%d lc=%d" % (lr, lc), ref, near(ref, lc), near(ref, max(lr, 4), 0.1))
    for mx in (2 * S, 2 * S + 1, 4 * S, 4 * S + 1, 8 * S, 8 * S + 1):
        ref = rand(mx)
        add("p1big mx=%d lr=%d" % (mx, mx), ref, near(ref, mx - 7), near(ref, 200, 0.1))
        cor = rand(mx)
        add("p1big mx=%d lc=%d" % (mx, mx), near(cor, mx - 3), cor, near(cor, 300, 0.1))

    # phase 2: rows (unc) in half-bands, columns by len(P1)/4, big tiers when lu > S or len(P1) >= Q4.
    # len(P1) = lr + lc - (matched pairs): a shared stretch plus letters from disjoint alphabets sets it exactly.
    def p1_pair(n1, lr):
        sh = max(0, min(2, S - (n1 - lr)))           # up to two shared letters, as many as keep len(cor) <= S
        lc = n1 - lr + sh
        shared = rand(sh)
        return shared + rand(lr - len(shared), "AC"), shared + rand(lc - len(shared), "GT")

    lus = (1, 8, 9, 32, 33, 64, 65, 128, 129, S, S + 1)
    for lu in lus:
        ref = rand(48)
        cor = near(ref, 50)
        add("p2 lu=%d" % lu, ref, cor, near(ref, lu, 0.1))       # len(P1) about 50
        ref, cor = p1_pair(500, 250)
        add("p2 lu=%d n1=500" % lu, ref, cor, near(ref + cor, lu, 0.1))
    for n1 in (Q4 - 2, Q4 - 1, Q4, Q4 + 1):
        for lu in (8, 128, 129, S):
            ref, cor = p1_pair(n1, S + (n1 > 2 * S))
            add("p2q n1=%d lu=%d" % (n1, lu), ref, cor, near(cor + ref, lu, 0.1))

    # cor is ref: the shortcut needs lr == lc <= S and lu <= S; the linear bins sort d = lu - lr into four classes
    for lr in (1, 8, 9, 128, 129, S - 1, S, S + 1):
        for lu in (1, 128, 129, S, S + 1):
            ref = rand(lr)
            add("id lr=%d lu=%d id=1" % (lr, lu), ref, ref, near(ref, lu, 0.1))
    for d in (-40, -7, -6, -3, -2, 1, 2, 5, 6, 9, 10, 40):
        ref = rand(60)
        add("idd lr=60 d=%d id=1" % d, ref, ref, near(ref, 60 + d, 0.1))

    # the band span limit of this maxabs, and one above it: Phase1P (lr + lc) and Phase2L (cor is ref: len(P1) + lu)
    B = band_span_limit(maxabs, k)
    for span in (B, B + 1):
        ref = rand(B // 2)
        add("band1 sum=%d" % span, ref, near(ref, span - len(ref), 0.02), near(ref, len(ref), 0.1))
        ref = rand(B // 2)
        add("band2 span2=%d id=1" % span, ref, ref, near(ref, span - len(ref), 0.1))

    # lopsided shapes
    for lr in (S, S + 1, 3000):
        ref = rand(lr)
        add("asym lr=%d lc=1" % lr, ref, "N", near(ref, lr, 0.1))
    ref = rand(1)
    add("asym lr=1 lc=300", ref, rand(300), rand(40))
    ref, cor = p1_pair(500, 250)
    add("asym lu=1 n1=500", ref, cor, "A")
    for lr in (60, 100):
        ref = rand(lr)
        add("asym lr=%d lu=%d" % (lr, 4 * lr), ref, near(ref, lr), near(ref * 4, 4 * lr, 0.1))

    # caps: len(ref) + len(cor) == kMaxNodes in both orientations, the longest uncorrected sequence, one node too many
    big = rand(NMAX - 534)
    add("cap lr=%d lc=534 lu=64 sum=%d" % (NMAX - 534, NMAX), big, near(big[30000:30534], 534), near(big[30000:30064], 64, 0.1))
    big = rand(NMAX - 534)
    add("cap lr=534 lc=%d lu=64 sum=%d" % (NMAX - 534, NMAX), near(big[20000:20534], 534), big, near(big[20000:20064], 64, 0.1))
    ref = rand(50)
    add("cap lr=50 lc=50 lu=%d" % k["kMaxWindowLen"], ref, near(ref, 50), fit(ref * (k["kMaxWindowLen"] // 50 + 1), k["kMaxWindowLen"]))
    add("toolarge sum=%d" % (NMAX + 1), rand(NMAX - 533), rand(534), rand(64))
    return out


def letter_variants(win, n, seed):
    """n windows of the shape of `win` (name, ref, cor, unc): a permutation of ACGT over all three sequences and, from the second
    on, one substitution in the uncorrected one.  Lengths, cor-is-ref and which letters match stay what they were, so every
    variant lands in the sort bin of the original."""
    import itertools
    rng = SplitMix64(seed)
    perms = list(itertools.permutations("ACGT"))
    name, ref, cor, unc = win
    out = []
    for i in range(n):
        tr = str.maketrans("ACGT", "".join(perms[i % len(perms)]))
        u = unc.translate(tr)
        if i:
            p = rng.below(len(u))
            u = u[:p] + "ACGT"[rng.below(4)] + u[p + 1:]
        out.append(("%s v%d" % (name, i), ref.translate(tr), cor.translate(tr), u))
    return out


# ---- merged reads at the edges of the tally kernel ----------------------------------------------------------------------
def tally_constants():
    """the constants of the tally kernel (tally_kernel.cuh), so that the edges of tally_edge_reads follow the code"""
    src = open(os.path.join(_CSRC, "tally_kernel.cuh")).read()
    out = {name: int(val) for name, val in re.findall(r"constexpr int (k\w+) = (\d+);", src)}
    out.update((name, int(val)) for name, val in re.findall(r"\b(T_THRESH2?) = (\d+)", src))
    return out


def msa_background(rng, L, raw_rate=0.10, keep=0.1, max_run=3, max_crun=3):
    """three aligned rows (R, C, U) of L columns with the error profile of config 1: every reference base has an error in the
    uncorrected row with probability raw_rate (insertion, deletion or substitution), which the corrected row keeps with
    probability `keep`.  No row has a dot run longer than max_run (max_crun for the corrected row) and the first and last three
    columns are plain bases, so the background alone never reaches a border gap, a gap stretch or a cr threshold."""
    R, C, U = [], [], []
    while len(R) < L:
        b = "ACGT"[rng.below(4)]
        if rng.unit() < raw_rate:
            k, kept, x = rng.below(3), rng.unit() < keep, "ACGT"[rng.below(4)]
            if k == 0:
                cols = [(".", x if kept else ".", x), (b, b, b)]
            elif k == 1:
                cols = [(b, "." if kept else b, ".")]
            else:
                cols = [(b, x if kept else b, x)]
        else:
            cols = [(b, b, b)]
        for r, c, u in cols:
            R.append(r); C.append(c); U.append(u)
    R, C, U = R[:L], C[:L], U[:L]
    run = [0, 0, 0]
    for i in range(L):
        run = [run[s] + 1 if row[i] == "." else 0 for s, row in enumerate((R, C, U))]
        if i < 3 or i >= L - 3 or max(run[0], run[2]) > max_run or run[1] > max_crun:
            R[i] = C[i] = U[i] = "ACGT"[rng.below(4)]
            run = [0, 0, 0]
    return R, C, U


def gap_counters(C, R):
    """(cg, cr) of findGapStretches (computeStats.py:104-189) after every column: the corrected-gap run and the reference-gap
    counter that advances only while the previous corrected column is a gap"""
    cg = cr = 0
    prev, out = None, []
    for c, r in zip(C, R):
        if prev == ".":
            if c == ".":
                cg = cg + 1 if cg > 0 else 2
            if r == ".":
                cr = cr + 1 if cr > 0 else 2
        if prev is None:
            cg, cr = cg + (c == "."), cr + (r == ".")
        if c != ".":
            cg = 0
        if r != ".":
            cr = 0
        out.append((cg, cr))
        prev = c
    return out


def _runs(row):
    out, i = set(), 0
    while i < len(row):
        if row[i] == ".":
            j = i
            while j + 1 < len(row) and row[j + 1] == ".":
                j += 1
            out.add("%d-%d" % (i, j))
            i = j + 1
        else:
            i += 1
    return out


def tally_measures(R, C, U):
    """what a tally edge tag may state about a merged read (values as strings): L, assessed, gl / gr (and per row glr, glu,
    grr, gru), ext (extended), nk and keys (the sorted gap stretches, 'a-b,...' or 'none'), crun / rrun (maximal dot runs of
    the corrected / reference row: a tag lists some of them), crmax (largest cr on a column where cg >= T_THRESH), dots2 /
    dots3 (columns where exactly two / all three rows are dots), iupac (R or U holds a letter outside ACGTacgt), lower (R or C
    holds g or c)"""
    from oracle import tally_oracle as to
    T = tally_constants()["T_THRESH"]
    m = dict(L=len(R), assessed=int(len(R) > 10), glr=to.nb_left_gaps(R), glu=to.nb_left_gaps(U), grr=to.nb_right_gaps(R),
             gru=to.nb_right_gaps(U), ext=to.tally_read(R, C, U)["extended"])
    m["gl"], m["gr"] = min(m["glr"], m["glu"]), min(m["grr"], m["gru"])
    keys = sorted(to.gap_stretch_keys(C, R))
    m["nk"], m["keys"] = len(keys), ",".join("%d-%d" % k for k in keys) or "none"
    m["crmax"] = max([cr for cg, cr in gap_counters(C, R) if cg >= T], default=0)
    ndots = [(r == ".") + (c == ".") + (u == ".") for r, c, u in zip(R, C, U)]
    m["dots2"], m["dots3"] = ndots.count(2), ndots.count(3)
    m["iupac"] = int(any(ch not in "ACGTacgt." for ch in R + U))
    m["lower"] = int(any(ch in "gc" for ch in R + C))
    m = {k: str(v) for k, v in m.items()}
    m["crun"], m["rrun"] = _runs(C), _runs(R)
    return m


def tally_tag_mismatches(tag, R, C, U):
    """the (key, stated, measured) triples of a tally edge tag that the read does not have"""
    m = tally_measures(R, C, U)
    bad = []
    for kv in tag.split()[1:]:          # the first word names the shape
        k, v = kv.split("=")
        if k in ("crun", "rrun"):
            bad += [(k, r, "absent") for r in v.split(",") if r not in m[k]]
        elif m[k] != v:
            bad.append((k, v, m[k]))
    return bad


def _tally_shapes():
    """(tag, L, segments, max_crun) of every tally edge read; a segment (pos, n, R, C, U) sets n columns from pos, each row
    given as one character for all n columns or as n characters: 'b' is the column's base (the same in every row that has 'b'),
    anything else is taken as it is.  Two plain columns on either side of each segment keep it apart from the background."""
    k = tally_constants()
    T, T2, S = k["T_THRESH"], k["T_THRESH2"], k["kSmemCols"]
    STEP = 32 * 32                     # next_pair_warp: 32 lanes, one 32-column word each
    out = []

    def add(tag, L, segs, max_crun=3):
        out.append((tag, L, segs, max_crun))

    def dots(s, n):                    # n characters, dots at the offsets in s
        return "".join("." if i in s else "b" for i in range(n))

    # lengths: not assessed / assessed, 16-column groups, 32-column words, 1 024-column steps, the shared-memory bitmasks
    for L in (10, 11, 15, 16, 17, 31, 32, 33, 1023, 1024, 1025, 2049, S - 1, S, S + 1, 65537, 150001):
        sparse = 1 if L > S else 3     # long reads: no counting run of the corrected row but the ones placed here
        add("len L=%d nk=0" % L, L, [], sparse)
        if L <= 10:
            continue
        if L < 64:
            add("lenb L=%d gl=%d gr=%d" % (L, T, T + 1), L, [(0, T, ".", "b", "."), (L - T, T, ".", "b", ".")])
            if L > 30:
                add("lenk L=%d keys=0-%d crun=2-%d" % (L, L - 1, L - 3), L, [(2, L - 4, "b", ".", "b")])
            continue
        segs = [(0, T, ".", "b", "."), (8, 33, "b", ".", "b"), (L - 40, 31, "b", ".", "b"), (L - 6, 6, ".", "b", ".")]
        crun = ["8-40", "%d-%d" % (L - 40, L - 10)]
        for j in range(1, min(L // STEP, 4) + 1):
            if 100 < j * STEP < L - 100:
                segs.append((j * STEP - 1, 2, "b", ".", "b")); crun.append("%d-%d" % (j * STEP - 1, j * STEP))
        if L > S + 100:
            segs.append((S - 1, 2, "b", ".", "b")); crun.append("%d-%d" % (S - 1, S))
        add("lenb L=%d gl=%d gr=7 keys=0-40,%d-%d crun=%s" % (L, T, L - 40, L - 1, ",".join(crun)), L, segs, sparse)

    # border gaps (nbLeftGaps / nbRightGaps and the extension): L = 400
    L = 400
    for n in (T - 1, T, T2 - 1, T2, T2 + 1):
        g = n if n >= T else 0
        add("bordl:n%d gl=%d ext=%d" % (n, g, g if g >= T2 else -1), L, [(0, n, ".", "b", ".")])
        add("bordr:n%d gr=%d ext=%d" % (n, g + (g > 0), g + 1 if g + 1 >= T2 else -1), L, [(L - n, n, ".", "b", ".")])
    for sep in (T, T + 1):             # two runs of T dots, sep bases apart: the second counts only while nt <= T
        g = 2 * T + sep if sep == T else T
        add("bordsepl:sep%d gl=%d" % (sep, g), L, [(0, T, ".", "b", "."), (T + sep, T, ".", "b", ".")])
        add("bordsepr:sep%d gr=%d" % (sep, g + 1), L, [(L - T, T, ".", "b", "."), (L - 2 * T - sep, T, ".", "b", ".")])
    add("bordw gl=40 gr=36 ext=76", L, [(0, 40, ".", "b", "."), (L - 35, 35, ".", "b", ".")])        # runs across a word
    add("bordmin glr=20 glu=7 gl=7 grr=7 gru=26 gr=7", L, [(0, 20, ".", "b", dots(range(7), 20)), (L - 25, 25, dots(range(19, 25), 25), "b", ".")])
    add("bordmin glr=6 glu=25 gl=6 grr=23 gru=10 gr=10 ext=-1", L, [(0, 25, dots(range(6), 25), "b", "."), (L - 22, 22, ".", "b", dots(range(13, 22), 22))])
    # extension with corrected dots inside; on the right the count starts one column after L - gr (computeStats.py:490)
    add("borde gl=25 gr=25 ext=45 dots3=5", L, [(0, 25, ".", dots({3, 4, 10}, 25), "."), (L - 25, 25, "b" + "." * 24, dots({0, 1, 24}, 25), "b" + "." * 24)])

    # runs of the corrected row (find_gap_stretches / next_pair_warp): a stretch's first column shows in a key (a, L-1) when it
    # ends within T2 columns of the right border, its last column in a key (0, b) when it starts within T2 of the left one
    for a in (31, 32, 95, 96, STEP - 1, STEP, 2 * STEP - 1, 2 * STEP):
        L = a + 40
        add("crunr:a%d keys=%d-%d crun=%d-%d" % (a, a, L - 1, a, a + 30), L, [(a, 31, "b", ".", "b")], 1)
    for b in (31, 32, 63, 64, STEP - 1, STEP, 2 * STEP - 1, 2 * STEP):
        add("crunl:b%d keys=0-%d crun=8-%d" % (b, b, b), b + 200, [(8, b - 7, "b", ".", "b")], 1)
    # the scan resumes after a 2-dot run at column 37, so the warp's steps start at word 1: a pair across the last word of one
    add("crunstep keys=%d-%d crun=37-38,%d-%d" % (STEP + 31, STEP + 54, STEP + 31, STEP + 35), STEP + 55,
        [(37, 2, "b", ".", "b"), (STEP + 31, 5, "b", ".", "b"), (STEP + 39, 12, "b", ".", "b")], 1)
    # runs of 1 (column 0 and elsewhere), 2, 4, 5, 6 dots; a pair whose second dot opens a word; a run of n dots ends 4 bases
    # before a stretch that reaches the right border: n >= T makes it a stretch of its own that the pending merge joins
    for n in (1, 2, T - 1, T, T + 1):
        L = 300
        segs = [(0, 1, "b", ".", "b"), (50, 1, "b", ".", "b"), (63, 2, "b", ".", "b"), (100, 2, "b", ".", "b"), (110, 4, "b", ".", "b"),
                (L - 45, n, "b", ".", "b"), (L - 45 + n + 3, 45 - n - 3 - 8, "b", ".", "b")]
        ka = L - 45 if n >= T else L - 45 + n + 3
        add("crunk:n%d keys=%d-%d crun=0-0,50-50,63-64,100-101,110-113,%d-%d" % (n, ka, L - 1, L - 45, L - 45 + n - 1), L, segs, 1)

    # reference-gap runs (cr): inside a stretch of the corrected row, before it (sr < st, with and without corrected dots in
    # between), from column 0, and words of a stretch without reference dots next to words with them
    for n in (T2 - 2, T2 - 1, T2, T2 + 1, T2 + 2):
        add("cr:n%d crmax=%d keys=0-%d" % (n, n, 8 + min(n, T2 - 1) - 1), 200, [(8, n, ".", ".", "b")], 1)
    add("crsr:k0 keys=0-28 crmax=31", 200, [(3, 48, ".", dots(range(7, 38), 48), "b")], 1)            # R dots from 3, C run 10..40
    add("crsr:k1 keys=0-27 crmax=32", 200, [(3, 48, ".", dots({2} | set(range(7, 38)), 48), "b")], 1)
    add("crsr:k1dot keys=0-27 crmax=32 rrun=3-50", 200, [(2, 49, "b" + "." * 48, dots({0} | set(range(8, 39)), 49), "b")], 1)   # the dot before sr
    add("crs0:k0 keys=0-28 rrun=0-50 crmax=31", 200, [(0, 51, ".", dots(range(10, 41), 51), "b")], 1)
    add("crs0:k1 keys=0-27 rrun=0-50 crmax=32", 200, [(0, 51, ".", dots({0} | set(range(10, 41)), 51), "b")], 1)
    # 15 single corrected dots inside the reference gap before the stretch: cr starts at 16 and no column qualifies until the
    # reference gap ends
    pre = set(range(2, 32, 2))
    add("crpre keys=167-204 crun=150-190 rrun=100-170", 205,
        [(100, 91, "." * 71 + "b" * 20, dots(pre | set(range(50, 91)), 91), "b")], 1)
    add("crrb keys=0-167 crun=8-220 rrun=8-40,150-221", 300, [(8, 214, dots(set(range(33)) | set(range(142, 214)), 214), dots(range(213), 214), "b")], 1)
    add("crrb keys=0-117 crun=8-300 rrun=100-301", 400, [(8, 294, dots(range(92, 294), 294), dots(range(293), 294), "b")], 1)

    # stretches within T2 of a border, pending stretches T and T + 1 apart, overlapping keys, the most keys a read can have
    for a in (T2, T2 + 1):
        add("slotl:a%d keys=%s" % (a, "0-%d" % (a + 30) if a <= T2 else "none"), 300, [(a, 31, "b", ".", "b")], 1)
    for d in (T2, T2 + 1):
        L = 300
        add("slotr:d%d keys=%s" % (d, "%d-%d" % (L - 60, L - 1) if d <= T2 else "none"), L, [(L - 60, 61 - d, "b", ".", "b")], 1)
    for g in (T, T + 1):
        L = 300
        ka = L - 60 if g <= T else L - 45 + g
        add("slotp:g%d keys=%d-%d" % (g, ka, L - 1), L, [(L - 60, 16, "b", ".", "b"), (L - 45 + g, 45 - g - 9, "b", ".", "b")], 1)
    for L, r in ((200, (130, 150, 170)), (433, (370, 390, 410))):
        # key 0 from a stretch at the left border; a stretch in the middle whose pending merge with the stretch that reaches the
        # right border keeps its start; that stretch's own key once a last stretch inside the border merges with it
        segs = [(3, 28, "b", ".", "b"), (L - 100, 21, "b", ".", "b"), (L - 76, 67, dots({x - (L - 76) for x in r}, 67), ".", "b"),
                (L - 7, 5, "b", ".", "b")]
        add("keys3 nk=3 keys=0-30,%d-%d,%d-%d" % (L - 100, L - 1, L - 76, L - 1), L, segs, 1)

    # classification: case, N and IUPAC letters, columns with two or three dots
    add("cls iupac=1 lower=1 dots3=1", 600,
        [(100, 16, "gGcCaAtTNRYKMSWn", "gGcCaAtTgcGCacgt", "GgCcNnRYKMSWBDHV"), (200, 1, ".", ".", "."), (210, 1, ".", ".", "b"),
         (220, 1, ".", "b", "."), (230, 1, "b", ".", "."), (300, 8, "NnRYacgt", "cCgGacgt", "gcGCNnKM")])
    # mask ends (gapsLeft, L - gapsRight, both ends of a key) at every offset inside a 16-column group
    for i in range(16):
        L, gl, gr = 700 + i, T + i, T + 1 + (2 * i) % 16   # a right run of n dots is gr = n + 1
        b = 40 + i
        segs = [(0, b + 1, "." * gl + "b" * (b + 1 - gl), "b" * 6 + "." * (b - 5), "." * gl + "b" * (b + 1 - gl)),
                (L - 45, 45, "b" * (46 - gr) + "." * (gr - 1), "." * 43 + "bb", "b" * (46 - gr) + "." * (gr - 1))]
        add("mask:i%d gl=%d gr=%d keys=0-%d,%d-%d" % (i, gl, gr, b, L - 45, L - 1), L, segs, 1)
    return out


def tally_edge_reads(seed=11, copies=3):
    """Merged reads (tag, R, C, U) at the edges of the tally kernel (tally_kernel.cuh): three rows of equal length without
    'n' in C, as the merge leaves them.  Each shape of _tally_shapes comes in `copies` copies on different config-1
    backgrounds (msa_background); its tag is 'group k=v ...' with measures tally_measures must find.

    The most gap stretches (keys) a read can have is 3, below kMaxStretchKeys: a key other than 0 ends at L - 1, so it comes
    from a pending entry merged into (or being) the first entry that ends at L - 1, i.e. the first stretch ending within T2
    of the right border; every later stretch starts inside the border and is too short for a key.  Key 0 is the third
    (group keys3 has all three), so the overflow branch of the kernel is dead code."""
    out = []
    for c in range(copies):
        rng = SplitMix64(seed * 1000003 + c)
        for tag, L, segs, max_crun in _tally_shapes():
            R, C, U = msa_background(rng, L, max_crun=max_crun)
            for pos, n, *_ in segs:                  # plain columns around every segment first, then the segments
                for i in list(range(pos - 2, pos)) + list(range(pos + n, pos + n + 2)):
                    if 0 <= i < L:
                        R[i] = C[i] = U[i] = "ACGT"[rng.below(4)]
            for pos, n, *rows in segs:
                rows = [r * n if len(r) == 1 else r for r in rows]
                assert all(len(r) == n for r in rows) and pos + n <= L, (tag, pos, n)
                for i in range(n):
                    b = "ACGT"[rng.below(4)]
                    for row, ch in zip((R, C, U), (r[i] for r in rows)):
                        row[pos + i] = b if ch == "b" else ch
            out.append((tag, "".join(R), "".join(C), "".join(U)))
    return out
