// TEST INFRASTRUCTURE ONLY -- runs the per-window device code (Phase1 / Phase2 ::run_window in
// elector_b200/csrc/poa_kernel.cuh, compiled as host code) on the CPU, so that the
// kernel's algorithmic restructuring (8-row register bands, two frontier sets, 2-bit
// moves, fused emit) can be checked against the oracle in the GPU-less container.
// It is never linked into the product library; the product has no CPU path.
//
// usage: poa_emul MATRIX|- REF.fa COR.fa UNC.fa OUT.pir [OUT.scores|-] [packed|dual-general|coop]
// packed: windows the library would run through the 16-bit packed kernels (poa_packed.cuh) do so here too
// stderr, first line: the matrix class ScoringSetup::analyse found
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../elector_b200/csrc/host_setup.hpp"
#include "../../elector_b200/csrc/bin_kernel.cuh"
#include "../../elector_b200/csrc/poa_packed.cuh"
#include "../../elector_b200/csrc/poa_coop.cuh"
#include "../../elector_b200/csrc/poa_dual.cuh"

using namespace elector;

// fast part of a window's layout: a separate "arena" for every other window, global scratch at o_fast for the rest
// (both placements of the library are exercised)
struct FastPart {
  std::vector<uint32_t> arena;
  template <class L>
  uint32_t *base(const L &layout, uint32_t *lane_scratch, int lane, size_t w) {
    if (w % 2 == 0) { arena.assign((size_t)layout.f_total * 32 + 32, 0xdeadbeefu); return arena.data() + lane; }
    return lane_scratch + (size_t)layout.o_fast * 32;
  }
};

template <bool GS>
static int run(const ScoringSetup &sc, FastaFile &R, FastaFile &C, FastaFile &U, FILE *pir, FILE *scores, bool packed, bool general_only, bool coop, bool dual) {
  long n_packed1 = 0, n_packed2 = 0, n_linear2 = 0, n_ident1 = 0, n_band_retry = 0;
  const int band_w = packed ? (getenv("ELECTOR_BAND_W") ? atoi(getenv("ELECTOR_BAND_W")) : 10) : 0;   // diagonal band of the packed linear kernels
  const size_t n = std::min(R.rec.size(), std::min(C.rec.size(), U.rec.size()));
  for (size_t w = 0; w < n; ++w) {
    const int lr = R.rec[w].len, lc = C.rec[w].len, lu = U.rec[w].len;
    const int lane = (int)(w % 32);
    const uint8_t *ref = (const uint8_t *)R.seq.data() + R.rec[w].off, *cor = (const uint8_t *)C.seq.data() + C.rec[w].off,
                  *unc = (const uint8_t *)U.seq.data() + U.rec[w].off;
    Scoring s;
    s.tab = &sc.tab; s.set(sc.match, sc.mismatch, sc.open, sc.ext);
    FastPart fp;
    // ---- phase 1 (caps deliberately larger than the window, as in a real group) ----
    std::vector<uint64_t> nodes64(((size_t)lr + lc) / 4 + 2, 0xdeaddeaddeaddeadull);
    uint16_t *nodes_p = reinterpret_cast<uint16_t *>(nodes64.data());
    int s1, spcode, n1;
    bool ident = false;   // cor is ref: no phase 1, phase 2 in the linear segments
    const int cap_r = lr + (int)(w % 3), cap_c = lc + (int)(w % 5);
    if (coop) {   // phase 1 through the warp-cooperative wavefront (lin(ref) as a node list)
      LayoutC1 L1;
      make_layout_c1(L1, cap_r, cap_c);
      std::vector<uint32_t> scratch1((size_t)L1.total * 32, 0xdeadbeefu);
      std::vector<uint32_t> bset((size_t)2 * kSlotWords, 0xdeadbeefu);
      Phase2<GS> p1;
      p1.scr.base = scratch1.data() + lane;
      p1.fs.base = p1.scr.base + (size_t)L1.l2.o_fast * 32;
      p1.bset = bset.data() + lane;
      p1.sc = s;
      p1.Lp = &L1.l2;
      coop1_before<GS>(p1, L1, ref, lr, cor, lc, nodes_p);
      int bj = -1;
      coop_dp_emulated<GS>(p1, bset.data(), lr, lc, s1, bj);
      n1 = coop1_after<GS>(p1, L1, lr, lc, bj, nodes_p, spcode);
    } else if (packed && !general_only && sc.small_packed() && lr == lc && lr <= kSmallMax && lu <= kSmallMax && memcmp(ref, cor, (size_t)lr) == 0) {
      // cor is ref: the size sort of the library (bin1_count_kernel) skips phase 1 -- P1 = lin(ref), every node carries both letters
      n1 = lr; s1 = 0; spcode = 0;
      ident = true;
      ++n_ident1;
    } else if (packed && sc.small_packed() && std::max(lr, lc) <= kSmallMax) {   // a small segment of the library (bin1_of)
      Layout1P L1;
      make_layout1p(L1, cap_r, cap_c);
      std::vector<uint32_t> scratch1((size_t)L1.total * 32, 0xdeadbeefu);
      Phase1P p1;
      p1.scr.base = scratch1.data() + lane;
      p1.fs.base = fp.base(L1, p1.scr.base, lane, w);
      p1.sc = s;
      p1.Lp = &L1;
      bool exact = true;
      if (band_w > 0 && cap_r + cap_c <= band_span_limit(sc.maxabs)) {   // diagonal band with the exactness test; run again without it when the test fails
        const int d = lc - lr;
        p1.bw = BandW{(d < 0 ? d : 0) - band_w - (int)((w * 7) % 13), (d > 0 ? d : 0) + band_w + (int)((w * 5) % 11), band_w, true};   // the union band of a warp: a superset of the window's own by what other lanes add
      }
      n1 = p1.run_window(ref, lr, cor, lc, nodes_p, s1, spcode, exact);
      if (!exact) {
        ++n_band_retry;
        p1.bw.on = false;
        n1 = p1.run_window(ref, lr, cor, lc, nodes_p, s1, spcode, exact);
      }
      ++n_packed1;
    } else {
      Layout1 L1;
      make_layout1(L1, cap_r, cap_c);
      std::vector<uint32_t> scratch1((size_t)L1.total * 32, 0xdeadbeefu);
      Phase1<GS> p1;
      p1.scr.base = scratch1.data() + lane;
      p1.fs.base = fp.base(L1, p1.scr.base, lane, w + 1);
      p1.sc = s;
      p1.Lp = &L1;
      bool exact;
      n1 = p1.run_window(ref, lr, cor, lc, nodes_p, s1, spcode, exact);
    }
    int bin, seg;
    bin2_of(n1, lu, spcode, ident, bin, seg);
    if (bin < 0 || bin >= kNumBins2 || seg < 0 || seg >= kNumSegs2) { fprintf(stderr, "bad phase-2 bin\n"); return 1; }
    // ---- phase 2 ----
    const int cap_n = n1 + (int)(w % 4), cap_u = lu + (int)(w % 2);
    int s2, nring, nring_emitted;
    // the three MSA rows go straight to their place (here: three word arrays), 4 letters per word
    const uint32_t row_words = (uint32_t)(n1 + lu) / 4 + 2;
    std::vector<uint32_t> rows((size_t)3 * row_words, 0xdeadbeefu);
    RowSink sink{rows.data(), rows.data() + row_words, rows.data() + 2 * row_words};
    const bool fits16 = packed && sc.small_packed() && seg >= kBigTiers;   // a small segment of the library (bin2_of)
    if (coop) {   // the warp-cooperative DP2 of poa_coop.cuh (32 lanes emulated one after the other), serial steps of Phase2
      Layout2 L2;
      make_layout2(L2, cap_n, cap_u);
      std::vector<uint32_t> scratch2((size_t)L2.total * 32, 0xdeadbeefu);
      std::vector<uint32_t> bset((size_t)2 * kSlotWords, 0xdeadbeefu);
      Phase2<GS> p2;
      p2.scr.base = scratch2.data() + lane;
      p2.fs.base = p2.scr.base + (size_t)L2.o_fast * 32;
      p2.bset = bset.data() + lane;
      p2.sc = s;
      p2.Lp = &L2;
      p2.fs.pack_codes(s.tab, unc, lu, L2.f_unc);
      const int nrings = p2.prepare(nodes_p, n1);
      int bj = -1;
      coop_dp_emulated<GS>(p2, bset.data(), n1, lu, s2, bj);
      AlignBits al = p2.bits();
      p2.traceback(n1, lu, bj, al);
      nring = columns_of(nrings, lu, al.nmatch);
      nring_emitted = p2.fuse_emit(al, n1, lu, sink);
    } else if (fits16 && seg >= kFirstLinSeg2 && !general_only) {     // P1 linear: the library runs Phase2L
      Layout2L L2;
      make_layout2l(L2, cap_n, cap_u);
      std::vector<uint32_t> scratch2((size_t)L2.total * 32, 0xdeadbeefu);
      Phase2L p2;
      p2.scr.base = scratch2.data() + lane;
      p2.fs.base = fp.base(L2, p2.scr.base, lane, w);
      p2.bset = nullptr;
      p2.sc = s;
      p2.Lp = &L2;
      bool exact = true;
      if (band_w > 0 && cap_n + cap_u <= band_span_limit(sc.maxabs)) {
        const int d = lu - n1;
        p2.bw = BandW{(d < 0 ? d : 0) - band_w - (int)((w * 3) % 7), (d > 0 ? d : 0) + band_w + (int)((w * 5) % 9), band_w, true};   // union band of a warp
      }
      AlignBits al = p2.bits();
      nring = p2.align_linear(ref, n1, unc, lu, s2, exact, al);
      if (!exact) {
        ++n_band_retry;
        p2.bw.on = false;
        al = p2.bits();
        nring = p2.align_linear(ref, n1, unc, lu, s2, exact, al);
      }
      nring_emitted = p2.fuse_emit(al, n1, lu, sink);
      ++n_linear2;
    } else if (fits16 && dual) {   // general windows: the dual-frontier packed kernel (poa_dual.cuh), as the library runs them
      Layout2 L2;
      make_layout2(L2, cap_n, cap_u);
      std::vector<uint32_t> scratch2((size_t)L2.total * 32, 0xdeadbeefu);
      Phase2D p2;
      p2.scr.base = scratch2.data() + lane;
      p2.fs.base = fp.base(L2, p2.scr.base, lane, w);
      p2.bset = nullptr;
      p2.sc = s;
      p2.Lp = &L2;
      AlignBits al = p2.bits();
      nring = p2.align_window(nodes_p, n1, unc, lu, s2, al);
      nring_emitted = p2.fuse_emit(al, n1, lu, sink);
      ++n_packed2;
    } else {
      Layout2 L2;
      make_layout2(L2, cap_n, cap_u);
      std::vector<uint32_t> scratch2((size_t)L2.total * 32, 0xdeadbeefu);
      std::vector<uint32_t> bset((size_t)2 * kSlotWords, 0xdeadbeefu);
      Phase2<GS> p2;
      p2.scr.base = scratch2.data() + lane;
      p2.fs.base = fp.base(L2, p2.scr.base, lane, w + 1);
      p2.bset = bset.data() + lane;
      p2.sc = s;
      p2.Lp = &L2;
      AlignBits al = p2.bits();
      nring = p2.align_window(nodes_p, n1, unc, lu, s2, al);
      nring_emitted = p2.fuse_emit(al, n1, lu, sink);
    }
    if (nring != nring_emitted) { fprintf(stderr, "window %zu: %d columns announced, %d emitted\n", w, nring, nring_emitted); return 1; }
    const FastaRecord *recs[3] = {&R.rec[w], &C.rec[w], &U.rec[w]};
    for (int r = 0; r < 3; ++r) {
      fprintf(pir, ">%s %s\n", recs[r]->name.c_str(), recs[r]->title.c_str());
      for (int k = 0; k < nring; ++k) fputc((rows[r * row_words + (k >> 2)] >> ((k & 3) * 8)) & 0xff, pir);
      fputc('\n', pir);
    }
    if (scores) fprintf(scores, "%d %d %d %d\n", s1, s2, n1, nring);
  }
  if (packed) fprintf(stderr, "packed: %ld (phase 1) + %ld (phase 1, cor is ref), %ld (phase 2 general) and %ld (phase 2 linear) of %zu windows; band half-width %d, %ld DPs run again without the band\n", n_packed1, n_ident1, n_packed2, n_linear2, n, band_w, n_band_retry);
  return 0;
}

int main(int argc, char **argv) {
  if (argc < 6) { fprintf(stderr, "usage: %s MATRIX|- REF COR UNC OUT.pir [OUT.scores]\n", argv[0]); return 2; }
  ScoreMatrix m;
  if (std::string(argv[1]) == "-") m.set_default();
  else if (m.load(argv[1]) <= 0) { fprintf(stderr, "cannot read matrix\n"); return 1; }
  ScoringSetup sc;
  if (!sc.analyse(m)) { fprintf(stderr, "unsupported matrix: %s\n", sc.error.c_str()); return 3; }
  // the class the library's kernel choice starts from (capi.cu seg_kind)
  fprintf(stderr, "matrix class: packed_ok %d generic_sub %d maxabs %d small_packed %d\n", (int)sc.packed_ok, (int)sc.generic_sub, sc.maxabs, (int)sc.small_packed());
  FastaFile R, C, U;
  if (read_fasta_file(argv[3], C) < 0 || read_fasta_file(argv[4], U) < 0 || read_fasta_file(argv[2], R) < 0) return 1;
  FILE *pir = fopen(argv[5], "w");
  FILE *scores = argc > 6 && argv[6][0] != '-' ? fopen(argv[6], "w") : nullptr;
  if (!pir) return 1;
  const bool dual = argc > 7 && (std::string(argv[7]) == "packed" || std::string(argv[7]) == "dual-general");   // "packed" = what the library runs
  const bool packed = dual;
  const bool general_only = argc > 7 && std::string(argv[7]) == "dual-general";   // linear windows through the general kernel as well
  const bool coop = argc > 7 && std::string(argv[7]) == "coop";   // phase 2 of every window through the warp-cooperative DP
  const int rc = sc.generic_sub ? run<true>(sc, R, C, U, pir, scores, packed, general_only, coop, dual) : run<false>(sc, R, C, U, pir, scores, packed, general_only, coop, dual);
  fclose(pir);
  if (scores) fclose(scores);
  return rc;
}
