// host_setup.hpp -- host-side preparation shared by the C-ABI and the CPU emulation test
// harness: which matrix class the kernels can run, the device symbol tables, and the
// per-thread scratch layout of a size class.
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "host_io.hpp"
#include "poa_kernel.cuh"
#include "poa_packed.cuh"

namespace elector {

struct ScoringSetup {
  SymbolTables tab;
  int match = 0, mismatch = 0, open = 0, ext = 0, maxabs = 0;
  bool generic_sub = false;
  bool packed_ok = false;  // the 16-bit packed kernels (poa_packed.cuh) are exact for this matrix
  std::string error;

  bool fail(const char *fmt, int a = 0, int b = 0, int c = 0) {
    char buf[256];
    snprintf(buf, sizeof buf, fmt, a, b, c);
    error = buf;
    return false;
  }

  // Supported class (DESIGN.md section 3): alphabet <= 32 symbols, identical x/y gap sets,
  // and an extension penalty that is flat over gap lengths 1..T+D, so that the reference's
  // 0..T+D+1 gap-length state (align_lpo_po2.c:224-249) collapses to "in a gap or not".
  bool analyse(const ScoreMatrix &m) {
    if (m.nsymbol <= 0 || m.nsymbol > 32) return fail("matrix alphabet has %d symbols; 1..32 supported", m.nsymbol);
    const int M = m.trunc_len + m.decay_len;
    if (M < 1) return fail("gap truncation+decay length must be >= 1");
    for (int i = 0; i <= M; ++i)
      if (m.pen_x[i] != m.pen_y[i]) return fail("GAP-PENALTIES-X differing from GAP-PENALTIES is not supported");
    for (int i = 2; i <= M; ++i)
      if (m.pen_x[i] != m.pen_x[1])
        return fail("gap extension penalty must be flat (A1 == A2 or decay length 0); got %d vs %d at length %d", m.pen_x[1], m.pen_x[i], i);
    open = m.pen_x[0];
    ext = m.pen_x[1];
    memset(&tab, 0, sizeof tab);
    bool reach[32] = {false};
    for (int b = 0; b < 256; ++b) {
      const int c = m.code_of(b);
      tab.code_lut[b] = (uint8_t)c;
      if (b) reach[c] = true;
    }
    for (int i = 0; i < m.nsymbol; ++i) tab.sym[i] = (uint8_t)m.symbol[i];
    maxabs = std::max(std::abs(open), std::abs(ext));
    for (int i = 0; i < m.nsymbol; ++i)
      for (int j = 0; j < m.nsymbol; ++j) {
        const int s = m.score[(size_t)i * m.nsymbol + j];
        if (s < -32000 || s > 32000) return fail("score %d out of range", s);
        tab.sub[i * 32 + j] = (int16_t)s;
        if (reach[i] && reach[j]) maxabs = std::max(maxabs, std::abs(s));
      }
    // uniform match/mismatch over the reachable symbols -> compare-select instead of a table
    bool uniform = true, have_d = false, have_o = false;
    int dval = 0, oval = 0;
    for (int i = 0; i < m.nsymbol && uniform; ++i)
      for (int j = 0; j < m.nsymbol && uniform; ++j) {
        if (!reach[i] || !reach[j]) continue;
        const int s = m.score[(size_t)i * m.nsymbol + j];
        if (i == j) { if (!have_d) { dval = s; have_d = true; } else if (s != dval) uniform = false; }
        else { if (!have_o) { oval = s; have_o = true; } else if (s != oval) uniform = false; }
      }
    generic_sub = !uniform;
    match = dval;
    mismatch = have_o ? oval : dval;
    // Packed class (poa_packed.cuh): match 0, mismatch in [-16, -1] (min.u16x2 of the letter difference), open >= ext > 0,
    // and every score a multiple of q >= open - ext.  Then "a match beats the gap" implies M - gap >= open - ext, which
    // makes s - pen(move) == max(M - open, gap - ext): one packed add-max instead of a select on the move.
    {
      auto gcd = [](int a, int b) { a = std::abs(a); b = std::abs(b); while (b) { const int t = a % b; a = b; b = t; } return a; };
      const int q = gcd(gcd(mismatch, open), ext);
      packed_ok = uniform && match == 0 && mismatch < 0 && mismatch >= -16 && ext > 0 && open >= ext && open - ext <= q;
    }
    return true;
  }

  // The small segments (every sequence <= kSmallMax, len(P1) < 4 kN1q) run the packed kernels: no score of a small window
  // leaves 16 bits.  The launcher's kernel choice (seg_kind), the cor-is-ref shortcut of the size sort and the CPU emulation
  // all ask this one question.
  bool small_packed() const { return packed_ok && (int64_t)maxabs * (kSmallMax + 4 * kN1q + 4) <= kPackedSpan; }
};

}  // namespace elector
