// poa_coop.cuh -- warp-cooperative DP2 for the LONG windows of a call.
//
// poa_kernel.cuh / poa_packed.cuh give one window to one thread.  That is the efficient mapping for the
// bulk (~50 x 50 cells), but a window of 200+ letters then is a serial chain of ~10^6 dependent integer
// instructions: one warp holding 32 such windows runs for milliseconds, long after the bulk of the call
// has finished (profiles/r1c_launches_packed.csv: the 32-warp launch of the longest windows takes 3.9 ms,
// the bulk of the same 650 k-window chunk 0.8 ms).  The longest windows therefore run here:
//
//   * a warp owns a small GROUP of windows (kCoopGroup, in lanes 0..kCoopGroup-1 of the lane-interleaved
//     scratch); the serial per-window steps (letter packing, node
//     preparation, traceback, fuse + MSA emit) stay thread-per-window and are the code of Phase2;
//   * the DP of each window of the group is computed by ALL 32 LANES: lane l owns rows 8l .. 8l+7 of a
//     256-row pass and runs ONE NODE BEHIND lane l-1 (a systolic wavefront over the columns).  What a band
//     of poa_kernel.cuh passes to the band below through the node records -- the node's shape, S and G of the
//     band's bottom row -- travels from lane to lane with __shfl_up_sync instead; the 2-bit moves of two
//     lanes (rows 0-7 and 8-15 of a 16-row band) are combined into the word the traceback of Phase2 expects.
//   * every lane keeps its own pair of frontier sets (8 rows each) exactly like a band of Phase2: which set
//     holds which frontier depends on the node shapes only, so lane l replays lane l-1's decisions one step
//     later (arrange_sets, with the ordinal bits of the odd lanes OR-ed into the band's ordinal words).
//
// Windows taller than 256 rows take several passes; between passes the bottom row of lane 31 goes through
// the node records (R2_BS / R2_BG), exactly like between the bands of Phase2.
//
// The arithmetic is update_column<8> of poa_kernel.cuh: results are bit-identical to the thread-per-window
// kernels by construction (tests/emul runs this file lane by lane on the CPU against the goldens).
#pragma once
#include "poa_kernel.cuh"

namespace elector {

constexpr int kCoopRows = 8;                    // rows per lane
constexpr int kCoopPassRows = 32 * kCoopRows;   // rows per pass of the warp
constexpr int kCoopGroup = 2;                   // windows per warp (measured: 1, 2 and 4 within 2 % of each other on config 1, 8 and more slower)

// what lane l hands to lane l+1 after it has finished a node
struct CoopLink {
  uint32_t ra;   // the node (letter + shape)
  uint32_t mv;   // the lane's moves of that node (rows 0-7 of a 16-row band in the upper half-word)
  int S, G;      // bottom row of the lane at that node
};

template <bool GENERIC_SUB>
struct CoopLane {
  int S[kCoopRows], G[kCoopRows], h;   // frontier set A (set B: shared memory slot, like Phase2::band)
  int kindA, kindB, bsel;
  uint32_t yw[kCoopRows / 4];
  int best, best_j;
  CoopLink out;

  EL_HDN void begin(const Phase2<GENERIC_SUB> &win, int r0) {
#pragma unroll
    for (int k = 0; k < kCoopRows / 4; ++k) yw[k] = win.fs.w(win.Lp->f_unc + (uint32_t)(r0 >> 2) + k);
#pragma unroll
    for (int r = 0; r < kCoopRows; ++r) S[r] = G[r] = 0;
    h = 0; kindA = kindB = 0; bsel = 0;
    best = -999999; best_j = -1;
    out.ra = out.mv = 0; out.S = out.G = 0;
  }

  // node j of the window `win` (scratch of the window's owner lane) in this lane's rows r0 .. r0+7:
  //   in          : the node and row r0-1 of its column (from the lane above, or from the node record for lane 0)
  //   bset        : this lane's two frontier-set slots
  //   odd         : the lane holds rows 8-15 of its 16-row band b; it stores the band's moves word
  //   store_alone : an even lane that is the last of the window (the band has 8 rows or fewer)
  //   boundary    : the pass is not the last one and this is lane 31: the bottom row goes to the node record
  //   final_row   : row (0..7) of the window's last letter if this lane holds it in the last pass, else -1
  EL_HDN void step(const Phase2<GENERIC_SUB> &win, uint32_t *bset, int r0, int b, bool odd, bool store_alone, bool boundary,
                   int final_row, int j, const CoopLink &in) {
    constexpr int R = kCoopRows;
    const uint32_t ra = in.ra;
    const int m = (ra >> 8) & 3;
    if ((ra & (NF_TWO | NF_NOPRED | NF_VIRT | NF_PREDC)) || kindA != m) {
      uint32_t *sa = bset + (1 - bsel) * kSlotWords, *sb = bset + bsel * kSlotWords;
#pragma unroll
      for (int r = 0; r < R; ++r) { sa[r * 32] = (uint32_t)S[r]; sa[(R + r) * 32] = (uint32_t)G[r]; }
      sa[2 * R * 32] = (uint32_t)h;
      uint32_t *po = nullptr;
      if (ra & (NF_VIRT | NF_TWO)) po = win.scr.at(win.Lp->o_ord + ((ra >> NF_SLOT_SHIFT) * win.Lp->ord_bands + (uint32_t)b) * 2);
      const uint32_t st = arrange_sets(sa, sb, R, r0, ra, kindA, kindB, win.sc.open, win.sc.ext, po, odd ? R : 0, odd);
      kindA = st & 3; kindB = (st >> 2) & 3;
      if (st & 16u) { bsel = 1 - bsel; sa = sb; }
#pragma unroll
      for (int r = 0; r < R; ++r) { S[r] = (int)sa[r * 32]; G[r] = (int)sa[(R + r) * 32]; }
      h = (int)sa[2 * R * 32];
    }
    const uint32_t mv = update_column<R, GENERIC_SUB>(win.sc, S, G, yw, ra & 0xff, h, in.G);
    h = in.S;
    uint32_t *p = win.rec((uint32_t)j);
    if (boundary) { p[R2_BS * 32] = (uint32_t)S[R - 1]; p[R2_BG * 32] = (uint32_t)G[R - 1]; }
    if (odd) p[(R2_MOVES + b) * 32] = in.mv | (mv >> 16);
    else if (store_alone) p[(R2_MOVES + b) * 32] = mv;
    if (final_row >= 0 && (ra & NF_FINAL)) {
      const int s = pick_row<R>(S, final_row);
      if (s > best) { best = s; best_j = j; }   // ties keep the smaller j (align_lpo_po2.c:410-417)
    }
    out.ra = ra; out.mv = mv; out.S = S[R - 1]; out.G = G[R - 1];
  }
};

// geometry of one pass
struct CoopPass {
  int row0, nl, band0;
  bool last;
  EL_HD void set(int ly, int p) {
    row0 = p * kCoopPassRows;
    const int left = ly - row0;
    nl = left >= kCoopPassRows ? 32 : (left + kCoopRows - 1) / kCoopRows;
    band0 = p * (kCoopPassRows / kBand);
    last = left <= kCoopPassRows;
  }
};
EL_HD int coop_passes(int ly) { return (ly + kCoopPassRows - 1) / kCoopPassRows; }

// ---- phase 1 through the same wavefront: DP1 is the DP of the linear partial order lin(ref) against lin(cor) ----
// The owner lane writes lin(ref) as a 16-bit node list (into the window's P1 slot, which fuse 1 overwrites afterwards),
// prepares it like any P1 and, after the cooperative DP and the traceback of Phase2, runs fuse 1 on the x2y fields.
struct LayoutC1 {
  Layout2 l2;        // rows = cor (f_unc holds the cor codes), nodes = lin(ref)
  uint32_t o_ref;    // packed ref codes (fuse 1 reads them)
  uint32_t total;
};
EL_HD void make_layout_c1(LayoutC1 &L, int LR, int LC) {
  make_layout2(L.l2, LR, LC);
  L.o_ref = L.l2.total;
  L.total = L.o_ref + cdiv_u((uint32_t)LR, 4) + 1;
}
EL_HDN inline void linear_node_list(const LaneScratch &scr, uint32_t o_ref, int lr, uint16_t *out, uint32_t carried = NF_REF) {
  uint64_t *out4 = reinterpret_cast<uint64_t *>(out);
  uint64_t acc = 0;
  for (int j = 0; j < lr; ++j) {
    const uint32_t v = (uint32_t)scr.code_at(o_ref, j) | carried | (j == 0 ? NF_INITIAL : 0u) | (j == lr - 1 ? NF_FINAL : 0u);
    acc |= (uint64_t)v << (16 * (j & 3));
    if ((j & 3) == 3) { out4[j >> 2] = acc; acc = 0; }
  }
  if (lr & 3) out4[lr >> 2] = acc;
}
// owner-lane steps of a cooperative phase 1 around the DP (the fast part of these long windows lives in global scratch)
template <bool GENERIC_SUB>
EL_HDN void coop1_before(const Phase2<GENERIC_SUB> &ph, const LayoutC1 &L, const uint8_t *ref, int lr, const uint8_t *cor, int lc, uint16_t *p1_slot) {
  ph.scr.pack_codes(ph.sc.tab, ref, lr, L.o_ref);
  ph.fs.pack_codes(ph.sc.tab, cor, lc, L.l2.f_unc);
  linear_node_list(ph.scr, L.o_ref, lr, p1_slot);
  ph.prepare(p1_slot, lr);
}
template <bool GENERIC_SUB>
EL_HDN int coop1_after(const Phase2<GENERIC_SUB> &ph, const LayoutC1 &L, int lr, int lc, int best_j, uint16_t *p1_slot, int &spcode) {
  AlignBits al = ph.bits();
  ph.traceback(lr, lc, best_j, al);
  // fuse 1 reads the ref codes from the slow part and the cor codes from the fast part: both through one accessor based at
  // the slow part (the fast part of these kernels is global scratch at o_fast, so its offsets are plain scratch offsets)
  return fuse1(ph.scr, L.o_ref, L.l2.o_fast + L.l2.f_unc, al, lr, lc, p1_slot, spcode);
}

#ifdef __CUDACC__
// DP2 of one window by the whole warp (align_lpo_po2.c:269-433): win = Phase2 view of the window (scratch of its
// owner lane), bset = this lane's frontier-set slots.  Returns the best FINAL score / node in every lane.
template <bool GENERIC_SUB>
__device__ __forceinline__ void coop_dp(const Phase2<GENERIC_SUB> &win, uint32_t *bset, int nx, int ly, int &best, int &best_j) {
  const int lane = threadIdx.x;
  CoopLane<GENERIC_SUB> st;
  const int np = coop_passes(ly);
  for (int p = 0; p < np; ++p) {
    CoopPass ps;
    ps.set(ly, p);
    const int r0 = ps.row0 + lane * kCoopRows;
    const int b = ps.band0 + (lane >> 1);
    const bool odd = lane & 1, mine = lane < ps.nl;
    const bool store_alone = !odd && lane == ps.nl - 1;
    const bool boundary = !ps.last && lane == 31;
    const int final_row = (ps.last && lane == ps.nl - 1) ? (ly - 1 - r0) : -1;
    __syncwarp();   // the node records written by the owner lane / by lane 31 of the previous pass are visible
    if (mine) st.begin(win, r0);
    else { st.out.ra = st.out.mv = 0; st.out.S = st.out.G = 0; st.best = -999999; st.best_j = -1; }
    CoopLink nxt;   // lane 0: node t + 1, loaded one step ahead
    nxt.ra = nxt.mv = 0; nxt.S = nxt.G = 0;
    if (lane == 0) { const uint32_t *q = win.rec(0); nxt.ra = q[R2_NODE * 32]; nxt.S = (int)q[R2_BS * 32]; nxt.G = (int)q[R2_BG * 32]; }
    const int steps = nx + ps.nl - 1;
#pragma unroll 1
    for (int t = 0; t < steps; ++t) {
      CoopLink in;
      in.ra = __shfl_up_sync(EL_WARP_FULL, st.out.ra, 1);
      in.mv = __shfl_up_sync(EL_WARP_FULL, st.out.mv, 1);
      in.S = __shfl_up_sync(EL_WARP_FULL, st.out.S, 1);
      in.G = __shfl_up_sync(EL_WARP_FULL, st.out.G, 1);
      if (lane == 0) {
        in = nxt;
        if (t + 1 < nx) { const uint32_t *q = win.rec((uint32_t)(t + 1)); nxt.ra = q[R2_NODE * 32]; nxt.S = (int)q[R2_BS * 32]; nxt.G = (int)q[R2_BG * 32]; }
      }
      const int j = t - lane;
      if (mine && j >= 0 && j < nx) st.step(win, bset, r0, b, odd, store_alone, boundary, final_row, j, in);
      __syncwarp();
    }
    if (ps.last) {
      best = __shfl_sync(EL_WARP_FULL, st.best, ps.nl - 1);
      best_j = __shfl_sync(EL_WARP_FULL, st.best_j, ps.nl - 1);
    }
  }
}

#ifndef EL_MIN_WARPS_COOP
#define EL_MIN_WARPS_COOP 24
#endif

// Phase 2 of the longest windows: groups of kCoopGroup windows per warp (owners = lanes 0..kCoopGroup-1).
template <bool GENERIC_SUB>
// linear_seg: the launch holds windows whose P1 is lin(ref) with every node carrying both letters (the linear segments of
// sort 2); their node list is rebuilt from the reference letters (windows whose cor is ref never ran phase 1, bin_kernel.cuh).
__global__ void __launch_bounds__(32, EL_MIN_WARPS_COOP) poa_dp2_coop_kernel(PoaArgs a, const SymbolTables *g_tab, bool linear_seg) {
  __shared__ uint32_t s_tab[(GENERIC_SUB ? sizeof(SymbolTables) : offsetof(SymbolTables, sub)) / 4];
  __shared__ Layout2 s_layout;
  __shared__ uint32_t s_bset[2 * kSlotWords];
  const int lane = threadIdx.x;
  __shared__ SegRun s_run;
  if (!seg_setup(a, s_run)) return;
  Phase2<GENERIC_SUB> c;
  uint32_t *const warp_scratch = s_run.scratch + (size_t)blockIdx.x * s_run.warp_words * 32;
  c.scr.base = warp_scratch + lane;
  c.bset = s_bset + lane;
  c.sc.tab = stage_tables<GENERIC_SUB>(s_tab, g_tab);
  c.sc.match = a.match; c.sc.mismatch = a.mismatch; c.sc.open = a.open; c.sc.ext = a.ext;
  c.sc.mis2 = a.mis2; c.sc.nopen2 = a.nopen2; c.sc.ext2 = a.ext2;
  c.Lp = &s_layout;
  for (;;) {
    int base = 0;
    if (lane == 0) base = atomicAdd(s_run.work_counter, kCoopGroup);
    base = __shfl_sync(EL_WARP_FULL, base, 0);
    if (base >= s_run.n_items) break;
    const int cnt = min(kCoopGroup, s_run.n_items - base);
    const bool owner = lane < cnt;
    int nring = 0, w = -1, n1 = 0, lu = 0;
    int64_t ro = 0, co = 0, uo = 0;
    if (owner) {
      w = s_run.items[base + lane];
      ro = a.ref_off[w]; co = a.cor_off[w]; uo = a.unc_off[w];
      lu = (int)(a.unc_off[w + 1] - uo);
      n1 = a.n1[w];
    }
    {
      const int mn = __reduce_max_sync(EL_WARP_FULL, n1), mu = __reduce_max_sync(EL_WARP_FULL, lu);
      __syncwarp();
      if (lane == 0) make_layout2(s_layout, mn, mu);
      __syncwarp();
    }
    if (s_layout.total > s_run.warp_words) { if (lane == 0) atomicExch(a.error_flag, 2); break; }  // cannot happen (monotone layout)
    c.fs.base = c.scr.base + (size_t)s_layout.o_fast * 32;   // long windows: the fast part stays in global scratch
    int nrings = 0;
    if (owner) {
      c.fs.pack_codes(c.sc.tab, a.unc + uo, lu, s_layout.f_unc);
      uint16_t *p1 = a.p1_nodes + p1_offset(ro - a.ro0, co - a.co0, w);
      if (linear_seg) {
        c.scr.pack_codes(c.sc.tab, a.ref + ro, n1, s_layout.o_tmp);
        linear_node_list(c.scr, s_layout.o_tmp, n1, p1, NF_REF | NF_COR);
      }
      nrings = c.prepare(p1, n1);
    }
    int s2 = 0, bj = -1;
    for (int i = 0; i < cnt; ++i) {
      const int nx = __shfl_sync(EL_WARP_FULL, n1, i), ly = __shfl_sync(EL_WARP_FULL, lu, i);
      Phase2<GENERIC_SUB> win = c;
      win.scr.base = warp_scratch + i;
      win.fs.base = win.scr.base + (size_t)s_layout.o_fast * 32;
      int best, best_j;
      coop_dp<GENERIC_SUB>(win, c.bset, nx, ly, best, best_j);
      if (lane == i) { s2 = best; bj = best_j; }
    }
    __syncwarp();
    AlignBits al = c.bits();
    if (owner) {
      c.traceback(n1, lu, bj, al);
      nring = columns_of(nrings, lu, al.nmatch);
      a.nring[w] = nring;
      if (a.score2) a.score2[w] = s2;
      if (a.cells) {
        const int64_t lr = a.ref_off[w + 1] - ro, lc = a.cor_off[w + 1] - co;
        a.cells[w] = lr * lc + (int64_t)n1 * lu;
      }
    }
    __syncwarp();
    RowSink out;
    if (alloc_window_rows(a, s_run.rows_cap, owner, w, nring, out)) c.fuse_emit(al, n1, lu, out);
    __syncwarp();
  }
}

// Phase 1 of the longest windows: same grouping; results and phase-2 bookkeeping as poa_dp1_kernel.
template <bool GENERIC_SUB>
__global__ void __launch_bounds__(32, EL_MIN_WARPS_COOP) poa_dp1_coop_kernel(PoaArgs a, const SymbolTables *g_tab) {
  __shared__ uint32_t s_tab[(GENERIC_SUB ? sizeof(SymbolTables) : offsetof(SymbolTables, sub)) / 4];
  __shared__ LayoutC1 s_layout;
  __shared__ uint32_t s_bset[2 * kSlotWords];
  const int lane = threadIdx.x;
  __shared__ SegRun s_run;
  if (!seg_setup(a, s_run)) return;
  Phase2<GENERIC_SUB> c;
  uint32_t *const warp_scratch = s_run.scratch + (size_t)blockIdx.x * s_run.warp_words * 32;
  c.scr.base = warp_scratch + lane;
  c.bset = s_bset + lane;
  c.sc.tab = stage_tables<GENERIC_SUB>(s_tab, g_tab);
  c.sc.match = a.match; c.sc.mismatch = a.mismatch; c.sc.open = a.open; c.sc.ext = a.ext;
  c.sc.mis2 = a.mis2; c.sc.nopen2 = a.nopen2; c.sc.ext2 = a.ext2;
  c.Lp = &s_layout.l2;
  for (;;) {
    int base = 0;
    if (lane == 0) base = atomicAdd(s_run.work_counter, kCoopGroup);
    base = __shfl_sync(EL_WARP_FULL, base, 0);
    if (base >= s_run.n_items) break;
    const int cnt = min(kCoopGroup, s_run.n_items - base);
    const bool owner = lane < cnt;
    int w = -1, lr = 0, lc = 0;
    int64_t ro = 0, co = 0;
    if (owner) {
      w = s_run.items[base + lane];
      ro = a.ref_off[w]; co = a.cor_off[w];
      lr = (int)(a.ref_off[w + 1] - ro); lc = (int)(a.cor_off[w + 1] - co);
    }
    {
      const int mr = __reduce_max_sync(EL_WARP_FULL, lr), mc = __reduce_max_sync(EL_WARP_FULL, lc);
      __syncwarp();
      if (lane == 0) make_layout_c1(s_layout, mr, mc);
      __syncwarp();
    }
    if (s_layout.total > s_run.warp_words) { if (lane == 0) atomicExch(a.error_flag, 2); break; }  // cannot happen (monotone layout)
    c.fs.base = c.scr.base + (size_t)s_layout.l2.o_fast * 32;
    uint16_t *p1_slot = owner ? a.p1_nodes + p1_offset(ro - a.ro0, co - a.co0, w) : nullptr;
    if (owner) coop1_before<GENERIC_SUB>(c, s_layout, a.ref + ro, lr, a.cor + co, lc, p1_slot);
    int s1 = 0, bj = -1;
    for (int i = 0; i < cnt; ++i) {
      const int nx = __shfl_sync(EL_WARP_FULL, lr, i), ly = __shfl_sync(EL_WARP_FULL, lc, i);
      Phase2<GENERIC_SUB> win = c;
      win.scr.base = warp_scratch + i;
      win.fs.base = win.scr.base + (size_t)s_layout.l2.o_fast * 32;
      int best, best_j;
      coop_dp<GENERIC_SUB>(win, c.bset, nx, ly, best, best_j);
      if (lane == i) { s1 = best; bj = best_j; }
    }
    __syncwarp();
    int spcode = 0, n1 = 0;
    if (owner) n1 = coop1_after<GENERIC_SUB>(c, s_layout, lr, lc, bj, p1_slot, spcode);
    phase1_epilogue(a, owner, w, n1, s1, spcode, lr, lc);
    __syncwarp();
  }
}
#endif  // __CUDACC__

// ---- the same wavefront, lane by lane, for the CPU emulation harness (tests/emul; never linked into the library) ----
template <bool GENERIC_SUB>
inline void coop_dp_emulated(const Phase2<GENERIC_SUB> &win, uint32_t *bset_warp /* 2 * kSlotWords words */, int nx, int ly, int &best, int &best_j) {
  CoopLane<GENERIC_SUB> st[32];
  const int np = coop_passes(ly);
  for (int p = 0; p < np; ++p) {
    CoopPass ps;
    ps.set(ly, p);
    for (int lane = 0; lane < 32; ++lane) {
      if (lane < ps.nl) st[lane].begin(win, ps.row0 + lane * kCoopRows);
      else { st[lane].out.ra = st[lane].out.mv = 0; st[lane].out.S = st[lane].out.G = 0; st[lane].best = -999999; st[lane].best_j = -1; }
    }
    const int steps = nx + ps.nl - 1;
    for (int t = 0; t < steps; ++t) {
      for (int lane = 31; lane >= 0; --lane) {   // descending: lane l reads what lane l-1 produced in step t-1
        CoopLink in;
        if (lane == 0) {
          in.mv = 0;
          if (t < nx) { const uint32_t *q = win.rec((uint32_t)t); in.ra = q[R2_NODE * 32]; in.S = (int)q[R2_BS * 32]; in.G = (int)q[R2_BG * 32]; }
          else { in.ra = 0; in.S = in.G = 0; }
        } else in = st[lane - 1].out;
        const int j = t - lane;
        if (lane < ps.nl && j >= 0 && j < nx) {
          const int r0 = ps.row0 + lane * kCoopRows;
          const bool odd = lane & 1;
          st[lane].step(win, bset_warp + lane, r0, ps.band0 + (lane >> 1), odd, !odd && lane == ps.nl - 1, !ps.last && lane == 31,
                        (ps.last && lane == ps.nl - 1) ? (ly - 1 - r0) : -1, j, in);
        }
      }
    }
    if (ps.last) { best = st[ps.nl - 1].best; best_j = st[ps.nl - 1].best_j; }
  }
}

}  // namespace elector
