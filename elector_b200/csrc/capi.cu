// capi.cu -- C-ABI (include/elector_poa.h) over the sm_100a kernels.  Host side of the
// `poa` drop-in: matrix analysis, size-class binning, scratch management, launches.
// There is NO CPU implementation of the alignment here: every entry point either runs
// the CUDA kernels or returns an error.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/elector_poa.h"
#include "host_io.hpp"
#include "poa_kernel.cuh"
#include "poa_packed.cuh"
#include "poa_coop.cuh"
#include "poa_dual.cuh"
#include "bin_kernel.cuh"
#include "host_setup.hpp"
#include "tally_kernel.cuh"
#include "wire_kernel.cuh"
#include "split_kernel.cuh"
#include "peak_kernel.cuh"
#include "report_host.hpp"
#include "prep_host.hpp"

using namespace elector;

namespace {

thread_local std::string g_init_error;

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

}  // namespace

struct elector_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  int resident_ph1 = 0, resident_ph2 = 0, resident_ph1p = 0, resident_ph2l = 0, resident_coop = 0;  // POA kernel CTAs (one warp each) resident per SM
  int arena_ph1 = 0, arena_ph2 = 0, arena_ph1p = 0, arena_ph2l = 0, arena_ph2d = 0;   // bytes of the per-warp shared-memory arena of each kernel (fast part of the layouts)
  int coop_group = kCoopGroupDefault;  // windows per warp of the warp-cooperative kernel; 0 = the longest windows stay thread-per-window (ELECTOR_COOP_GROUP)
  int64_t *h_totals = nullptr;             // pinned: letters of ref / cor of the current call
  cudaStream_t stream = nullptr;
  cudaStream_t side[16] = {};   // one per segment that does not run on the main stream
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr, uev0 = nullptr, uev1 = nullptr, ev_fork = nullptr, ev_rows = nullptr;
  cudaStream_t lin_stream = nullptr;   // the sort of the linear segments of phase 2 (next to that of phase 1), then the sort of the general ones
  cudaEvent_t ev_fork_v[6] = {}, ev_sorted = nullptr, ev_lin_done = nullptr, ev_lin_sorted = nullptr, ev_bulk1 = nullptr;
  cudaEvent_t ev_view[3][2][2] = {};   // ELECTOR_TRACE=2: start / end of the launches of a view (phase 1, linear, general) x (cooperative, others)
  float last_ms_phase1 = 0.f;  // sort 1 + phase-1 kernels of the last run (last_ms covers everything)
  cudaEvent_t ev_join[16] = {};
  elector::BinTable *h_bintab = nullptr;  // pinned: the two tables of the last call as the device left them (errors, scratch needs)
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   // H2D / D2H of the pipelined host entry point
  cudaEvent_t ev_call = nullptr;                        // ELECTOR_TRACE: start of a pipelined call on the device
  ScoreMatrix mat;
  ScoringSetup sc;
  DevBuf d_tab, d_ref, d_cor, d_unc, d_roff, d_coff, d_uoff, d_items, d_scratch, d_scratch_lin, d_scratch2, d_ctrl, d_hist, d_bintab, d_key, d_key2, d_n1, d_p1;
  DevBuf d_rows, d_rowoff, d_stride, d_nring, d_s1, d_s2, d_cells;
  int64_t merged_cap = 0;  // bytes per merged-row buffer of the last merge
  // worker contexts of the pipelined entry points (worker_slots): children on this device, one per extra worker thread
  std::vector<elector_ctx *> workers;
  std::vector<elector_ctx *> peers;   // worker contexts of elector_reads_pipeline_run on the other devices
  int64_t *h_sums = nullptr;   // pinned: global counters of a chunk + the tally overflow flag
  DevBuf d_pk[3], d_exc_pos, d_exc_byte, d_rel, d_nib[3], d_esc_pos, d_esc_byte;   // compact wire format: packed letters, exceptions, 32-bit offsets in; 4-bit merged rows and their escapes out
  void *h_stage = nullptr; size_t h_stage_cap = 0;   // pinned staging of a chunk's 32-bit offsets
  DevBuf d_stretch; int64_t stretch_reads = 0;
  DevBuf d_wdst, d_sums, d_tally_scan, d_tally_out, d_readfirst, d_mtot, d_moff, d_mlen, d_mref, d_mcor, d_munc;
  bool trace = false;
  int band_w = 6;          // ELECTOR_BAND_W: base half-width of the diagonal band of the packed linear kernels (+ rows/16 in phase 1, + rows/8 in phase 2; 0 = full DP)
  int resident_ph2d = 0;   // 0: the general windows of phase 2 run the INT32 kernel with frontier sets
  unsigned side_used = 0;        // side streams with launches that `st` has not been made to wait for yet
  elector::BinTable *h_plan = nullptr;   // pinned: the plans of phase 1 / phase 2 of the current call (read_plans)
  // rows of a pipelined chunk in two regions: the windows of the linear segments of phase 2 (most windows, finished early)
  // write theirs behind their own cursor, so that they can leave for the host while the general windows still compute
  bool split_rows = false;          // set by process_chunk around run_device
  int64_t region_b_base = 0;        // out: where the linear region starts in the caller's row buffer
  cudaEvent_t ev_lin = nullptr;     // the linear region is complete; its cursor and start are in h_totals[6..7]
  cudaEvent_t ev_merged = nullptr;  // the merge of a chunk is done and its rows are packed for the wire (before the tally); the merged columns of the chunk are in h_totals[2]
  cudaEvent_t wait_in[2] = {nullptr, nullptr};   // run_device: phase 1 / phase 2 wait for these (letters still on their way), when set
  cudaEvent_t ev_in[2] = {nullptr, nullptr};
  void *split_state = nullptr;   // device buffers of the window cutting (split_capi.inl)
  cudaEvent_t ev_split0 = nullptr, ev_split1 = nullptr, ev_mt0 = nullptr, ev_mt1 = nullptr;   // window cutting; merge + tally of elector_reads_run
  float last_ms_split = 0.f, last_ms_tally = 0.f;
  std::string err;
  float last_ms = 0.f;
  int last_launches = 0;

  int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    err = buf;
    return code;
  }
};

#define CU(call)                                                                       \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess) return ctx->fail(ELECTOR_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

namespace {

int merge_device(elector_ctx *ctx, int64_t n_reads, const int64_t *h_read_first, int64_t n_windows, const uint8_t *d_rows,
                 int64_t rows_bytes, const int64_t *d_row_off, const int32_t *d_row_stride, const int32_t *d_nring);
int tally_device(elector_ctx *ctx, int64_t n_reads, const uint8_t *dR, const uint8_t *dC, const uint8_t *dU,
                 const int64_t *d_off, const int32_t *d_len, int64_t *d_counters, int64_t total_bytes);
int check_scan_overflow(elector_ctx *ctx, int64_t n_reads);

const size_t kCtrlWords = 64;  // d_ctrl: [0..1] rows cursor (u64), [2] error flag, [3] tally overflow, [4..19] phase-1 and [20..35] phase-2 work counters, [36..37] rows cursor of the linear region, [38..39] where that region starts, [41] abort flag
const int kAbortWord = 41;     // d_ctrl[41]: the alignment kernels of the call did not (all) run; merge and tally leave at once
const int kSideStreams = 16;   // >= kMaxSegs: no two segments of a phase share a side stream
const int kScratchRetries = 3; // runs of an alignment again after its scratch pools were grown (check_tables)

#ifndef EL_MIN_WARPS_PH1P
#define EL_MIN_WARPS_PH1P 28  // packed DP1: register cap 72 (64 spills since the diagonal band: 28 warps measured 0.2 ms per step faster than 32)
#endif
#ifndef EL_MIN_WARPS_PH2D
#define EL_MIN_WARPS_PH2D 20  // dual-frontier packed DP2: register cap 96 (measured: 9.94 ms per config-1 step against 10.26 ms at 24 warps / 80 registers)
#endif
#ifndef EL_MIN_WARPS_PH2L
#define EL_MIN_WARPS_PH2L 28  // packed linear DP2: register cap 72
#endif

// kind of a segment's kernel: INT32 cells (poa_kernel.cuh), 16-bit packed cells (poa_packed.cuh), or -- phase 2 only --
// the packed linear x linear kernel for windows whose P1 is linear
// or -- phase 2 only -- the warp-cooperative INT32 kernel for the segments that hold the longest windows (poa_coop.cuh)
enum SegKind { kInt32 = 0, kPacked = 1, kLinear = 2, kCoop = 3, kDual = 4 };

template <bool GS>
cudaError_t launch_phase(int phase, int kind, cudaStream_t st, PoaArgs &a, int grid, const SymbolTables *tab, int coop_group, bool linear_seg,
                         const elector_ctx *ctx) {
  auto arena = [&](int bytes) { a.arena_words = (uint32_t)(bytes / 128); return (size_t)bytes; };
  if (kind == kCoop && phase == 1) { a.arena_words = 0; poa_dp1_coop_kernel<GS><<<grid, 32, 0, st>>>(a, tab, coop_group); }
  else if (kind == kCoop) { a.arena_words = 0; poa_dp2_coop_kernel<GS><<<grid, 32, 0, st>>>(a, tab, coop_group, linear_seg); }
  else if (phase == 1) {
    if (kind == kPacked) poa_dp1_kernel<Phase1P, EL_MIN_WARPS_PH1P><<<grid, 32, arena(ctx->arena_ph1p), st>>>(a, tab);
    else poa_dp1_kernel<Phase1<GS>, EL_MIN_WARPS_PH1><<<grid, 32, arena(ctx->arena_ph1), st>>>(a, tab);
  } else if (kind == kLinear) poa_dp2_kernel<Phase2L, EL_MIN_WARPS_PH2L><<<grid, 32, arena(ctx->arena_ph2l), st>>>(a, tab);
  else if (kind == kDual) poa_dp2_kernel<Phase2D, EL_MIN_WARPS_PH2D><<<grid, 32, arena(ctx->arena_ph2d), st>>>(a, tab);
  else poa_dp2_kernel<Phase2<GS>, EL_MIN_WARPS_PH2><<<grid, 32, arena(ctx->arena_ph2), st>>>(a, tab);
  return cudaGetLastError();
}

// Residency of a thread-per-window kernel (one-warp CTAs: registers bound it) and the largest per-warp arena in dynamic
// shared memory that keeps it: the SM's shared memory divided among the resident CTAs, minus the kernel's static part and
// the 1 KB the system reserves per CTA.
template <class K>
void size_arena(K kernel, size_t smem_per_sm, int &resident, int &arena_bytes) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, 32, 0);
  arena_bytes = 0;
  if (resident < 1) return;
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kernel) != cudaSuccess) return;
  long per_cta = (long)(smem_per_sm / (size_t)resident) - (long)fa.sharedSizeBytes - 1024;
  per_cta = std::min<long>(per_cta, 40 * 1024) & ~127L;
  for (; per_cta > 0; per_cta -= 128) {
    int r = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, kernel, 32, (size_t)per_cta) == cudaSuccess && r >= resident) break;
  }
  arena_bytes = per_cta > 0 ? (int)per_cta : 0;
  if (arena_bytes > 48 * 1024 - (int)fa.sharedSizeBytes) arena_bytes = (48 * 1024 - (int)fa.sharedSizeBytes) & ~127;
}

template <bool GS>
void resident_warps_per_sm(elector_ctx *ctx, size_t smem_per_sm) {
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->resident_coop, poa_dp2_coop_kernel<GS>, 32, 0);
  int coop1 = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&coop1, poa_dp1_coop_kernel<GS>, 32, 0);
  ctx->resident_coop = std::min(ctx->resident_coop, coop1);
  size_arena(poa_dp2_kernel<Phase2L, EL_MIN_WARPS_PH2L>, smem_per_sm, ctx->resident_ph2l, ctx->arena_ph2l);
  size_arena(poa_dp1_kernel<Phase1<GS>, EL_MIN_WARPS_PH1>, smem_per_sm, ctx->resident_ph1, ctx->arena_ph1);
  size_arena(poa_dp2_kernel<Phase2<GS>, EL_MIN_WARPS_PH2>, smem_per_sm, ctx->resident_ph2, ctx->arena_ph2);
  size_arena(poa_dp1_kernel<Phase1P, EL_MIN_WARPS_PH1P>, smem_per_sm, ctx->resident_ph1p, ctx->arena_ph1p);
  size_arena(poa_dp2_kernel<Phase2D, EL_MIN_WARPS_PH2D>, smem_per_sm, ctx->resident_ph2d, ctx->arena_ph2d);
}

// ---- device-side planning of a sort view's segments --------------------------------------------------------------
// A sort view = a contiguous range of one table's segments and bins, sorted and launched together: phase 1; the linear
// segments of phase 2 (windows whose cor is ref: sorted by the size sort itself, launched while phase 1 runs); the
// general segments of phase 2 (sorted after phase 1).  What the host knows before the sort runs is static: which kernel a
// segment runs and how many CTAs its launch has.  Everything else -- the segment's slice of the work list, the scratch
// layout of its maxima, how many CTAs take work and where their scratch starts -- is computed here, on the device.
struct SegStatic {
  int8_t kind[kMaxSegs];     // SegKind of the segment's kernel
  int32_t grid[kMaxSegs];    // CTAs of the segment's launch
  int32_t seg0, seg1;        // the view's segments
  int32_t phase;             // 1 or 2
  int32_t coop_group;
  int32_t counter0;          // control word of segment 0's work counter
  unsigned long long pool_words;     // scratch pool of the view
  unsigned long long budget_words;   // no single segment takes more than this
};

__device__ uint32_t layout_words(int phase, int kind, int m0, int m1) {
  if (phase == 1) {
    if (kind == kCoop) { LayoutC1 L; make_layout_c1(L, m0, m1); return L.total; }
    if (kind == kPacked) { Layout1P L; make_layout1p(L, m0, m1); return L.total; }
    Layout1 L; make_layout1(L, m0, m1); return L.total;
  }
  if (kind == kLinear) { Layout2L L; make_layout2l(L, m0, m1); return L.total; }
  Layout2 L; make_layout2(L, m0, m1); return L.total;
}

// one warp: a segment per lane, then lane 0 adds up the scratch.  split_rows: the view is the linear one of a call whose rows
// go to two regions -- the linear segments write [cap_a, rows_cap), the general ones [cursor, cap_a); ctrl64[18] = cursor of
// the linear region, [19] = cap_a
__global__ void plan_segments_kernel(BinTable *tab, SegStatic ss, unsigned long long *ctrl64, long long rows_cap, int split_rows) {
  __shared__ unsigned long long s_words[32];
  __shared__ int s_big;
  const int lane = threadIdx.x, s = ss.seg0 + lane;
  if (lane == 0) s_big = 0;
  __syncwarp();
  SegPlanDev pl;
  pl.start = pl.count = pl.max_ctas = pl.counter = 0; pl.warp_words = pl.pad = 0; pl.scratch_off = 0;
  unsigned long long words = 0;
  if (s < ss.seg1) {
    pl.start = tab->seg[s].start; pl.count = tab->seg[s].count; pl.counter = ss.counter0 + s;
    if (pl.count > 0) {
      pl.warp_words = layout_words(ss.phase, ss.kind[s], tab->seg_max[s * 4], tab->seg_max[s * 4 + 1]);
      const int per = ss.kind[s] == kCoop ? ss.coop_group : 32;
      long long ctas = ((long long)pl.count + per - 1) / per;
      if (ctas > ss.grid[s]) ctas = ss.grid[s];
      const unsigned long long per_warp = (unsigned long long)pl.warp_words * 32;
      while (ctas > 1 && per_warp * (unsigned long long)ctas > ss.budget_words / 2) ctas = (ctas + 1) / 2;   // huge windows: fewer warps in flight
      pl.max_ctas = (int32_t)ctas;
      words = per_warp * (unsigned long long)ctas;
      if (words > ss.budget_words) s_big = 1;
    }
  }
  s_words[lane] = words;
  __syncwarp();
  unsigned long long off = 0, total = 0;
  for (int k = 0; k < 32; ++k) { if (k == lane) off = total; total += s_words[k]; }
  const bool invalid = ss.phase == 1 && (tab->err_code == 1 || tab->err_code == 2);   // a window the kernels cannot take (the size sort said so)
  const bool overflow = total > ss.pool_words || s_big;
  if (s < ss.seg1) {
    pl.scratch_off = off;
    if (overflow) pl.max_ctas = 0;   // nothing of this view runs; the host grows the pool and runs the call again
    tab->plan[s] = pl;
  }
  if (lane == 0) {
    if (overflow) {
      if (tab->err_code == 0) tab->err_code = s_big ? 4 : 3;
      if (total > tab->need_words) tab->need_words = total;
    }
    if (overflow || invalid) reinterpret_cast<int32_t *>(ctrl64)[kAbortWord] = 1;   // merge and tally have nothing defined to work on
    if (split_rows) {
      const unsigned long long cap_a = (unsigned long long)((rows_cap - (long long)tab->lin_bytes) & ~15ll);
      ctrl64[18] = cap_a;
      ctrl64[19] = cap_a;
    }
  }
}

struct SortView {
  BinTable *dtab; int phase, seg0, seg1, bin0, bin1;
  int32_t *hist;      // the table's histogram (all bins)
  int32_t *chunks;    // chunk totals of this view
  const int32_t *key; int32_t *items;
  DevBuf *pool;
  int counter0;
};

// kernel of a segment (static: known before the sort runs, see SegStatic)
int seg_kind(const elector_ctx *ctx, int phase, int s) {
  const bool small16 = ctx->sc.small_packed();
  // windows of more than 128 rows run a warp per window: the big tiers and the first small segment (129 .. 256 rows) of phase 1,
  // of the general and of the linear segments of phase 2
  if (phase == 1) return (s <= kBigTiers && ctx->coop_group > 0) ? kCoop : (s >= kBigTiers && small16) ? kPacked : kInt32;
  const bool longest = s <= kBigTiers || s == kFirstLinSeg2;
  if (longest && ctx->coop_group > 0) return kCoop;
  if (s < kBigTiers || !small16) return kInt32;
  return s >= kFirstLinSeg2 ? kLinear : ctx->resident_ph2d > 0 ? kDual : kInt32;
}
int seg_resident(const elector_ctx *ctx, int phase, int kind) {
  switch (kind) {
    case kCoop: return ctx->resident_coop;
    case kPacked: return ctx->resident_ph1p;
    case kLinear: return ctx->resident_ph2l;
    case kDual: return ctx->resident_ph2d;
    default: return phase == 1 ? ctx->resident_ph1 : ctx->resident_ph2;
  }
}

// scan + scatter + plan of one view, all on `st`
int sort_view(elector_ctx *ctx, cudaStream_t st, const SortView &v, int32_t n, SegStatic &ss, long long rows_cap, bool split_rows) {
  const int nb = v.bin1 - v.bin0, nch = (nb + kScanChunk - 1) / kScanChunk;
  bin_scan_chunks_kernel<<<nch, kScanChunk, 0, st>>>(nb, v.hist + v.bin0, v.chunks);
  bin_scan_totals_kernel<<<1, 1024, 0, st>>>(nch, v.chunks, v.hist, v.dtab, v.seg0, v.seg1, v.bin0, v.bin1);
  const int end_bit = 32 - __builtin_clz((unsigned)nb);   // bits of bin - bin0, and of the "not in this view" key nb
  bin_scatter_kernel<<<(int)(((int64_t)n + kScatterTile - 1) / kScatterTile), kScatterThreads, 0, st>>>(n, v.key, v.hist, v.chunks, v.items,
                                                                                                        v.bin0, v.bin1, end_bit);
  memset(&ss, 0, sizeof ss);
  ss.seg0 = v.seg0; ss.seg1 = v.seg1; ss.phase = v.phase; ss.coop_group = std::max(1, ctx->coop_group); ss.counter0 = v.counter0;
  ss.pool_words = v.pool->cap / 4;
  ss.budget_words = ((unsigned long long)24 << 30) / 4;
  for (int s = v.seg0; s < v.seg1; ++s) {
    const int kind = seg_kind(ctx, v.phase, s);
    ss.kind[s] = (int8_t)kind;
    ss.grid[s] = std::max(1, seg_resident(ctx, v.phase, kind)) * ctx->sm_count;
  }
  plan_segments_kernel<<<1, 32, 0, st>>>(v.dtab, ss, ctx->d_ctrl.as<unsigned long long>(), rows_cap, split_rows ? 1 : 0);
  CU(cudaGetLastError());
  ctx->last_launches += 4;
  return ELECTOR_OK;
}

// every segment of a view on its own side stream (side[first_side ...]), forked from `fork_from` (default `st`) and joined
// back into `st` by join_view.  which: 0 = the warp-cooperative segments, 1 = the others, 2 = all (cooperative first).
// A segment with a large share of the call's windows (bulk) goes to `st` itself, behind the bulk segments launched before it;
// the others get a side stream each, starting behind what `fork_from` holds at this moment.  (Measured on config 1: two bulk kernels
// side by side are slower than one after the other -- each alone fills the SMs, together they evict each other's scratch
// from the L2.)  join_view makes `st` wait for the side streams -- after ALL launches of a phase: a join between two passes
// would serialise them.
int launch_view(elector_ctx *ctx, cudaStream_t st, const SortView &v, const SegStatic &ss, PoaArgs base, int first_side, bool region_b, int64_t n,
                int which = 2, cudaStream_t fork_from = nullptr) {
  if (!fork_from) fork_from = st;
  cudaEvent_t fork = ctx->ev_fork_v[(v.phase == 1 ? 0 : v.seg0 >= kFirstLinSeg2 ? 1 : 2) + (which == 1 ? 3 : 0)];
  const BinTable &plans = ctx->h_plan[v.phase - 1];   // read_plans
  CU(cudaEventRecord(fork, fork_from));
  const int vi = v.phase == 1 ? 0 : v.seg0 >= kFirstLinSeg2 ? 1 : 2;
  if (ctx->trace) for (int w2 = 0; w2 < 2; ++w2) if (which == 2 || which == w2) CU(cudaEventRecord(ctx->ev_view[vi][w2][0], fork_from));
  int nregb = 0;
  // the warp-cooperative segments first (they hold the longest windows and set the latency floor of a call)
  for (int pass = 0; pass < 2; ++pass)
    for (int s = v.seg0; s < v.seg1; ++s) {
      const int kind = ss.kind[s];
      if ((kind == kCoop) != (pass == 0) || (which != 2 && which != pass)) continue;
      // only the segments that have work are launched, with the grids the device planned
      const SegPlanDev &pl = plans.plan[s];
      if (pl.max_ctas == 0) continue;
      const int grid = pl.max_ctas;
      const bool bulk = kind != kCoop && (int64_t)pl.count * 8 > n;
      const int side = first_side + (s - v.seg0);
      cudaStream_t ls = bulk ? st : ctx->side[side];
      if (!bulk) CU(cudaStreamWaitEvent(ls, fork, 0));
      PoaArgs a = base;
      a.tab = v.dtab; a.seg = s; a.items_base = v.items; a.scratch_base = v.pool->as<uint32_t>(); a.ctrl = ctx->d_ctrl.as<int32_t>();
      const bool linear_seg = v.phase == 2 && s >= kFirstLinSeg2;
      const cudaError_t e = ctx->sc.generic_sub ? launch_phase<true>(v.phase, kind, ls, a, grid, ctx->d_tab.as<SymbolTables>(), ss.coop_group, linear_seg, ctx)
                                                : launch_phase<false>(v.phase, kind, ls, a, grid, ctx->d_tab.as<SymbolTables>(), ss.coop_group, linear_seg, ctx);
      if (e != cudaSuccess) return ctx->fail(ELECTOR_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
      ++ctx->last_launches;
      cudaEvent_t done = ctx->ev_join[side];
      if (!bulk || region_b) CU(cudaEventRecord(done, ls));
      if (!bulk) ctx->side_used |= 1u << side;
      if (region_b && nregb < 8) { CU(cudaStreamWaitEvent(ctx->copy_out, done, 0)); ++nregb; }
    }
  return ELECTOR_OK;
}
// The plans of `ntab` tables from phase `phase` on, read back on `a` (one wait of the host, for `a` alone): the host launches
// only the segments that have work, with exact grids.  Measured on config 1: fixed-grid launches of all 27 segments (most of
// them empty, thousands of CTAs that leave at once) cost 0.4 ms per phase, a read-back 0.03 ms.
int read_plans(elector_ctx *ctx, int phase, int ntab, BinTable *dtab, cudaStream_t a) {
  CU(cudaMemcpyAsync(&ctx->h_plan[phase - 1], dtab, ntab * sizeof(BinTable), cudaMemcpyDeviceToHost, a));
  CU(cudaStreamSynchronize(a));
  return ELECTOR_OK;
}
// `st` waits for the side streams side[first .. first + count - 1] that have launched something since the last join
int join_view(elector_ctx *ctx, cudaStream_t st, int first, int count, int view) {
  for (int k = first; k < first + count; ++k)
    if (ctx->side_used & (1u << k)) { CU(cudaStreamWaitEvent(st, ctx->ev_join[k], 0)); ctx->side_used &= ~(1u << k); }
  if (ctx->trace) { CU(cudaEventRecord(ctx->ev_view[view][0][1], st)); CU(cudaEventRecord(ctx->ev_view[view][1][1], st)); }
  return ELECTOR_OK;
}

// Core: all pointers are device pointers; the host waits for the device twice, for the plans (read_plans).  Launch structure
// of one call:
//   main stream  : set-up -> size sort (recognises the windows whose cor is ref) -> sort + plan of phase 1 -> [read-back of
//                  the plans of phase 1 and of the linear segments] -> phase-1 bulk -> linear bulk -> general bulk
//   linear stream: sort + plan of the linear segments of phase 2 (next to that of phase 1); once phase 1 is done, sort + plan
//                  of the general segments -> [read-back of their plans]
// A segment that is not bulk runs on a side stream of its own.  h_roff / h_coff (host copies of the offsets) spare a read-back of four
// totals; errors (bad window, scratch pool too small) are left in the tables, which travel to h_bintab at the end.
int run_device(elector_ctx *ctx, int64_t n, const char *d_ref, const int64_t *d_roff, const char *d_cor,
               const int64_t *d_coff, const char *d_unc, const int64_t *d_uoff, const int64_t *h_roff, const int64_t *h_coff,
               char *d_rows, int64_t rows_cap, int64_t *d_rowoff, int32_t *d_stride, int32_t *d_nring, int32_t *d_s1, int32_t *d_s2,
               int64_t *d_cells, unsigned long long *d_cursor, int32_t *d_errflag, int64_t cursor_init = 0) {
  if (n == 0) return ELECTOR_OK;
  if (n > 0x7fffffff - 64) return ctx->fail(ELECTOR_EINVAL, "too many windows in one call");
  cudaStream_t st = ctx->stream;
  CU(ctx->d_items.reserve((size_t)n * 3 * sizeof(int32_t)));
  CU(ctx->d_key.reserve((size_t)n * sizeof(int32_t)));
  CU(ctx->d_key2.reserve((size_t)n * sizeof(int32_t)));
  CU(ctx->d_n1.reserve((size_t)n * sizeof(int32_t)));
  CU(ctx->d_hist.reserve((size_t)(kNumBins1 + kNumBins2 + 3 * kMaxChunks) * sizeof(int32_t)));
  CU(ctx->d_bintab.reserve(2 * sizeof(BinTable)));
  int32_t *hist1 = ctx->d_hist.as<int32_t>(), *hist2 = hist1 + kNumBins1, *chunks1 = hist2 + kNumBins2, *chunksL = chunks1 + kMaxChunks, *chunks2 = chunksL + kMaxChunks;
  BinTable *dtab1 = ctx->d_bintab.as<BinTable>(), *dtab2 = dtab1 + 1;
  int32_t *items1 = ctx->d_items.as<int32_t>(), *itemsL = items1 + n, *items2 = itemsL + n;
  // letters of ref and cor of the call (size of the P1 node lists) and their first offsets
  int64_t tot[4];
  if (h_roff && h_coff) { tot[0] = h_roff[n]; tot[1] = h_coff[n]; tot[2] = h_roff[0]; tot[3] = h_coff[0]; }
  else {   // slow path: a read-back
    CU(cudaMemcpyAsync(&ctx->h_totals[0], d_roff + n, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&ctx->h_totals[1], d_coff + n, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&ctx->h_totals[2], d_roff, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&ctx->h_totals[3], d_coff, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int k = 0; k < 4; ++k) tot[k] = ctx->h_totals[k];
  }
  CU(ctx->d_p1.reserve((size_t)(tot[0] - tot[2] + tot[1] - tot[3] + 8 * n + 8) * sizeof(uint16_t)));
  // scratch pools: kept from call to call; a call that needs more says so in its tables and its caller runs it again (check_tables)
  for (DevBuf *pool : {&ctx->d_scratch, &ctx->d_scratch_lin, &ctx->d_scratch2})
    if (pool->cap == 0) CU(pool->reserve(std::max<size_t>((size_t)64 << 20, std::min<size_t>((size_t)n * 1024, (size_t)2 << 30))));
  CU(cudaEventRecord(ctx->ev0, st));
  // control words, histograms and the two segment tables are set up by a kernel and memsets: nothing of a call's
  // set-up goes through the host-to-device copy engine, where it would queue behind the letters of a pipelined call
  CU(cudaMemsetAsync(ctx->d_hist.p, 0, (size_t)(kNumBins1 + kNumBins2) * sizeof(int32_t), st));
  {
    BinTable stat[2];   // the static part of the tables: first bin of every segment
    BinTable *htab1 = &stat[0], *htab2 = &stat[1];
    memset(stat, 0, sizeof stat);
    fill_segments1(*htab1);
    fill_segments2(*htab2);
    SegFirstBins fb;
    for (int k = 0; k <= kMaxSegs; ++k) { fb.first1[k] = htab1->seg[k].first_bin; fb.first2[k] = htab2->seg[k].first_bin; }
    fb.nseg1 = htab1->nseg; fb.nbins1 = htab1->nbins; fb.nseg2 = htab2->nseg; fb.nbins2 = htab2->nbins;
    init_call_kernel<<<1, 128, 0, st>>>(ctx->d_ctrl.as<int32_t>(), (int)kCtrlWords, (unsigned long long)cursor_init, dtab1, fb);
    CU(cudaGetLastError());
    ++ctx->last_launches;
  }
  const int bgrid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8);
  // ---- size sort ----
  // windows whose corrected letters are the reference letters need no phase 1 (bin_kernel.cuh): the sort then reads the
  // letters, so it waits for them too.  Only when their phase 2 needs no node list: Phase2L for the small linear segments,
  // the warp-cooperative kernel (which rebuilds lin(ref)) for the long ones.
  const bool ident_ok = ctx->sc.small_packed() && ctx->coop_group > 0;
  if (ident_ok && ctx->wait_in[0]) CU(cudaStreamWaitEvent(st, ctx->wait_in[0], 0));
  IdentArgs ida{(const uint8_t *)d_ref, (const uint8_t *)d_cor, ctx->d_n1.as<int32_t>(), ctx->d_key2.as<int32_t>(), hist2, dtab2->seg_max, d_s1, &dtab2->lin_bytes};
  bin1_count_kernel<<<bgrid, 256, 0, st>>>((int32_t)n, d_roff, d_coff, d_uoff, ctx->d_key.as<int32_t>(), hist1, dtab1, ident_ok, ida);
  CU(cudaGetLastError());
  ++ctx->last_launches;
  const int lin_bin0 = kBigTiers + kSmallBins2;
  const SortView v1{dtab1, 1, 0, kNumSegs1, 0, kNumBins1, hist1, chunks1, ctx->d_key.as<int32_t>(), items1, &ctx->d_scratch, 4};
  const SortView vL{dtab2, 2, kFirstLinSeg2, kNumSegs2, lin_bin0, kNumBins2, hist2, chunksL, ctx->d_key2.as<int32_t>(), itemsL, &ctx->d_scratch_lin, 20};
  const SortView v2{dtab2, 2, 0, kFirstLinSeg2, 0, lin_bin0, hist2, chunks2, ctx->d_key2.as<int32_t>(), items2, &ctx->d_scratch2, 20};
  SegStatic ss1, ssL, ss2;
  // the sort of phase 1 on the main stream; that of the linear segments of phase 2 (their keys and histogram are complete
  // after the size sort) on the linear stream, next to phase 1
  cudaStream_t sl = ctx->lin_stream;
  CU(cudaEventRecord(ctx->ev_sorted, st));
  CU(cudaStreamWaitEvent(sl, ctx->ev_sorted, 0));
  int rc = sort_view(ctx, st, v1, (int32_t)n, ss1, rows_cap, false);
  if (rc == ELECTOR_OK) rc = sort_view(ctx, sl, vL, (int32_t)n, ssL, rows_cap, ctx->split_rows);
  if (rc != ELECTOR_OK) return rc;
  CU(cudaEventRecord(ctx->ev_lin_sorted, sl));

  PoaArgs a;
  memset(&a, 0, sizeof a);
  a.ref = (const uint8_t *)d_ref; a.cor = (const uint8_t *)d_cor; a.unc = (const uint8_t *)d_unc;
  a.ref_off = d_roff; a.cor_off = d_coff; a.unc_off = d_uoff;
  a.match = ctx->sc.match; a.mismatch = ctx->sc.mismatch; a.open = ctx->sc.open; a.ext = ctx->sc.ext;
  { Scoring pk; pk.set(a.match, a.mismatch, a.open, a.ext); a.mis2 = pk.mis2; a.nopen2 = pk.nopen2; a.ext2 = pk.ext2; }
  a.ro0 = tot[2]; a.co0 = tot[3];
  a.p1_nodes = ctx->d_p1.as<uint16_t>(); a.n1 = ctx->d_n1.as<int32_t>(); a.key2 = ctx->d_key2.as<int32_t>();
  a.hist2 = hist2; a.seg2_max = dtab2->seg_max;
  a.rows_out = (uint8_t *)d_rows; a.rows_cursor = d_cursor; a.rows_cap = rows_cap;
  a.row_off = d_rowoff; a.row_stride = d_stride; a.nring = d_nring; a.score1 = d_s1; a.score2 = d_s2; a.cells = d_cells;
  a.error_flag = d_errflag;
  a.band_w = ctx->band_w;
  a.band_span = band_span_limit(ctx->sc.maxabs);

  // ---- phase 1, then the linear segments of phase 2 behind it ----
  // one read-back brings the plans of phase 1 and of the linear view (table 2; the general view's plans follow after sort 2)
  CU(cudaStreamWaitEvent(st, ctx->ev_lin_sorted, 0));
  rc = read_plans(ctx, 1, 2, dtab1, st);
  if (rc != ELECTOR_OK) return rc;
  if (ctx->wait_in[0]) CU(cudaStreamWaitEvent(st, ctx->wait_in[0], 0));
  rc = launch_view(ctx, st, v1, ss1, a, 0, false, n);
  if (rc != ELECTOR_OK) return rc;
  CU(cudaEventRecord(ctx->ev_bulk1, st));
  PoaArgs al = a, ag = a;
  if (ctx->split_rows) {
    al.rows_cursor = ctx->d_ctrl.as<unsigned long long>() + 18;   // two row regions: the linear segments behind their own cursor, up to the end of the buffer
    ag.rows_cap_dev = reinterpret_cast<const long long *>(ctx->d_ctrl.as<unsigned long long>() + 19);   // the general region ends where the linear one starts
  }
  // The linear segments need nothing from phase 1 (their windows skip it): their bulk runs on `st` right behind phase 1's,
  // their cooperative segments on side streams forked there, so that they do not wait for phase 1's cooperative ones.
  // (Starting them next to phase 1 instead was measured slower on config 1, 6.96 against 6.72 ms per step: the kernels of the
  // two phases evict each other's scratch from the L2.)
  if (ctx->wait_in[1]) CU(cudaStreamWaitEvent(st, ctx->wait_in[1], 0));
  rc = launch_view(ctx, st, vL, ssL, al, 12, ctx->split_rows, n);
  if (rc != ELECTOR_OK) return rc;
  if (ctx->split_rows) {   // the copy stream learns where the linear region starts and ends as soon as its last segment is done
    CU(cudaMemcpyAsync(&ctx->h_totals[6], ctx->d_ctrl.as<unsigned long long>() + 18, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->copy_out));
    CU(cudaEventRecord(ctx->ev_lin, ctx->copy_out));
  }
  CU(cudaEventRecord(ctx->ev_lin_done, st));
  // ---- sort 2 on the linear stream once phase 1 is done (its bulk on `st`, its other segments on side[0 .. 11]) ----
  CU(cudaStreamWaitEvent(sl, ctx->ev_bulk1, 0));
  rc = join_view(ctx, sl, 0, 12, 0);
  if (rc != ELECTOR_OK) return rc;
  CU(cudaEventRecord(ctx->ev_mid, sl));
  rc = sort_view(ctx, sl, v2, (int32_t)n, ss2, rows_cap, false);
  if (rc == ELECTOR_OK) rc = read_plans(ctx, 2, 1, dtab2, sl);   // the host waits for sort 2 alone; the linear segments run meanwhile
  if (rc != ELECTOR_OK) return rc;
  if (ctx->wait_in[1]) CU(cudaStreamWaitEvent(sl, ctx->wait_in[1], 0));
  // ---- the general segments of phase 2: bulk on `st` behind the linear bulk, the others forked from the linear stream
  // (phase 1 and sort 2 are done there), on side[0 .. 11]: they never queue behind a linear segment ----
  rc = launch_view(ctx, st, v2, ss2, ag, 0, false, n, 2, sl);
  if (rc == ELECTOR_OK) rc = join_view(ctx, st, 0, 16, 2);
  if (rc != ELECTOR_OK) return rc;
  CU(cudaMemcpyAsync(ctx->h_bintab, dtab1, 2 * sizeof(BinTable), cudaMemcpyDeviceToHost, st));   // errors and needs of the call
  CU(cudaEventRecord(ctx->ev1, st));
  return ELECTOR_OK;
}

// after the stream has been synchronised: what the tables say.  ELECTOR_OK, an error, or 1 = a scratch pool was too small
// and has been grown: run the call again
int check_tables(elector_ctx *ctx) {
  const BinTable *t1 = ctx->h_bintab, *t2 = ctx->h_bintab + 1;
  if (t1->err_code || t2->err_code) cudaMemsetAsync(ctx->d_ctrl.as<int32_t>() + kAbortWord, 0, sizeof(int32_t), ctx->stream);   // for stand-alone merge / tally calls
  if (t1->err_code == 1) return ctx->fail(ELECTOR_EINVAL, "window %d has an empty sequence (undefined in the reference)", t1->err_window);
  if (t1->err_code == 2) return ctx->fail(ELECTOR_ETOOLARGE, "window %d: a sequence longer than %d letters, or reference + corrected longer than %d (16-bit node indices)", t1->err_window, kMaxWindowLen, kMaxNodes);
  if (t1->err_code == 4 || t2->err_code == 4) return ctx->fail(ELECTOR_ETOOLARGE, "a segment of the call needs %llu MiB of scratch (windows too long)", (unsigned long long)((std::max(t1->need_words, t2->need_words) * 4) >> 20));
  if (t1->err_code == 3 || t2->err_code == 3) {
    const size_t need1 = (size_t)t1->need_words * 4, need2 = (size_t)t2->need_words * 4;
    if (need1 > ((size_t)60 << 30) || need2 > ((size_t)60 << 30)) return ctx->fail(ELECTOR_ETOOLARGE, "call needs %zu MiB of scratch", std::max(need1, need2) >> 20);
    if (need1 > ctx->d_scratch.cap) CU(ctx->d_scratch.reserve(need1));
    if (need2 > ctx->d_scratch_lin.cap) CU(ctx->d_scratch_lin.reserve(need2));   // the two views of table 2 report one maximum
    if (need2 > ctx->d_scratch2.cap) CU(ctx->d_scratch2.reserve(need2));
    return 1;
  }
  return ELECTOR_OK;
}

// adds the device time between ev0 and ev1 (both already reached) to the running total of a call
void add_kernel_ms(elector_ctx *ctx) {
  float ms = 0.f;
  if (ctx->trace) {
    const char *lvl = getenv("ELECTOR_TRACE");
    if (lvl && lvl[0] >= '2') {
#ifdef EL_DP_CLOCKS
      {
        unsigned long long h[2][8], z[2][8] = {};
        cudaMemcpyFromSymbol(h, g_dp_clk, sizeof h);
        cudaMemcpyToSymbol(g_dp_clk, z, sizeof z);
        static const char *ph[8] = {"set-up", "pack", "prepare", "dp", "traceback", "alloc+fuse+emit", "rest", ""};
        for (int k = 0; k < 2; ++k) {
          double tot = 0;
          for (int i = 0; i < 7; ++i) tot += (double)h[k][i];
          fprintf(stderr, "[elector clocks] %s:", k ? "Phase2D" : "Phase2L");
          for (int i = 0; i < 7; ++i) fprintf(stderr, " %s %.1f%%", ph[i], tot > 0 ? 100.0 * h[k][i] / tot : 0.0);
          fprintf(stderr, " (%.3g warp cycles)\n", tot);
        }
      }
#endif
      if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev_mid) == cudaSuccess) fprintf(stderr, "[elector trace]   phase 1 done %.3f ms", ms);
      if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev_lin_done) == cudaSuccess) fprintf(stderr, ", linear segments of phase 2 done %.3f ms", ms);
      if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) fprintf(stderr, ", all done %.3f ms\n", ms);
      static const char *vn[3] = {"phase 1", "phase 2 linear", "phase 2 general"};
      for (int v = 0; v < 3; ++v) {
        float t[4] = {-1, -1, -1, -1};
        for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&t[k], ctx->ev0, ctx->ev_view[v][k >> 1][k & 1]);
        fprintf(stderr, "[elector trace]     %-16s launched at %.3f (cooperative) / %.3f (others), joined at %.3f ms\n", vn[v], t[0], t[2], t[3] > t[1] ? t[3] : t[1]);
      }
    }
  }
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms += ms;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev_mid) == cudaSuccess) ctx->last_ms_phase1 += ms;
  (void)cudaGetLastError();   // an event of a view that did not run this call has no time: not an error of the call
}

// One alignment on ctx's stream, waited for: run_device, the rows cursor read back, check_tables; a run whose scratch pools
// were too small runs again with the grown pools.  d_rows_used (device memory, may be NULL) receives the rows cursor.
int align_device(elector_ctx *ctx, int64_t n, const char *d_ref, const int64_t *d_roff, const char *d_cor, const int64_t *d_coff,
                 const char *d_unc, const int64_t *d_uoff, const int64_t *h_roff, const int64_t *h_coff, char *d_rows, int64_t rows_cap,
                 int64_t *d_rowoff, int32_t *d_stride, int32_t *d_nring, int32_t *d_s1, int32_t *d_s2, int64_t *d_cells, int64_t *d_rows_used) {
  for (int attempt = 0;; ++attempt) {
    int rc = run_device(ctx, n, d_ref, d_roff, d_cor, d_coff, d_unc, d_uoff, h_roff, h_coff, d_rows, rows_cap, d_rowoff, d_stride, d_nring, d_s1, d_s2,
                        d_cells, ctx->d_ctrl.as<unsigned long long>(), ctx->d_ctrl.as<int32_t>() + 2);
    if (rc != ELECTOR_OK) return rc;
    if (d_rows_used) CU(cudaMemcpyAsync(d_rows_used, ctx->d_ctrl.p, sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    CU(cudaMemcpyAsync(&ctx->h_totals[4], ctx->d_ctrl.p, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // the one wait of the alignment
    if (n == 0) return ELECTOR_OK;            // run_device queued nothing: no tables, no times
    rc = check_tables(ctx);
    if (rc == 1 && attempt < kScratchRetries) continue;
    if (rc != ELECTOR_OK) return rc == 1 ? ctx->fail(ELECTOR_ECUDA, "scratch pools keep overflowing") : rc;
    break;
  }
  add_kernel_ms(ctx);
  if ((int32_t)(ctx->h_totals[5] & 0xffffffff)) return ctx->fail(ELECTOR_ECAPACITY, "row buffer capacity %lld too small", (long long)rows_cap);
  return ELECTOR_OK;
}


struct ChunkJob { int64_t w0, w1, r0, r1, rows_base, rows_len, m_base; bool split; int index; };
struct PipeArgs {
  const elector_pipeline_io *io;
  const int64_t *ro, *co, *uo;      // = io->ref_off ...
  bool packed;                      // 2-bit letters + 32-bit offsets on the wire
  cudaEvent_t ev_call;   // start of the call on the device (ELECTOR_TRACE)
  // the chunks' inputs cross PCIe in chunk order (a worker queues its copies when it is its chunk's turn, behind the
  // previous chunk's): chunk 0 computes while chunk 1 is still arriving
  std::atomic<int> *h2d_turn;
  cudaEvent_t *h2d_prev;
  std::atomic<long long> *n_esc;    // escapes of the 4-bit merged rows appended so far (all chunks)
};

// One chunk of a pipelined call on one worker context: everything is queued on the worker's stream (the segment launches
// fork to its side streams) and the function returns when the chunk's results are in the caller's host buffers.  Adds the
// chunk's tally sums to sums; failed (run_pool) ends the wait for an input turn that an earlier chunk will not pass on.
int process_chunk(elector_ctx *ctx, const PipeArgs &pa, const ChunkJob &j, int64_t *sums, const std::atomic<int> &failed) {
  const elector_pipeline_io &io = *pa.io;
  const int64_t w0 = j.w0, w1 = j.w1, nw = w1 - w0, r0 = j.r0, r1 = j.r1, nr = r1 - r0;
  const int64_t first[3] = {pa.ro[w0], pa.co[w0], pa.uo[w0]};
  const int64_t len[3] = {pa.ro[w1] - first[0], pa.co[w1] - first[1], pa.uo[w1] - first[2]};
  const int64_t br0 = first[0], bc0 = first[1], bu0 = first[2], br = len[0], bc = len[1], bu = len[2];
  DevBuf *d_let[3] = {&ctx->d_ref, &ctx->d_cor, &ctx->d_unc};
  DevBuf *d_off[3] = {&ctx->d_roff, &ctx->d_coff, &ctx->d_uoff};
  const int64_t *h_off[3] = {pa.ro, pa.co, pa.uo};
  const char *h_let[3] = {io.ref, io.cor, io.unc};
  const elector_packed *h_pk[3] = {io.pref, io.pcor, io.punc};
  for (int k = 0; k < 3; ++k) { CU(d_let[k]->reserve(len[k] + 8)); CU(d_off[k]->reserve((nw + 1) * 8)); }
  CU(ctx->d_rows.reserve(j.rows_len)); CU(ctx->d_rowoff.reserve(nw * 8)); CU(ctx->d_stride.reserve(nw * 4));
  CU(ctx->d_nring.reserve(nw * 4)); CU(ctx->d_s1.reserve(nw * 4)); CU(ctx->d_s2.reserve(nw * 4)); CU(ctx->d_cells.reserve(nw * 8));
  if (nr > 0) { CU(ctx->d_tally_out.reserve(nr * ELECTOR_TALLY_K * 8)); CU(ctx->d_sums.reserve(ELECTOR_TALLY_K * 8)); }
  // compact wire format: the 32-bit offsets of the chunk (relative to its first letter) are made here, on the worker's
  // thread, while the chunks before it are on their way; the exceptions of the chunk are found by binary search
  int64_t exc0[3] = {0, 0, 0}, exc1[3] = {0, 0, 0};
  int32_t *stage = nullptr;
  bool use_len = false;
  if (pa.packed) {
    const size_t need = (size_t)3 * (nw + 1) * sizeof(int32_t);
    if (need > ctx->h_stage_cap) {
      if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
      ctx->h_stage = nullptr; ctx->h_stage_cap = 0;
      CU(cudaMallocHost(&ctx->h_stage, need + need / 4));
      ctx->h_stage_cap = need + need / 4;
    }
    stage = static_cast<int32_t *>(ctx->h_stage);
    const int32_t *h_len[3] = {io.ref_len, io.cor_len, io.unc_len};
    const bool len16 = io.ref_len16 && io.cor_len16 && io.unc_len16;
    use_len = ((h_len[0] && h_len[1] && h_len[2]) || len16) && nw <= 1024 * 1024;   // the caller's 32-bit (or 16-bit) lengths cross the link as they are
    for (int k = 0; k < 3; ++k) {
      if (len[k] > 0x7fffffff) return ctx->fail(ELECTOR_ETOOLARGE, "a chunk holds more than 2^31 letters of one kind");
      if (!use_len) {
        int32_t *dst = stage + (size_t)k * (nw + 1);
        const int64_t *src = h_off[k] + w0, f = first[k];
        for (int64_t i = 0; i <= nw; ++i) dst[i] = (int32_t)(src[i] - f);
      }
      const int64_t *ep = h_pk[k]->exc_pos, ne = h_pk[k]->n_exc;
      exc0[k] = std::lower_bound(ep, ep + ne, first[k]) - ep;
      exc1[k] = std::lower_bound(ep, ep + ne, first[k] + len[k]) - ep;
      CU(ctx->d_pk[k].reserve((size_t)(len[k] / 4 + 8)));
    }
    CU(ctx->d_rel.reserve(need + 3 * 1032 * sizeof(long long) + (size_t)3 * (nw + 4) * sizeof(uint16_t)));
    const int64_t ne_tot = (exc1[0] - exc0[0]) + (exc1[1] - exc0[1]) + (exc1[2] - exc0[2]);
    CU(ctx->d_exc_pos.reserve((size_t)(ne_tot + 1) * 8)); CU(ctx->d_exc_byte.reserve((size_t)ne_tot + 8));
  }
  cudaStream_t st = ctx->stream;
  while (pa.h2d_turn->load(std::memory_order_acquire) != j.index) {
    if (failed.load() != ELECTOR_OK) return ctx->fail(ELECTOR_ECUDA, "another chunk of the call failed");
    std::this_thread::yield();
  }
  struct PassTurn {   // whatever happens below, the next chunk gets its turn
    const PipeArgs &pa; int next; bool passed;
    void pass() { if (!passed) { passed = true; pa.h2d_turn->store(next, std::memory_order_release); } }
    ~PassTurn() { pass(); }
  } pass_turn{pa, j.index + 1, false};
  if (*pa.h2d_prev) CU(cudaStreamWaitEvent(st, *pa.h2d_prev, 0));
  if (ctx->trace) CU(cudaEventRecord(ctx->uev0, st));
  // the offsets first, on the compute stream: the size sort needs nothing else.  The letters follow on the copy stream --
  // ref and cor (phase 1 waits for them), then unc (phase 2 waits for it) -- while the sort and phase 1 run.
  if (pa.packed && use_len) {   // 32-bit lengths in, added up on the device
    const int32_t *h_len[3] = {io.ref_len, io.cor_len, io.unc_len};
    const uint16_t *h_len16[3] = {io.ref_len16, io.cor_len16, io.unc_len16};
    const bool len16 = h_len16[0] && h_len16[1] && h_len16[2];
    const int nblocks = (int)((nw + 1023) / 1024);
    long long *totals = reinterpret_cast<long long *>(ctx->d_rel.as<int32_t>() + (size_t)3 * (nw + 1) + ((nw + 1) & 1));
    uint16_t *d16 = reinterpret_cast<uint16_t *>(totals + 3 * 1032);
    for (int k = 0; k < 3; ++k) {
      int32_t *dl = ctx->d_rel.as<int32_t>() + (size_t)k * (nw + 1);
      if (len16) {
        uint16_t *dk = d16 + (size_t)k * (nw + 4);
        CU(cudaMemcpyAsync(dk, h_len16[k] + w0, (size_t)nw * 2, cudaMemcpyHostToDevice, st));
        widen_len16_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(nw, dk, dl);
      } else
        CU(cudaMemcpyAsync(dl, h_len[k] + w0, (size_t)nw * 4, cudaMemcpyHostToDevice, st));
      len_scan_blocks_kernel<<<nblocks, 1024, 0, st>>>(nw, dl, totals + (size_t)k * 1032);
      len_scan_totals_kernel<<<1, 1024, 0, st>>>(nblocks, totals + (size_t)k * 1032);
      len_to_offsets_kernel<<<(unsigned)((nw + 256) / 256), 256, 0, st>>>(nw, dl, totals + (size_t)k * 1032, nblocks, first[k], d_off[k]->as<int64_t>());
    }
    CU(cudaGetLastError());
    ctx->last_launches += 9;
  } else if (pa.packed) {
    CU(cudaMemcpyAsync(ctx->d_rel.p, stage, (size_t)3 * (nw + 1) * 4, cudaMemcpyHostToDevice, st));
    for (int k = 0; k < 3; ++k)
      widen_offsets_kernel<<<(unsigned)((nw + 256) / 256), 256, 0, st>>>(nw + 1, ctx->d_rel.as<int32_t>() + (size_t)k * (nw + 1), first[k], d_off[k]->as<int64_t>());
    CU(cudaGetLastError());
    ctx->last_launches += 3;
  } else
    for (int k = 0; k < 3; ++k) CU(cudaMemcpyAsync(d_off[k]->p, h_off[k] + w0, (nw + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaEventRecord(ctx->ev_fork, st));
  CU(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_fork, 0));   // the copy engine serves the offsets first
  int64_t exc_done = 0;
  for (int k = 0; k < 3; ++k) {
    if (pa.packed) {   // packed bytes that hold the chunk's letters (+ one of padding), expanded on the device; then the exceptions
      const int64_t b0 = first[k] >> 2, b1 = (first[k] + len[k] + 3) >> 2;
      const int64_t have = (h_pk[k]->n_letters + 3) >> 2;
      CU(cudaMemcpyAsync(ctx->d_pk[k].p, h_pk[k]->bits + b0, (size_t)std::min(b1 + 1, have) - b0, cudaMemcpyHostToDevice, ctx->copy_in));
      if (len[k] > 0) unpack2_kernel<<<(unsigned)std::min<int64_t>((len[k] / 4 + 256) / 256, (int64_t)ctx->sm_count * 16), 256, 0, ctx->copy_in>>>(
          ctx->d_pk[k].as<uint8_t>(), (int)(first[k] & 3), len[k], d_let[k]->as<uint8_t>());
      const int64_t ne = exc1[k] - exc0[k];
      if (ne > 0) {
        CU(cudaMemcpyAsync(ctx->d_exc_pos.as<int64_t>() + exc_done, h_pk[k]->exc_pos + exc0[k], ne * 8, cudaMemcpyHostToDevice, ctx->copy_in));
        CU(cudaMemcpyAsync(ctx->d_exc_byte.as<uint8_t>() + exc_done, h_pk[k]->exc_byte + exc0[k], ne, cudaMemcpyHostToDevice, ctx->copy_in));
        patch_letters_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, ctx->copy_in>>>(ne, ctx->d_exc_pos.as<int64_t>() + exc_done, ctx->d_exc_byte.as<uint8_t>() + exc_done,
                                                                                   first[k], d_let[k]->as<uint8_t>());
        exc_done += ne;
      }
      CU(cudaGetLastError());
      ctx->last_launches += ne > 0 ? 2 : 1;
    } else
      CU(cudaMemcpyAsync(d_let[k]->p, h_let[k] + first[k], len[k], cudaMemcpyHostToDevice, ctx->copy_in));
    if (k >= 1) CU(cudaEventRecord(ctx->ev_in[k - 1], ctx->copy_in));
  }
  ctx->wait_in[0] = ctx->ev_in[0]; ctx->wait_in[1] = ctx->ev_in[1];
  *pa.h2d_prev = ctx->ev_in[1];
  pass_turn.pass();
  // the offsets stay those of the whole call: the letter pointers are moved back by the chunk's first offset, the row
  // pointer by the chunk's base in the caller's row buffer (row_off[] then indexes the caller's buffer directly)
  char *d_rows_v = ctx->d_rows.as<char>() - j.rows_base;
  cudaStream_t so = ctx->copy_out;
  const bool want_rows = io.rows_out != nullptr;
  const bool want_merged = io.m_ref != nullptr;
  for (int attempt = 0;; ++attempt) {
    ctx->split_rows = j.split && want_rows;
    int rc = run_device(ctx, nw, ctx->d_ref.as<char>() - br0, ctx->d_roff.as<int64_t>(), ctx->d_cor.as<char>() - bc0, ctx->d_coff.as<int64_t>(),
                        ctx->d_unc.as<char>() - bu0, ctx->d_uoff.as<int64_t>(), pa.ro + w0, pa.co + w0, d_rows_v, j.rows_base + j.rows_len,
                        ctx->d_rowoff.as<int64_t>(), ctx->d_stride.as<int32_t>(), ctx->d_nring.as<int32_t>(), ctx->d_s1.as<int32_t>(),
                        ctx->d_s2.as<int32_t>(), ctx->d_cells.as<int64_t>(), ctx->d_ctrl.as<unsigned long long>(), ctx->d_ctrl.as<int32_t>() + 2, j.rows_base);
    const bool split = ctx->split_rows;
    ctx->split_rows = false;
    if (rc != ELECTOR_OK) { ctx->wait_in[0] = ctx->wait_in[1] = nullptr; cudaStreamSynchronize(ctx->copy_in); cudaStreamSynchronize(st); return rc; }
    CU(cudaMemcpyAsync(&ctx->h_totals[4], ctx->d_ctrl.p, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(ctx->ev_rows, st));
    if (nr > 0) {
      std::vector<int64_t> rf(io.read_first + r0, io.read_first + r1 + 1);
      for (int64_t &v : rf) v -= w0;
      CU(cudaMemsetAsync(ctx->d_sums.p, 0, ELECTOR_TALLY_K * 8, st));
      rc = merge_device(ctx, nr, rf.data(), nw, reinterpret_cast<const uint8_t *>(d_rows_v), 3 * (br + bc + bu), ctx->d_rowoff.as<int64_t>(),
                        ctx->d_stride.as<int32_t>(), ctx->d_nring.as<int32_t>());
      if (rc != ELECTOR_OK) { ctx->wait_in[0] = ctx->wait_in[1] = nullptr; cudaStreamSynchronize(st); return rc; }
      // the merged rows are packed and on their way before the tally runs: the copy stream takes them while the tally kernels run
      if (want_merged && io.m_nibbles == 2) {   // one byte per column for the three rows together; characters outside the code go to the escape list
        CU(ctx->d_nib[0].reserve((size_t)ctx->merged_cap + 16));
        CU(ctx->d_esc_pos.reserve((size_t)(io.m_esc_cap + 3) * 8)); CU(ctx->d_esc_byte.reserve((size_t)io.m_esc_cap + 8));
        CU(cudaMemsetAsync(ctx->d_ctrl.as<unsigned long long>() + 21, 0, 8, st));
        column_pack_kernel<<<(unsigned)nr, 128, 0, st>>>(nr, ctx->d_mref.as<uint8_t>(), ctx->d_mcor.as<uint8_t>(), ctx->d_munc.as<uint8_t>(),
            ctx->d_moff.as<int64_t>(), ctx->d_mlen.as<int32_t>(), ctx->d_nib[0].as<uint8_t>(), j.m_base,
            ctx->d_ctrl.as<unsigned long long>() + 21, ctx->d_esc_pos.as<int64_t>(), ctx->d_esc_byte.as<uint8_t>(), io.m_esc_cap, ctx->d_ctrl.as<int32_t>() + kAbortWord);
        CU(cudaGetLastError());
        ++ctx->last_launches;
      } else if (want_merged && io.m_nibbles) {   // two columns per byte before they leave; the few characters outside the code go to the escape list
        for (int k = 0; k < 3; ++k) CU(ctx->d_nib[k].reserve((size_t)ctx->merged_cap / 2 + 16));
        CU(ctx->d_esc_pos.reserve((size_t)(io.m_esc_cap + 1) * 8)); CU(ctx->d_esc_byte.reserve((size_t)io.m_esc_cap + 8));
        CU(cudaMemsetAsync(ctx->d_ctrl.as<unsigned long long>() + 21, 0, 8, st));
        nibble_pack_kernel<<<(unsigned)((3 * nr + 3) / 4), 128, 0, st>>>(nr, ctx->d_mref.as<uint8_t>(), ctx->d_mcor.as<uint8_t>(), ctx->d_munc.as<uint8_t>(),
            ctx->d_moff.as<int64_t>(), ctx->d_mlen.as<int32_t>(), ctx->d_nib[0].as<uint8_t>(), ctx->d_nib[1].as<uint8_t>(), ctx->d_nib[2].as<uint8_t>(), j.m_base,
            ctx->d_ctrl.as<unsigned long long>() + 21, ctx->d_esc_pos.as<int64_t>(), ctx->d_esc_byte.as<uint8_t>(), io.m_esc_cap, ctx->d_ctrl.as<int32_t>() + kAbortWord);
        CU(cudaGetLastError());
        ++ctx->last_launches;
      }
      CU(cudaMemcpyAsync(&ctx->h_totals[2], ctx->d_moff.as<int64_t>() + nr, sizeof(int64_t), cudaMemcpyDeviceToHost, st));      // merged columns of the chunk
      CU(cudaMemcpyAsync(&ctx->h_totals[3], ctx->d_ctrl.as<unsigned long long>() + 21, sizeof(int64_t), cudaMemcpyDeviceToHost, st));   // escapes
      CU(cudaEventRecord(ctx->ev_merged, st));
      rc = tally_device(ctx, nr, ctx->d_mref.as<uint8_t>(), ctx->d_mcor.as<uint8_t>(), ctx->d_munc.as<uint8_t>(), ctx->d_moff.as<int64_t>(),
                        ctx->d_mlen.as<int32_t>(), ctx->d_tally_out.as<int64_t>(), ctx->merged_cap);
      if (rc != ELECTOR_OK) { ctx->wait_in[0] = ctx->wait_in[1] = nullptr; cudaStreamSynchronize(st); return rc; }
      tally_sum_kernel<<<std::min<int>(64, (int)((nr + 7) / 8)), 256, 0, st>>>(nr, ctx->d_tally_out.as<int64_t>(), ctx->d_sums.as<unsigned long long>());
      CU(cudaGetLastError());
      ++ctx->last_launches;
      CU(cudaEventRecord(ctx->ev1, st));   // the chunk's device time covers merge + tally too
      CU(cudaMemcpyAsync(ctx->h_sums, ctx->d_sums.p, ELECTOR_TALLY_K * 8, cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(ctx->h_sums + ELECTOR_TALLY_K, ctx->d_ctrl.as<int32_t>() + 3, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      if (io.counters_out) CU(cudaMemcpyAsync(io.counters_out + r0 * ELECTOR_TALLY_K, ctx->d_tally_out.p, nr * ELECTOR_TALLY_K * 8, cudaMemcpyDeviceToHost, st));
      if (io.m_off) CU(cudaMemcpyAsync(io.m_off + r0, ctx->d_moff.p, nr * 8, cudaMemcpyDeviceToHost, st));
      if (io.m_len) CU(cudaMemcpyAsync(io.m_len + r0, ctx->d_mlen.p, nr * 4, cudaMemcpyDeviceToHost, st));
    }
    // the alignment results leave on the copy stream while merge and tally run: the host waits for the POA kernels only
    // to learn how many row bytes the chunk used.  The linear region first: its segments run next to phase 1 and finish early.
    const int64_t end_b = j.rows_base + j.rows_len;
    int64_t base_b = end_b, used_b = end_b;
    if (split) {
      CU(cudaEventSynchronize(ctx->ev_lin));
      used_b = ctx->h_totals[6]; base_b = ctx->h_totals[7];
      if (base_b >= j.rows_base && used_b > base_b && used_b <= end_b)
        CU(cudaMemcpyAsync(io.rows_out + base_b, d_rows_v + base_b, used_b - base_b, cudaMemcpyDeviceToHost, so));
    }
    CU(cudaEventSynchronize(ctx->ev_rows));
    ctx->wait_in[0] = ctx->wait_in[1] = nullptr;   // the letters have arrived: a second attempt does not wait for them again
    rc = check_tables(ctx);
    if (rc == 1 && attempt < kScratchRetries) {   // a scratch pool was too small (first call, or longer windows than before): grown, run the chunk again
      CU(cudaStreamSynchronize(st));
      CU(cudaStreamSynchronize(so));
      if (ctx->trace) fprintf(stderr, "[elector trace] chunk w%lld: scratch pools grown to %zu / %zu / %zu MiB, running it again\n", (long long)w0,
                              ctx->d_scratch.cap >> 20, ctx->d_scratch_lin.cap >> 20, ctx->d_scratch2.cap >> 20);
      continue;
    }
    if (rc != ELECTOR_OK) { cudaStreamSynchronize(st); cudaStreamSynchronize(so); return rc == 1 ? ctx->fail(ELECTOR_ECUDA, "scratch pools keep overflowing") : rc; }
    const int64_t used = ctx->h_totals[4];
    if ((int32_t)(ctx->h_totals[5] & 0xffffffff) || used > base_b || used_b > end_b) {
      cudaStreamSynchronize(st);
      cudaStreamSynchronize(so);
      return ctx->fail(ELECTOR_ECAPACITY, "rows of a chunk exceed their bound (%lld + %lld > %lld)", (long long)(used - j.rows_base), (long long)(used_b - base_b),
                       (long long)j.rows_len);
    }
    if (want_rows) {
      CU(cudaMemcpyAsync(io.rows_out + j.rows_base, ctx->d_rows.p, used - j.rows_base, cudaMemcpyDeviceToHost, so));
      CU(cudaMemcpyAsync(io.row_off + w0, ctx->d_rowoff.p, nw * 8, cudaMemcpyDeviceToHost, so));
      CU(cudaMemcpyAsync(io.row_stride + w0, ctx->d_stride.p, nw * 4, cudaMemcpyDeviceToHost, so));
    }
    if (io.nring) CU(cudaMemcpyAsync(io.nring + w0, ctx->d_nring.p, nw * 4, cudaMemcpyDeviceToHost, so));
    if (io.score1) CU(cudaMemcpyAsync(io.score1 + w0, ctx->d_s1.p, nw * 4, cudaMemcpyDeviceToHost, so));
    if (io.score2) CU(cudaMemcpyAsync(io.score2 + w0, ctx->d_s2.p, nw * 4, cudaMemcpyDeviceToHost, so));
    if (io.cells) CU(cudaMemcpyAsync(io.cells + w0, ctx->d_cells.p, nw * 8, cudaMemcpyDeviceToHost, so));
    if (nr > 0 && want_merged) {   // the merged rows: their size is known once the merge has run
      CU(cudaEventSynchronize(ctx->ev_merged));
      const int64_t cols = ctx->h_totals[2];
      if (j.m_base + cols > io.m_cap) { cudaStreamSynchronize(st); cudaStreamSynchronize(so); return ctx->fail(ELECTOR_ECAPACITY, "merged rows need more than m_cap = %lld columns", (long long)io.m_cap); }
      char *dst[3] = {io.m_ref, io.m_cor, io.m_unc};
      DevBuf *srcb[3] = {&ctx->d_mref, &ctx->d_mcor, &ctx->d_munc};
      if (io.m_nibbles == 2) CU(cudaMemcpyAsync(dst[0] + j.m_base, ctx->d_nib[0].p, (size_t)cols, cudaMemcpyDeviceToHost, so));
      else for (int k = 0; k < 3; ++k) {
        if (io.m_nibbles) CU(cudaMemcpyAsync(dst[k] + j.m_base / 2, ctx->d_nib[k].p, (size_t)(cols + 1) / 2, cudaMemcpyDeviceToHost, so));
        else CU(cudaMemcpyAsync(dst[k] + j.m_base, srcb[k]->p, (size_t)cols, cudaMemcpyDeviceToHost, so));
      }
      if (io.m_nibbles) {
        const int64_t ne = ctx->h_totals[3];
        if (ne > 0) {
          const long long at = pa.n_esc->fetch_add(ne);
          if (at + ne > io.m_esc_cap || ne > io.m_esc_cap) { cudaStreamSynchronize(st); cudaStreamSynchronize(so); return ctx->fail(ELECTOR_ECAPACITY, "more than m_esc_cap = %lld characters outside the 4-bit code", (long long)io.m_esc_cap); }
          CU(cudaMemcpyAsync(io.m_esc_pos + at, ctx->d_esc_pos.p, (size_t)ne * 8, cudaMemcpyDeviceToHost, so));
          CU(cudaMemcpyAsync(io.m_esc_byte + at, ctx->d_esc_byte.p, (size_t)ne, cudaMemcpyDeviceToHost, so));
        }
      }
    }
    if (ctx->trace) CU(cudaEventRecord(ctx->uev1, so));
    CU(cudaStreamSynchronize(st));
    CU(cudaStreamSynchronize(so));
    if (nr > 0 && io.m_off) for (int64_t r = r0; r < r1; ++r) io.m_off[r] += j.m_base;   // chunk-relative -> the caller's buffers
    break;
  }
  if (ctx->trace) {   // device timeline of the chunk, ms after the start of the call
    float t[6] = {0, 0, 0, 0, 0, 0};
    cudaEventElapsedTime(&t[0], pa.ev_call, ctx->uev0); cudaEventElapsedTime(&t[1], pa.ev_call, ctx->ev0);
    cudaEventElapsedTime(&t[2], pa.ev_call, ctx->ev_mid); cudaEventElapsedTime(&t[3], pa.ev_call, ctx->ev_rows);
    cudaEventElapsedTime(&t[4], pa.ev_call, ctx->ev1); cudaEventElapsedTime(&t[5], pa.ev_call, ctx->uev1);
    fprintf(stderr, "[elector trace] chunk w%lld: h2d %.2f | sort1 %.2f | phase 1 done %.2f | phase 2 done %.2f | merge+tally done %.2f | results on host %.2f\n",
            (long long)w0, t[0], t[1], t[2], t[3], t[4], t[5]);
    (void)cudaGetLastError();
  }
  add_kernel_ms(ctx);
  if (nr > 0) {
    if ((int32_t)ctx->h_sums[ELECTOR_TALLY_K]) {
      cudaMemsetAsync(ctx->d_ctrl.as<int32_t>() + 3, 0, sizeof(int32_t), st);
      return ctx->fail(ELECTOR_EUNSUPPORTED, "a read has more than %d gap stretches at its borders", kMaxStretchKeys);
    }
    for (int f = 0; f < ELECTOR_TALLY_K; ++f) sums[f] += ctx->h_sums[f];
  }
  return ELECTOR_OK;
}

int create_context(int device, const ScoreMatrix &mat, elector_ctx **out, int worker = 0);

}  // namespace

extern "C" {

int elector_poa_init(int device, const char *matrix_path, elector_ctx **out) {
  if (!out) return ELECTOR_EINVAL;
  *out = nullptr;
  ScoreMatrix mat;
  if (matrix_path) {
    if (mat.load(matrix_path) <= 0) {
      char buf[512];
      snprintf(buf, sizeof buf, "Error reading matrix file %s", matrix_path);
      g_init_error = buf;
      return ELECTOR_EMATRIX;
    }
  } else mat.set_default();
  return create_context(device, mat, out);
}

}  // extern "C"

namespace {
// a context for `device` with the scoring of `mat` (elector_poa_init; worker contexts of the pipelined entry point).
// worker k > 0: its streams get a lower priority than those of worker k - 1 -- the chunks of a pipelined call then finish one
// after the other instead of all together, and the results of one leave while the next computes.
int create_context(int device, const ScoreMatrix &mat, elector_ctx **out, int worker) {
  elector_ctx *ctx = new elector_ctx();
  auto bail = [&](int code) {
    g_init_error = ctx->err;
    elector_poa_free(ctx);
    return code;
  };
  ctx->mat = mat;
  if (!ctx->sc.analyse(ctx->mat)) { ctx->err = ctx->sc.error; return bail(ELECTOR_EUNSUPPORTED); }
  ctx->trace = getenv("ELECTOR_TRACE") != nullptr;
  if (const char *e = getenv("ELECTOR_BAND_W")) ctx->band_w = std::max(0, std::min(64, atoi(e)));
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    ctx->fail(ELECTOR_ECUDA, "no CUDA device available (%s); this library has no CPU path", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return bail(ELECTOR_ECUDA);
  }
  if (device < 0 || device >= ndev) { ctx->fail(ELECTOR_EINVAL, "device %d out of range (0..%d)", device, ndev - 1); return bail(ELECTOR_EINVAL); }
  ctx->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess) { ctx->fail(ELECTOR_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); return bail(ELECTOR_ECUDA); }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // numerically lower = higher priority
  const int prio = std::min(prio_lo, prio_hi + worker);
  if ((e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_mid)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_split0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_split1)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_mt0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_mt1)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_rows)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_lin, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_merged, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_in[0], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_in[1], cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->uev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->uev1)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_call)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaStreamCreateWithPriority(&ctx->lin_stream, cudaStreamNonBlocking, prio)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_sorted, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev_lin_done)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_lin_sorted, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_bulk1, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMallocHost((void **)&ctx->h_bintab, 2 * sizeof(BinTable))) != cudaSuccess ||
      (e = cudaMallocHost((void **)&ctx->h_plan, 2 * sizeof(BinTable))) != cudaSuccess ||
      (e = cudaMallocHost((void **)&ctx->h_totals, 8 * sizeof(int64_t))) != cudaSuccess ||
      (e = cudaMallocHost((void **)&ctx->h_sums, (ELECTOR_TALLY_K + 1) * sizeof(int64_t))) != cudaSuccess ||
      (e = ctx->d_tab.reserve(sizeof(SymbolTables))) != cudaSuccess ||
      (e = ctx->d_ctrl.reserve(kCtrlWords * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMemset(ctx->d_ctrl.p, 0, kCtrlWords * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMemcpy(ctx->d_tab.p, &ctx->sc.tab, sizeof(SymbolTables), cudaMemcpyHostToDevice)) != cudaSuccess) {
    ctx->fail(ELECTOR_ECUDA, "context setup: %s", cudaGetErrorString(e));
    return bail(ELECTOR_ECUDA);
  }
  for (int k = 0; k < 12; ++k) cudaEventCreate(&ctx->ev_view[k / 4][(k / 2) & 1][k & 1]);
  for (int k = 0; k < 6; ++k)
    if ((e = cudaEventCreateWithFlags(&ctx->ev_fork_v[k], cudaEventDisableTiming)) != cudaSuccess) {
      ctx->fail(ELECTOR_ECUDA, "context setup: %s", cudaGetErrorString(e));
      return bail(ELECTOR_ECUDA);
    }
  for (int k = 0; k < kSideStreams; ++k)
    if ((e = cudaStreamCreateWithPriority(&ctx->side[k], cudaStreamNonBlocking, prio)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->ev_join[k], cudaEventDisableTiming)) != cudaSuccess) {
      ctx->fail(ELECTOR_ECUDA, "context setup: %s", cudaGetErrorString(e));
      return bail(ELECTOR_ECUDA);
    }
  if (ctx->sc.generic_sub) resident_warps_per_sm<true>(ctx, prop.sharedMemPerMultiprocessor);
  else resident_warps_per_sm<false>(ctx, prop.sharedMemPerMultiprocessor);
  if (const char *e = getenv("ELECTOR_COOP_GROUP")) ctx->coop_group = std::max(0, std::min(32, atoi(e)));
  if (ctx->resident_coop < 1) ctx->coop_group = 0;
  if (ctx->trace)
    fprintf(stderr, "[elector trace] resident warps / arena bytes per warp: Phase1P %d / %d, Phase2L %d / %d, Phase2D %d / %d, Phase1 %d / %d, Phase2 %d / %d, coop %d\n",
            ctx->resident_ph1p, ctx->arena_ph1p, ctx->resident_ph2l, ctx->arena_ph2l, ctx->resident_ph2d, ctx->arena_ph2d, ctx->resident_ph1, ctx->arena_ph1,
            ctx->resident_ph2, ctx->arena_ph2, ctx->resident_coop);
  if (ctx->resident_ph1 < 1 || ctx->resident_ph2 < 1) { ctx->fail(ELECTOR_ECUDA, "POA kernel does not fit on this device"); return bail(ELECTOR_ECUDA); }
  *out = ctx;
  return ELECTOR_OK;
}

// The worker contexts of a pipelined call: per_device contexts on every one of `devices` (a device may be listed more than
// once), max_slots in all at most.  On ctx's device the first is ctx and the k-th after it ctx->workers[k - 1]; on other devices
// they are ctx->peers.  Missing ones are created here and kept until elector_poa_free.
int worker_slots(elector_ctx *ctx, const std::vector<int> &devices, int per_device, size_t max_slots, std::vector<elector_ctx *> &slots) {
  slots.clear();
  for (size_t i = 0; i < devices.size() && slots.size() < max_slots; ++i)
    for (int w = 0; w < per_device && slots.size() < max_slots; ++w) {
      int used = 0;   // contexts of this device already taken by earlier slots
      for (elector_ctx *s : slots) used += s->device == devices[i];
      elector_ctx *wk = nullptr;
      if (devices[i] == ctx->device) {
        while ((int)ctx->workers.size() < used) {
          elector_ctx *child = nullptr;
          const int rc = create_context(ctx->device, ctx->mat, &child, (int)ctx->workers.size() + 1);
          if (rc != ELECTOR_OK) return ctx->fail(rc, "worker context: %s", g_init_error.c_str());
          ctx->workers.push_back(child);
        }
        wk = used == 0 ? ctx : ctx->workers[(size_t)used - 1];
      } else {
        int seen = 0;
        for (elector_ctx *p : ctx->peers)
          if (p->device == devices[i] && seen++ == used) { wk = p; break; }
        if (!wk) {
          const int rc = create_context(devices[i], ctx->mat, &wk, used);
          cudaSetDevice(ctx->device);
          if (rc != ELECTOR_OK) return ctx->fail(rc, "worker context on device %d: %s", devices[i], g_init_error.c_str());
          ctx->peers.push_back(wk);
        }
      }
      slots.push_back(wk);
    }
  return ELECTOR_OK;
}

// Runs body(worker, slot, chunk, sums, failed) for the chunks 0 .. n_chunks - 1 of a pipelined call on the worker contexts
// `slots`: slot 0 on the calling thread, every other slot on a thread of its own, each taking the next chunk until none is left
// or a chunk has failed.  The body adds its chunk's tally sums to `sums` (the slot's own) and returns an error code; `failed`
// lets a body that waits for another chunk see that the call has failed.  The first error wins: its code is returned and its
// message is in ctx->err.  The device times and launch counts of the slots are summed into ctx; sums_out (may be NULL)
// receives the tally sums of a call without error.  The calling thread is back on ctx's device afterwards.
template <class Body>
int run_pool(elector_ctx *ctx, const std::vector<elector_ctx *> &slots, size_t n_chunks, int64_t *sums_out, Body body) {
  std::atomic<size_t> next{0};
  std::atomic<int> failed{ELECTOR_OK};
  int first = -1;   // slot of the first error: written by the one thread that sets `failed`, read after the join
  std::vector<int64_t> sums(slots.size() * ELECTOR_TALLY_K, 0);
  auto work = [&](int id) {
    elector_ctx *wk = slots[(size_t)id];
    wk->trace = ctx->trace;
    wk->last_ms = wk->last_ms_phase1 = wk->last_ms_split = wk->last_ms_tally = 0.f;
    wk->last_launches = 0;
    int rc = cudaSetDevice(wk->device) == cudaSuccess ? ELECTOR_OK : wk->fail(ELECTOR_ECUDA, "cudaSetDevice(%d) failed", wk->device);
    while (rc == ELECTOR_OK) {
      const size_t k = next.fetch_add(1);
      if (k >= n_chunks || failed.load() != ELECTOR_OK) break;
      rc = body(wk, id, k, &sums[(size_t)id * ELECTOR_TALLY_K], failed);
    }
    int ok = ELECTOR_OK;
    if (rc != ELECTOR_OK && failed.compare_exchange_strong(ok, rc)) first = id;
  };
  std::vector<std::thread> threads;
  for (size_t i = 1; i < slots.size(); ++i) threads.emplace_back(work, (int)i);
  work(0);
  for (std::thread &t : threads) t.join();
  cudaSetDevice(ctx->device);
  float ms = 0.f, ms_phase1 = 0.f, ms_split = 0.f, ms_tally = 0.f;
  int launches = 0;
  for (const elector_ctx *wk : slots) {
    ms += wk->last_ms; ms_phase1 += wk->last_ms_phase1; ms_split += wk->last_ms_split; ms_tally += wk->last_ms_tally; launches += wk->last_launches;
  }
  ctx->last_ms = ms; ctx->last_ms_phase1 = ms_phase1; ctx->last_ms_split = ms_split; ctx->last_ms_tally = ms_tally; ctx->last_launches = launches;
  if (first >= 0) {
    if (slots[(size_t)first] != ctx) ctx->err = slots[(size_t)first]->err;
    return failed.load();
  }
  if (sums_out)
    for (int f = 0; f < ELECTOR_TALLY_K; ++f) {
      sums_out[f] = 0;
      for (size_t i = 0; i < slots.size(); ++i) sums_out[f] += sums[i * ELECTOR_TALLY_K + (size_t)f];
    }
  return ELECTOR_OK;
}
}  // namespace

extern "C" {

void elector_split_release(elector_ctx *ctx);
void elector_poa_free(elector_ctx *ctx) {
  if (!ctx) return;
  elector_split_release(ctx);
  for (elector_ctx *w : ctx->workers) elector_poa_free(w);
  ctx->workers.clear();
  for (elector_ctx *w : ctx->peers) { cudaSetDevice(w->device); elector_poa_free(w); }   // their buffers and streams belong to their device
  if (!ctx->peers.empty()) cudaSetDevice(ctx->device);
  ctx->peers.clear();
  if (ctx->h_sums) cudaFreeHost(ctx->h_sums);
  DevBuf *bufs[] = {&ctx->d_tab, &ctx->d_ref, &ctx->d_cor, &ctx->d_unc, &ctx->d_roff, &ctx->d_coff, &ctx->d_uoff,
                    &ctx->d_items, &ctx->d_scratch, &ctx->d_scratch_lin, &ctx->d_scratch2, &ctx->d_ctrl, &ctx->d_hist, &ctx->d_bintab, &ctx->d_key, &ctx->d_key2, &ctx->d_n1, &ctx->d_p1, &ctx->d_rows, &ctx->d_rowoff, &ctx->d_stride,
                    &ctx->d_nring, &ctx->d_s1, &ctx->d_s2, &ctx->d_cells, &ctx->d_wdst, &ctx->d_sums, &ctx->d_stretch, &ctx->d_tally_scan, &ctx->d_tally_out,
                    &ctx->d_readfirst, &ctx->d_mtot, &ctx->d_moff, &ctx->d_mlen, &ctx->d_mref, &ctx->d_mcor, &ctx->d_munc};
  for (DevBuf *b : bufs) b->release();
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->ev_mid) cudaEventDestroy(ctx->ev_mid);
  for (cudaEvent_t ev : {ctx->ev_split0, ctx->ev_split1, ctx->ev_mt0, ctx->ev_mt1}) if (ev) cudaEventDestroy(ev);
  if (ctx->ev_rows) cudaEventDestroy(ctx->ev_rows);
  for (int k = 0; k < 2; ++k) if (ctx->ev_in[k]) cudaEventDestroy(ctx->ev_in[k]);
  if (ctx->ev_lin) cudaEventDestroy(ctx->ev_lin);
  if (ctx->ev_merged) cudaEventDestroy(ctx->ev_merged);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  for (DevBuf *b : {&ctx->d_pk[0], &ctx->d_pk[1], &ctx->d_pk[2], &ctx->d_nib[0], &ctx->d_nib[1], &ctx->d_nib[2], &ctx->d_exc_pos, &ctx->d_exc_byte, &ctx->d_rel, &ctx->d_esc_pos, &ctx->d_esc_byte}) b->release();
  if (ctx->uev0) cudaEventDestroy(ctx->uev0);
  if (ctx->uev1) cudaEventDestroy(ctx->uev1);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_sorted) cudaEventDestroy(ctx->ev_sorted);
  if (ctx->ev_lin_done) cudaEventDestroy(ctx->ev_lin_done);
  for (int k = 0; k < 6; ++k) if (ctx->ev_fork_v[k]) cudaEventDestroy(ctx->ev_fork_v[k]);
  if (ctx->ev_lin_sorted) cudaEventDestroy(ctx->ev_lin_sorted);
  if (ctx->ev_bulk1) cudaEventDestroy(ctx->ev_bulk1);
  for (int k = 0; k < 12; ++k) if (ctx->ev_view[k / 4][(k / 2) & 1][k & 1]) cudaEventDestroy(ctx->ev_view[k / 4][(k / 2) & 1][k & 1]);
  if (ctx->lin_stream) cudaStreamDestroy(ctx->lin_stream);
  for (int k = 0; k < kSideStreams; ++k) {
    if (ctx->ev_join[k]) cudaEventDestroy(ctx->ev_join[k]);
    if (ctx->side[k]) cudaStreamDestroy(ctx->side[k]);
  }
  if (ctx->h_bintab) cudaFreeHost(ctx->h_bintab);
  if (ctx->h_plan) cudaFreeHost(ctx->h_plan);
  if (ctx->ev_call) cudaEventDestroy(ctx->ev_call);
  if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
  if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
  if (ctx->h_totals) cudaFreeHost(ctx->h_totals);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *elector_last_error(const elector_ctx *ctx) { return ctx ? ctx->err.c_str() : g_init_error.c_str(); }

// a window's three rows take 3 * (columns rounded up to 4) bytes and columns <= letters of the window
int64_t elector_poa_rows_bound(int64_t n, const int64_t *ro, const int64_t *co, const int64_t *uo) {
  if (n <= 0 || !ro || !co || !uo) return 0;
  return (3 * ((ro[n] - ro[0]) + (co[n] - co[0]) + (uo[n] - uo[0]) + 3 * n) + 31) & ~(int64_t)15;   // 16-byte granules + one spare
}

int elector_poa_run_device(elector_ctx *ctx, int64_t n, const char *d_ref, const int64_t *d_roff, const char *d_cor,
                           const int64_t *d_coff, const char *d_unc, const int64_t *d_uoff, const int64_t *h_roff,
                           const int64_t *h_coff, const int64_t *h_uoff, char *d_rows, int64_t rows_cap,
                           int64_t *d_rowoff, int32_t *d_stride, int32_t *d_nring, int32_t *d_s1, int32_t *d_s2,
                           int64_t *d_cells, int64_t *d_rows_used) {
  if (!ctx) return ELECTOR_EINVAL;
  if (n < 0 || (n > 0 && (!d_ref || !d_cor || !d_unc || !d_roff || !d_coff || !d_uoff || !d_rows || !d_rowoff || !d_stride || !d_nring)))
    return ctx->fail(ELECTOR_EINVAL, "null argument");
  CU(cudaSetDevice(ctx->device));
  (void)h_uoff;   // binning happens on the device; the host copies of the ref / cor offsets spare a read-back of their totals
  ctx->trace = getenv("ELECTOR_TRACE") != nullptr;
  ctx->last_ms = ctx->last_ms_phase1 = 0.f;
  ctx->last_launches = 0;
  return align_device(ctx, n, d_ref, d_roff, d_cor, d_coff, d_unc, d_uoff, h_roff, h_coff, d_rows, rows_cap, d_rowoff, d_stride, d_nring, d_s1, d_s2,
                      d_cells, d_rows_used);
}

int elector_poa_run(elector_ctx *ctx, int64_t n, const char *ref, const int64_t *ro, const char *cor, const int64_t *co,
                    const char *unc, const int64_t *uo, char *rows_out, int64_t rows_cap, int64_t *row_off,
                    int32_t *row_stride, int32_t *nring, int32_t *score1, int32_t *score2, int64_t *cells) {
  return elector_pipeline_run(ctx, n, ref, ro, cor, co, unc, uo, 0, nullptr, rows_out, rows_cap, row_off, row_stride, nring,
                              score1, score2, cells, nullptr, nullptr);
}

int elector_pipeline_run(elector_ctx *ctx, int64_t n, const char *ref, const int64_t *ro, const char *cor, const int64_t *co,
                         const char *unc, const int64_t *uo, int64_t n_reads, const int64_t *read_first, char *rows_out,
                         int64_t rows_cap, int64_t *row_off, int32_t *row_stride, int32_t *nring, int32_t *score1,
                         int32_t *score2, int64_t *cells, int64_t *counters_out, int64_t *sums_out) {
  if (!ctx) return ELECTOR_EINVAL;
  if (n > 0 && (!rows_out || !row_off || !row_stride || !nring)) return ctx->fail(ELECTOR_EINVAL, "null argument");
  if (n_reads > 0 && !counters_out) return ctx->fail(ELECTOR_EINVAL, "null argument");
  elector_pipeline_io io;
  memset(&io, 0, sizeof io);
  io.n_windows = n; io.n_reads = n_reads;
  io.ref = ref; io.cor = cor; io.unc = unc; io.ref_off = ro; io.cor_off = co; io.unc_off = uo; io.read_first = read_first;
  io.rows_out = rows_out; io.rows_cap = rows_cap; io.row_off = row_off; io.row_stride = row_stride;
  io.nring = nring; io.score1 = score1; io.score2 = score2; io.cells = cells;
  io.counters_out = counters_out; io.sums_out = sums_out;
  return elector_pipeline_run2(ctx, &io);
}

int64_t elector_merged_bound(int64_t n, int64_t n_reads, const int64_t *ro, const int64_t *co, const int64_t *uo) {
  if (n <= 0 || !ro || !co || !uo) return 0;
  return ((ro[n] - ro[0]) + (co[n] - co[0]) + (uo[n] - uo[0]) + 32 * n_reads + 31) & ~(int64_t)15;
}

void elector_unpack_columns(const uint8_t *codes, int64_t n, char *ref, char *cor, char *unc) {
  static const char sym[] = ELECTOR_COLUMN_CHARS;
  for (int64_t i = 0; i < n; ++i) {
    const unsigned c = codes[i];
    if (c < 216) { ref[i] = sym[c % 6]; cor[i] = sym[(c / 6) % 6]; unc[i] = sym[c / 36]; }
    else ref[i] = cor[i] = unc[i] = '?';   // 255: the three characters are in the escape list
  }
}

int64_t elector_pack_letters(const char *letters, int64_t n, uint8_t *bits, int64_t *exc_pos, uint8_t *exc_byte, int64_t exc_cap) {
  if (n <= 0 || !letters || !bits) return 0;
  static const struct Lut { int8_t v[256]; Lut() { memset(v, -1, sizeof v); v['A'] = v['a'] = 0; v['C'] = v['c'] = 1; v['G'] = v['g'] = 2; v['T'] = v['t'] = 3; } } lut;
  int64_t ne = 0;
  for (int64_t i = 0; i < n; i += 4) {
    unsigned b = 0;
    for (int k = 0; k < 4 && i + k < n; ++k) {
      const unsigned char c = (unsigned char)letters[i + k];
      const int v = lut.v[c];
      if (v < 0) { if (ne < exc_cap && exc_pos && exc_byte) { exc_pos[ne] = i + k; exc_byte[ne] = c; } ++ne; }
      else b |= (unsigned)v << (2 * k);
    }
    bits[i >> 2] = (uint8_t)b;
  }
  return ne;
}

// Host buffers in, host buffers out.  The call is cut into chunks of whole reads; every chunk is processed start to
// finish -- inputs to the device, both POA phases, merge, tally, results back -- by one of a few WORKER contexts (this
// context and children it creates once), each on its own host thread and streams.  While one worker's chunk computes,
// another's inputs arrive and a third's results leave.
int elector_pipeline_run2(elector_ctx *ctx, const elector_pipeline_io *iop) {
  if (!ctx) return ELECTOR_EINVAL;
  if (!iop) return ctx->fail(ELECTOR_EINVAL, "null argument");
  const elector_pipeline_io &io = *iop;
  const int64_t n = io.n_windows, n_reads = io.n_reads;
  const int64_t *ro = io.ref_off, *co = io.cor_off, *uo = io.unc_off, *read_first = io.read_first;
  const bool packed = io.pref || io.pcor || io.punc;
  if (n < 0 || n_reads < 0) return ctx->fail(ELECTOR_EINVAL, "negative count");
  if (n > 0 && (!ro || !co || !uo)) return ctx->fail(ELECTOR_EINVAL, "null offsets");
  if (n > 0 && packed && !(io.pref && io.pcor && io.punc && io.pref->bits && io.pcor->bits && io.punc->bits)) return ctx->fail(ELECTOR_EINVAL, "packed letters: all three kinds or none");
  if (n > 0 && !packed && !(io.ref && io.cor && io.unc)) return ctx->fail(ELECTOR_EINVAL, "null letters");
  if (n > 0 && io.rows_out && !(io.row_off && io.row_stride && io.nring)) return ctx->fail(ELECTOR_EINVAL, "rows_out needs row_off, row_stride and nring");
  if (n_reads > 0 && !read_first) return ctx->fail(ELECTOR_EINVAL, "null read_first");
  if (io.m_nibbles < 0 || io.m_nibbles > 2) return ctx->fail(ELECTOR_EINVAL, "m_nibbles must be 0, 1 or 2");
  if (io.m_ref && !((io.m_nibbles == 2 || (io.m_cor && io.m_unc)) && io.m_off && io.m_len && n_reads > 0)) return ctx->fail(ELECTOR_EINVAL, "merged rows need all three buffers (one with m_nibbles = 2), m_off, m_len and reads");
  if (io.m_ref && io.m_nibbles && io.m_esc_cap > 0 && !(io.m_esc_pos && io.m_esc_byte)) return ctx->fail(ELECTOR_EINVAL, "null escape arrays");
  if (io.sums_out) memset(io.sums_out, 0, ELECTOR_TALLY_K * sizeof(int64_t));
  if (io.m_n_esc) *io.m_n_esc = 0;
  ctx->last_ms = ctx->last_ms_phase1 = 0.f;
  ctx->last_launches = 0;
  if (n == 0) return ELECTOR_OK;
  if (ro[0] != 0 || co[0] != 0 || uo[0] != 0) return ctx->fail(ELECTOR_EINVAL, "offsets must start at 0");
  if (n_reads > 0 && (read_first[0] != 0 || read_first[n_reads] != n)) return ctx->fail(ELECTOR_EINVAL, "read_first must span 0..n_windows");
  if (packed && (io.pref->n_letters < ro[n] || io.pcor->n_letters < co[n] || io.punc->n_letters < uo[n])) return ctx->fail(ELECTOR_EINVAL, "packed letters shorter than the offsets say");
  CU(cudaSetDevice(ctx->device));
  const bool trace = ctx->trace = getenv("ELECTOR_TRACE") != nullptr;
  // ---- chunk boundaries (windows; whole reads when reads are given) ----
  // Large chunks: the kernels run 32 windows of one sorted size class in lock step and finish a class with its slowest
  // group, so their throughput grows with the number of windows sorted together -- but chunks on several workers overlap
  // their transfers with each other's kernels: three chunks of ~0.65 M windows on three workers are the measured best for
  // 10 000 reads of 10 kb.  ELECTOR_PIPELINE_CHUNKS forces a chunk count.
  // With packed letters the inputs are a quarter of the bytes and fewer, larger chunks win: two chunks of ~1 M windows measured
  // best for all output formats (counters only: 8.9 ms against 9.3 in three chunks and 11.9 in one).
  const int64_t chunk_windows = packed ? 1000000 : 700000;
  int want_workers = 3;
  if (const char *e = getenv("ELECTOR_PIPELINE_WORKERS")) want_workers = std::max(1, std::min(8, atoi(e)));
  int64_t want_chunks = (n + chunk_windows - 1) / chunk_windows;
  if (const char *e = getenv("ELECTOR_PIPELINE_CHUNKS")) want_chunks = std::max(1, atoi(e));
  std::vector<ChunkJob> jobs;
  {
    int64_t w = 0, r = 0;
    for (int64_t k = 0; w < n; ++k) {
      ChunkJob j;
      j.w0 = w; j.r0 = r;
      int64_t want = k + 1 >= want_chunks ? n : (int64_t)((double)n * (double)(k + 1) / (double)want_chunks);
      want = std::min<int64_t>(n, std::max<int64_t>(want, w + std::min<int64_t>(n, 65536)));
      if (n_reads > 0) {   // first read boundary at or after the target (binary search on read_first)
        int64_t lo = r + 1, hi = n_reads;
        while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (read_first[mid] >= want) hi = mid; else lo = mid + 1; }
        r = lo;
        w = read_first[r];
      } else w = want;
      j.w1 = w; j.r1 = r;
      // merged rows of the chunk in the caller's buffers: from the bound of the reads before it (letters + 32 per read, 16-aligned)
      j.m_base = (ro[j.w0] + co[j.w0] + uo[j.w0] + 32 * j.r0) & ~(int64_t)15;
      jobs.push_back(j);
    }
  }
  // rows of chunk k land at rows_out + rows_base(k): the bound of the windows before it.  The O(1) bound when the
  // caller's buffer allows it (or takes no rows at all), else the exact one (one pass over the offsets).
  const bool loose = !io.rows_out || io.rows_cap >= elector_poa_rows_bound(n, ro, co, uo);
  if (loose) {
    // region k = [lo4(bound of the windows before it), lo4(bound of the windows up to its end)): the regions tile the O(1)
    // bound of the call whatever the chunking.  A window's share of the bound is 3 * (letters + 3) bytes and it needs at most
    // 3 * ((columns + 3) & ~3) with columns <= letters - 1 (every DP aligns something or, at worst, ('AAAAA','C','G')-like
    // inputs give letters - 1 columns): at least 3 spare bytes per window, so the rounding of a region to the 4-byte row
    // words (at most 3 bytes) fits even a chunk of one window.  (Rounding to 16 bytes did not: a call of one window with as
    // many columns as letters - 1 overflowed its region.)  Two regions per chunk lose up to 30 bytes more to the 16-byte
    // boundary between them, so a chunk is only split when it has 64 windows or more (192 spare bytes); the kernels check
    // rows_cap anyway, so the failure mode of a wrong margin is ELECTOR_ECAPACITY, never a stray write.
    auto before = [&](int64_t w) { return (3 * (ro[w] + co[w] + uo[w] + 3 * w)) & ~(int64_t)3; };
    for (ChunkJob &j : jobs) { j.rows_base = before(j.w0); j.rows_len = before(j.w1) - j.rows_base; j.split = j.w1 - j.w0 >= 64; }
  } else {
    int64_t base = 0;
    for (ChunkJob &j : jobs) {
      j.rows_base = base;
      j.split = false;   // two row regions need the spare bytes of the O(1) bound (the boundary is aligned to 16 bytes)
      int64_t t = 0;
      for (int64_t w = j.w0; w < j.w1; ++w) t += ((ro[w + 1] - ro[w]) + (co[w + 1] - co[w]) + (uo[w + 1] - uo[w]) + 3) & ~(int64_t)3;
      j.rows_len = 3 * t;
      base += j.rows_len;
    }
    if (base > io.rows_cap) return ctx->fail(ELECTOR_ECAPACITY, "rows_out capacity %lld too small (%lld needed)", (long long)io.rows_cap, (long long)base);
  }
  // ---- workers ----
  std::vector<elector_ctx *> slots;
  int rc = worker_slots(ctx, {ctx->device}, want_workers, jobs.size(), slots);
  if (rc != ELECTOR_OK) return rc;
  std::atomic<int> h2d_turn{0};
  std::atomic<long long> n_esc{0};
  cudaEvent_t h2d_prev = nullptr;
  for (size_t k = 0; k < jobs.size(); ++k) jobs[k].index = (int)k;
  PipeArgs pa{iop, ro, co, uo, packed, ctx->ev_call, &h2d_turn, &h2d_prev, &n_esc};
  if (trace) CU(cudaEventRecord(pa.ev_call, ctx->stream));
  const auto host_t0 = std::chrono::steady_clock::now();
  rc = run_pool(ctx, slots, jobs.size(), io.sums_out, [&](elector_ctx *wk, int id, size_t k, int64_t *sums, const std::atomic<int> &failed) {
    const double t_in = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
    const int rc = process_chunk(wk, pa, jobs[k], sums, failed);
    if (trace)
      fprintf(stderr, "[elector trace] chunk %zu (worker %d): %lld windows, host clock %.2f -> %.2f ms\n", k, id, (long long)(jobs[k].w1 - jobs[k].w0), t_in,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count());
    return rc;
  });
  if (rc != ELECTOR_OK) return rc;
  if (io.m_n_esc) *io.m_n_esc = n_esc.load();
  if (trace) fprintf(stderr, "[elector trace] call returned at %.2f ms (host clock), %zu chunks on %zu workers\n",
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count(), jobs.size(), slots.size());
  return ELECTOR_OK;
}

int elector_poa_files(elector_ctx *ctx, const char *ref_fa, const char *cor_fa, const char *unc_fa, const char *pir_out,
                      int print_perm) {
  if (!ctx) return ELECTOR_EINVAL;
  if (!ref_fa || !cor_fa || !unc_fa || !pir_out) return ctx->fail(ELECTOR_EINVAL, "null path");
  FastaFile C, U, R;
  // same open order and failure behaviour as main.c:242-262
  if (read_fasta_file(cor_fa, C) < 0) return ctx->fail(ELECTOR_EIO, "Couldn't open sequence file %s", cor_fa);
  if (read_fasta_file(unc_fa, U) < 0) return ctx->fail(ELECTOR_EIO, "Couldn't open sequence file %s", cor_fa);
  if (read_fasta_file(ref_fa, R) < 0) return ctx->fail(ELECTOR_EIO, "Couldn't open sequence file %s", cor_fa);
  if (R.rec.empty()) return ctx->fail(ELECTOR_EIO, "Error reading sequence file %s", cor_fa);
  // The reference indexes all three arrays with the reference count and runs off the end
  // when they disagree (undefined); we align the common prefix and report the mismatch.
  size_t n = std::min(R.rec.size(), std::min(C.rec.size(), U.rec.size()));
  const bool ragged = !(R.rec.size() == C.rec.size() && R.rec.size() == U.rec.size());
  FILE *out = fopen(pir_out, "w");
  if (!out) return ctx->fail(ELECTOR_EIO, "cannot write %s", pir_out);
  int rc = ELECTOR_OK;
  if (n > 0) {
    std::vector<int64_t> ro = R.offsets(), co = C.offsets(), uo = U.offsets();
    ro.resize(n + 1); co.resize(n + 1); uo.resize(n + 1);
    const int64_t bound = elector_poa_rows_bound((int64_t)n, ro.data(), co.data(), uo.data());
    std::vector<char> rows(bound);
    std::vector<int64_t> roff(n);
    std::vector<int32_t> stride(n), nring(n);
    rc = elector_poa_run(ctx, (int64_t)n, R.seq.data(), ro.data(), C.seq.data(), co.data(), U.seq.data(), uo.data(),
                         rows.data(), bound, roff.data(), stride.data(), nring.data(), nullptr, nullptr, nullptr);
    if (rc == ELECTOR_OK) {
      std::string buf;
      buf.reserve(1 << 20);
      for (size_t w = 0; w < n; ++w) {
        const FastaRecord *recs[3] = {&R.rec[w], &C.rec[w], &U.rec[w]};
        for (int s = 0; s < 3; ++s) {
          buf += '>'; buf += recs[s]->name; buf += ' '; buf += recs[s]->title; buf += '\n';
          buf.append(rows.data() + roff[w] + (int64_t)s * stride[w], nring[w]);
          buf += '\n';
        }
        if (buf.size() > (1 << 20) - 65536) { fwrite(buf.data(), 1, buf.size(), out); buf.clear(); }
      }
      fwrite(buf.data(), 1, buf.size(), out);
      if (print_perm) {
        std::string perm;
        for (size_t w = 0; w < n; ++w) perm += "0 1 2 \n";
        fwrite(perm.data(), 1, perm.size(), stdout);
      }
    }
  }
  fclose(out);
  if (rc != ELECTOR_OK) return rc;
  if (ragged) return ctx->fail(ELECTOR_EIO, "record counts differ (ref %zu, corrected %zu, uncorrected %zu); aligned the first %zu", R.rec.size(), C.rec.size(), U.rec.size(), n);
  return ELECTOR_OK;
}

int elector_event_record(elector_ctx *ctx, int which) {
  if (!ctx) return ELECTOR_EINVAL;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(which ? ctx->uev1 : ctx->uev0, ctx->stream));
  return ELECTOR_OK;
}

int elector_event_elapsed_ms(elector_ctx *ctx, float *ms) {
  if (!ctx || !ms) return ELECTOR_EINVAL;
  CU(cudaEventSynchronize(ctx->uev1));
  CU(cudaEventElapsedTime(ms, ctx->uev0, ctx->uev1));
  return ELECTOR_OK;
}

int elector_int32_peak(elector_ctx *ctx, double *tiops_mixed, double *tiops_alu) {
  if (!ctx) return ELECTOR_EINVAL;
  CU(cudaSetDevice(ctx->device));
  const int grid = ctx->sm_count * 8, iters = 4096;
  CU(ctx->d_scratch.reserve((size_t)grid * 256 * 4));
  double res[2] = {0, 0};
  for (int mode = 0; mode < 2; ++mode) {
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
      CU(cudaEventRecord(ctx->ev0, ctx->stream));
      if (mode == 0) int32_peak_kernel<true><<<grid, 256, 0, ctx->stream>>>(ctx->d_scratch.as<int>(), iters, 3, 7);
      else int32_peak_kernel<false><<<grid, 256, 0, ctx->stream>>>(ctx->d_scratch.as<int>(), iters, 3, 7);
      CU(cudaEventRecord(ctx->ev1, ctx->stream));
      CU(cudaEventSynchronize(ctx->ev1));
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
      if (rep > 0 && ms < best) best = ms;
    }
    // lane-operations per iteration of the unrolled body: mixed = 8*(4 IMAD + 2*(IADD+IMNMX) + 2*(LOP+IADD)) = 8*12,
    // alu-only = 8*(4*(IADD+IMNMX) + 4*(LOP+IADD)) = 8*16
    const double ops = (double)grid * 256 * iters * (mode == 0 ? 96.0 : 128.0);
    res[mode] = ops / (best * 1e-3) / 1e12;
  }
  if (tiops_mixed) *tiops_mixed = res[0];
  if (tiops_alu) *tiops_alu = res[1];
  return ELECTOR_OK;
}

int elector_last_phase_ms(const elector_ctx *ctx, float *ms_phase1, float *ms_total) {
  if (!ctx) return ELECTOR_EINVAL;
  if (ms_phase1) *ms_phase1 = ctx->last_ms_phase1;
  if (ms_total) *ms_total = ctx->last_ms;
  return ELECTOR_OK;
}

int elector_last_reads_ms(const elector_ctx *ctx, float *ms_split, float *ms_poa, float *ms_merge_tally) {
  if (!ctx) return ELECTOR_EINVAL;
  if (ms_split) *ms_split = ctx->last_ms_split;
  if (ms_poa) *ms_poa = ctx->last_ms - ctx->last_ms_split - ctx->last_ms_tally;
  if (ms_merge_tally) *ms_merge_tally = ctx->last_ms_tally;
  return ELECTOR_OK;
}

int elector_last_kernel_ms(const elector_ctx *ctx, float *ms, int *launches) {
  if (!ctx) return ELECTOR_EINVAL;
  if (ms) *ms = ctx->last_ms;
  if (launches) *launches = ctx->last_launches;
  return ELECTOR_OK;
}

}  // extern "C"

#include "tally_capi.inl"
#include "split_capi.inl"
#include "report_capi.inl"
