// bin_kernel.cuh -- device-side scheduling of the windows of one call.
//
// The POA kernels run one window per thread in lock step, so a warp is only efficient when
// its 32 windows have the same loop shape.  Each phase therefore sorts the window ids with a
// counting sort (histogram -> chunked scan -> scatter), largest first, and cuts the sorted
// list into a few SEGMENTS (one launch each) whose per-warp scratch is sized by the segment's
// own maxima:
//   phase 1 (DP1, cost ~ bands(cor) x len(ref)):  key = (8-row half-bands of cor, len(ref)/2)
//   phase 2 (DP2, cost ~ bands(unc) x len(P1)):   key = (half-bands of unc, len(P1)/4, where and how
//            ref and cor first differ) -- computed by the phase-1 kernel itself (bin2_of)
// Everything stays on the device; the host reads back one small table per phase.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "poa_kernel.cuh"
#ifdef __CUDACC__
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>
#endif

namespace elector {

constexpr int kXq1 = 129;                         // len(ref)/2 quanta of a small window
constexpr int kSmallBins1 = kNbMax * kXq1;
constexpr int kNumBins1 = kBigTiers + kSmallBins1;
constexpr int kNumSegs1 = kBigTiers + 3;
constexpr int kMaxSegs = kNumSegs2 > kNumSegs1 ? kNumSegs2 : kNumSegs1;
constexpr int kMaxBins = kNumBins2 > kNumBins1 ? kNumBins2 : kNumBins1;
constexpr int kScanChunk = 1024;
constexpr int kMaxChunks = (kMaxBins + kScanChunk - 1) / kScanChunk;
// Longest window the kernels take.  The reference has no cap of its own (fasta_format.c:20 reads any line in 32 KiB chunks,
// seq_util.h:22) but allocates len_y * len_x two-byte moves per DP (align_lpo_po2.c:258-266): 8.6 GB at these lengths.  Here
// the node records hold predecessor indices in 16 bits (0xffff = none) and ordinal slots in 15, so len(P1) <= len(ref) +
// len(cor) must stay below 65 535; the uncorrected sequence is bounded the same way (and by the scratch of the call).
constexpr int kMaxWindowLen = 65534;              // each sequence of a window
constexpr int kMaxNodes = 65534;                  // len(ref) + len(cor) >= len(P1)

struct SegInfo {      // one launch of a POA kernel
  int32_t first_bin;  // in: first bin of the segment (bins of a segment are contiguous)
  int32_t start;      // out: first position in the sorted item list
  int32_t count;      // out: windows
  int32_t pad;
};

// what a segment's kernel needs to know about its work, computed on the device (plan_segments_kernel) once the sort
// knows the segment's size and maxima: the host launches every segment with a fixed grid and never reads a table back
struct SegPlanDev {
  int32_t start, count;     // the segment's slice of the sorted item list
  int32_t max_ctas;         // CTAs (one warp each) that take work; the others of the launch leave at once
  int32_t counter;          // index of the segment's work counter in the control words
  uint32_t warp_words;      // scratch words per lane (layout of the segment's maxima)
  uint32_t pad;
  unsigned long long scratch_off;   // first scratch word of the segment in the phase's pool
};

struct BinTable {
  SegInfo seg[kMaxSegs + 1];   // [nseg].first_bin = number of bins
  int32_t seg_max[kMaxSegs * 4];  // per segment maxima: phase 1 {lr, lc}, phase 2 {n1, lu}
  SegPlanDev plan[kMaxSegs];
  int32_t nseg, nbins;
  int32_t err_code;    // 0 ok, 1 empty sequence, 2 sequence longer than kMaxWindowLen or len(ref) + len(cor) > kMaxNodes, 3 scratch pool too small
  int32_t err_window;  // smallest offending window id
  unsigned long long lin_bytes;  // phase-2 table: row bytes (3 x columns bound, rounded to 4) of the windows in the linear segments
  unsigned long long need_words; // err_code 3: scratch words the call needs in the pool that was too small
};

#ifdef __CUDACC__
__device__ __forceinline__ bool seg_setup(const PoaArgs &a, SegRun &run) {
  const SegPlanDev &pl = a.tab->plan[a.seg];
  if ((int)blockIdx.x >= pl.max_ctas) return false;   // uniform over the CTA
  if (threadIdx.x == 0) {
    run.items = a.items_base + pl.start;
    run.n_items = pl.count;
    run.scratch = a.scratch_base + pl.scratch_off;
    run.warp_words = pl.warp_words;
    run.work_counter = a.ctrl + pl.counter;
    run.rows_cap = a.rows_cap_dev ? *a.rows_cap_dev : a.rows_cap;
  }
  __syncwarp();
  return true;
}
#endif

__host__ __device__ inline int seg1_of_nb(int nb8) { return kBigTiers + (nb8 > 16 ? 0 : nb8 > 8 ? 1 : 2); }
__host__ __device__ inline void bin1_of(int lr, int lc, int &bin, int &seg) {
  const int mx = lr > lc ? lr : lc;
  if (mx > kSmallMax) {
    bin = seg = kBigTiers - big_tier(mx);   // the largest tier comes first
  } else {
    const int nb8 = (lc + 7) >> 3;
    const int small = (nb8 - 1) * kXq1 + (lr >> 1);
    bin = kBigTiers + (kSmallBins1 - 1 - small);
    seg = seg1_of_nb(nb8);
  }
}
// first bin of every segment (host side, goes into BinTable::seg[].first_bin)
inline void fill_segments1(BinTable &t) {
  t.nseg = kNumSegs1; t.nbins = kNumBins1;
  for (int s = 0; s < kBigTiers; ++s) t.seg[s].first_bin = s;
  const int hi[3] = {32, 16, 8};
  for (int k = 0; k < 3; ++k) t.seg[kBigTiers + k].first_bin = kBigTiers + (kSmallBins1 - 1 - ((hi[k] - 1) * kXq1 + (kXq1 - 1)));
  t.seg[kNumSegs1].first_bin = kNumBins1;
}
inline void fill_segments2(BinTable &t) {
  t.nseg = kNumSegs2; t.nbins = kNumBins2;
  for (int s = 0; s < kBigTiers; ++s) t.seg[s].first_bin = s;
  const int hi[4] = {32, 16, 8, 4};
  for (int k = 0; k < 4; ++k) {
    t.seg[kBigTiers + k].first_bin = kBigTiers + (kSmallBins2 - 1 - (((hi[k] - 1) * kN1q + (kN1q - 1)) * kSpCodes + (kSpCodes - 1)));
    t.seg[kFirstLinSeg2 + k].first_bin = kBigTiers + kSmallBins2 + (kLinBins2 - 1 - (((hi[k] - 1) * kN1q + (kN1q - 1)) * kDcls + (kDcls - 1)));
  }
  t.seg[kNumSegs2].first_bin = kNumBins2;
}

// set-up of one call on the device: control words (rows cursor = words 0..1), both segment tables
struct SegFirstBins { int32_t first1[kMaxSegs + 1], first2[kMaxSegs + 1], nseg1, nbins1, nseg2, nbins2; };
__global__ void init_call_kernel(int32_t *ctrl, int nctrl, unsigned long long cursor_init, BinTable *tabs, SegFirstBins fb) {
  int32_t *t = reinterpret_cast<int32_t *>(tabs);
  for (int i = threadIdx.x; i < (int)(2 * sizeof(BinTable) / 4); i += blockDim.x) t[i] = 0;
  for (int i = threadIdx.x; i < nctrl; i += blockDim.x) ctrl[i] = 0;
  __syncthreads();
  if ((int)threadIdx.x <= kMaxSegs) { tabs[0].seg[threadIdx.x].first_bin = fb.first1[threadIdx.x]; tabs[1].seg[threadIdx.x].first_bin = fb.first2[threadIdx.x]; }
  if (threadIdx.x == 0) {
    tabs[0].nseg = fb.nseg1; tabs[0].nbins = fb.nbins1; tabs[1].nseg = fb.nseg2; tabs[1].nbins = fb.nbins2;
    tabs[0].err_window = 0x7fffffff;
    *reinterpret_cast<unsigned long long *>(ctrl) = cursor_init;
  }
}

__global__ void set_u64_kernel(unsigned long long *p, unsigned long long v) { *p = v; }

// phase 1: key[w] = bin (or -1 for an invalid window), hist[bin] += 1, segment maxima
// Windows whose corrected letters ARE the reference letters (byte for byte; most windows at ELECTOR's corrected error
// rates) need no phase 1 at all when the matrix makes the diagonal the unique optimum of DP1 (match 0, everything else
// negative: the packed class): P1 is lin(ref) with every node carrying both letters, best score 0.  With `id` non-null
// the sort recognises them, leaves them out of the phase-1 work list (key -2) and does what phase 1 would have left for
// phase 2: len(P1), the phase-2 sort bin and histogram, the segment maxima and the row bytes of the linear region.
#ifdef __CUDACC__
// The letters from p on as consecutive 16-byte words, whatever p's alignment: aligned 16-byte loads, realigned by a
// word select and a funnel shift (the shift is fixed for the whole string).  A load never touches a 16-byte block that
// holds no letter of [p, end); bytes past end are left to the caller to ignore.
struct Letters16 {
  const uint4 *q;
  uint4 cur;
  uint32_t sel, sh;
  const uint8_t *end;
  __device__ __forceinline__ void init(const uint8_t *p, const uint8_t *e) {
    q = reinterpret_cast<const uint4 *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)15);
    sel = (uint32_t)(reinterpret_cast<uintptr_t>(p) >> 2) & 3u;
    sh = 8u * ((uint32_t)reinterpret_cast<uintptr_t>(p) & 3u);
    end = e;
    cur = __ldg(q);
  }
  __device__ __forceinline__ uint4 next() {
    ++q;
    const uint4 nx = reinterpret_cast<const uint8_t *>(q) < end ? __ldg(q) : make_uint4(0, 0, 0, 0);
    // words sel .. sel + 4 of cur : nx
    const bool s2 = sel & 2u, s1 = sel & 1u;
    const uint32_t t0 = s2 ? cur.z : cur.x, t1 = s2 ? cur.w : cur.y, t2 = s2 ? nx.x : cur.z, t3 = s2 ? nx.y : cur.w, t4 = s2 ? nx.z : nx.x,
                   t5 = s2 ? nx.w : nx.y;
    const uint32_t u0 = s1 ? t1 : t0, u1 = s1 ? t2 : t1, u2 = s1 ? t3 : t2, u3 = s1 ? t4 : t3, u4 = s1 ? t5 : t4;
    cur = nx;
    return make_uint4(__funnelshift_r(u0, u1, sh), __funnelshift_r(u1, u2, sh), __funnelshift_r(u2, u3, sh), __funnelshift_r(u3, u4, sh));
  }
};
#endif

struct IdentArgs {
  const uint8_t *ref, *cor;
  int32_t *n1, *key2, *hist2, *seg2_max, *score1;
  unsigned long long *lin_bytes;
};
__global__ void __launch_bounds__(256) bin1_count_kernel(int32_t n, const int64_t *ro, const int64_t *co, const int64_t *uo,
                                                          int32_t *key, int32_t *hist, BinTable *tab, bool use_ident, IdentArgs id) {
  unsigned long long lin = 0;
  for (int32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < n; w += gridDim.x * blockDim.x) {
    const int64_t lr = ro[w + 1] - ro[w], lc = co[w + 1] - co[w], lu = uo[w + 1] - uo[w];
    int bin = -1;
    if (lr <= 0 || lc <= 0 || lu <= 0) { atomicMax(&tab->err_code, 1); atomicMin(&tab->err_window, w); }
    else if (lr > kMaxWindowLen || lc > kMaxWindowLen || lu > kMaxWindowLen || lr + lc > kMaxNodes) { atomicMax(&tab->err_code, 2); atomicMin(&tab->err_window, w); }
    else {
      bool ident = false;
      if (use_ident && lr == lc && lr <= kSmallMax && lu <= kSmallMax) {
        const uint8_t *a = id.ref + ro[w], *b = id.cor + co[w];
        const int len = (int)lr;
        Letters16 sa, sb;
        sa.init(a, a + len);
        sb.init(b, b + len);
        uint32_t d = 0;
        for (int i = 0; i < len && !d; i += 16) {   // 16 letters of each per step, from aligned 16-byte loads
          const uint4 x = sa.next(), y = sb.next();
          const uint32_t e[4] = {x.x ^ y.x, x.y ^ y.y, x.z ^ y.z, x.w ^ y.w};
          const int m = len - i;   // letters left; bytes of a word past them are not compared
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int v = m - 4 * k;
            d |= v >= 4 ? e[k] : v > 0 ? e[k] & ((1u << (8 * v)) - 1u) : 0u;
          }
        }
        ident = d == 0;
      }
      if (ident) {
        int bin2, seg2;
        bin2_of((int)lr, (int)lu, 0, true, bin2, seg2);
        id.n1[w] = (int)lr;
        id.key2[w] = bin2;
        if (id.score1) id.score1[w] = 0;
        warp_hist_add(id.hist2, bin2);
        if ((int)lr > id.seg2_max[seg2 * 4]) atomicMax(&id.seg2_max[seg2 * 4], (int)lr);
        if ((int)lu > id.seg2_max[seg2 * 4 + 1]) atomicMax(&id.seg2_max[seg2 * 4 + 1], (int)lu);
        lin += 3ull * (unsigned long long)((lr + lc + lu + 3) & ~(int64_t)3);
        bin = -2;
      } else {
        int seg;
        bin1_of((int)lr, (int)lc, bin, seg);
        if (use_ident) id.key2[w] = -1;   // its phase-2 bin comes from phase 1; the early sort of the linear segments must not see a stale key
        warp_hist_add(hist, bin);
        int32_t *mx = &tab->seg_max[seg * 4];
        if ((int)lr > mx[0]) atomicMax(&mx[0], (int)lr);
        if ((int)lc > mx[1]) atomicMax(&mx[1], (int)lc);
      }
    }
    key[w] = bin;
  }
  if (use_ident) {
    for (int d = 16; d > 0; d >>= 1) lin += __shfl_xor_sync(0xffffffffu, lin, d);
    if ((threadIdx.x & 31) == 0 && lin) atomicAdd(id.lin_bytes, lin);
  }
}

// A sort works on a contiguous sub-range of a table's bins and segments (phase 2 is sorted twice: its linear segments as
// soon as the size sort has seen the windows whose cor is ref, its general segments after phase 1).
// exclusive scan of each 1024-bin chunk in place + the chunk totals; hist points at the range's first bin
__global__ void __launch_bounds__(kScanChunk) bin_scan_chunks_kernel(int32_t nbins, int32_t *hist, int32_t *chunk_total) {
  __shared__ int32_t warp_sum[32];
  const int i = blockIdx.x * kScanChunk + threadIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int32_t v = i < nbins ? hist[i] : 0;
  int32_t incl = v;
  for (int d = 1; d < 32; d <<= 1) { const int32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
  if (lane == 31) warp_sum[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int32_t s = warp_sum[lane];
    for (int d = 1; d < 32; d <<= 1) { const int32_t t = __shfl_up_sync(0xffffffffu, s, d); if (lane >= d) s += t; }
    warp_sum[lane] = s;
  }
  __syncthreads();
  const int32_t before = (wid ? warp_sum[wid - 1] : 0) + incl - v;
  if (i < nbins) hist[i] = before;
  if (threadIdx.x == kScanChunk - 1) chunk_total[blockIdx.x] = before + v;
}

// exclusive scan of the chunk totals (in place -> chunk bases) and the start / count of the segments seg0 .. seg1-1, whose
// bins are bin0 .. bin1-1 of the table (hist = the table's histogram, already scanned per chunk from bin0 on)
__global__ void __launch_bounds__(1024) bin_scan_totals_kernel(int32_t nchunks, int32_t *chunk_total, const int32_t *hist, BinTable *tab,
                                                                int32_t seg0, int32_t seg1, int32_t bin0, int32_t bin1) {
  __shared__ int32_t part[1024];
  const int32_t v = (int)threadIdx.x < nchunks ? chunk_total[threadIdx.x] : 0;
  part[threadIdx.x] = v;
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {
    const int32_t t = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += t;
    __syncthreads();
  }
  const int32_t total = part[1023];
  if ((int)threadIdx.x < nchunks) chunk_total[threadIdx.x] = part[threadIdx.x] - v;
  __syncthreads();
  const int s = seg0 + (int)threadIdx.x;
  if (s < seg1) {
    auto pos_of = [&](int bin) { return bin >= bin1 ? total : chunk_total[(bin - bin0) / kScanChunk] + hist[bin]; };
    const int32_t p0 = pos_of(tab->seg[s].first_bin), p1 = pos_of(tab->seg[s + 1].first_bin);
    tab->seg[s].start = p0;
    tab->seg[s].count = p1 - p0;
  }
}

// keys in bin0 .. bin1-1 only; cursor = the table's scanned histogram, chunk_base relative to bin0.
// Each CTA takes a contiguous tile of windows and sorts it by bin in shared memory (stable radix sort on the bits of
// bin - bin0, end_bit = bits of bin1 - bin0): a run of equal bins then reserves its range with one global atomic.  A
// window-by-window atomic would serialise in the L2 on the few hundred bins that hold most windows.  Inside a bin the
// windows of a tile keep their id order.
constexpr int kScatterThreads = 256, kScatterItems = 8, kScatterTile = kScatterThreads * kScatterItems;
#ifdef __CUDACC__
__global__ void __launch_bounds__(kScatterThreads) bin_scatter_kernel(int32_t n, const int32_t *key, int32_t *cursor, const int32_t *chunk_base,
                                                                       int32_t *items, int32_t bin0, int32_t bin1, int end_bit) {
  using Sort = cub::BlockRadixSort<uint32_t, kScatterThreads, kScatterItems, int32_t>;
  using Scan = cub::BlockScan<int32_t, kScatterThreads>;
  __shared__ union { typename Sort::TempStorage sort; typename Scan::TempStorage scan; uint32_t key[kScatterTile]; } sm;
  __shared__ int32_t run_base[kScatterTile];
  const uint32_t none = (uint32_t)(bin1 - bin0);   // invalid window, one that needs no phase 1, another sort's, past the end
  const int p0 = threadIdx.x * kScatterItems;     // blocked: thread t holds tile positions p0 .. p0 + kScatterItems - 1
  uint32_t k[kScatterItems];
  int32_t w[kScatterItems];
#pragma unroll
  for (int i = 0; i < kScatterItems; ++i) {
    const int64_t x = (int64_t)blockIdx.x * kScatterTile + p0 + i;
    const int bin = x < n ? key[x] : -1;
    k[i] = (bin >= bin0 && bin < bin1) ? (uint32_t)(bin - bin0) : none;
    w[i] = (int32_t)x;
  }
  Sort(sm.sort).Sort(k, w, 0, end_bit);   // stable: the tile in (bin, window id) order
  __syncthreads();
#pragma unroll
  for (int i = 0; i < kScatterItems; ++i) sm.key[p0 + i] = k[i];
  __syncthreads();
  int32_t start[kScatterItems];   // first position of the item's run of equal bins
  bool last[kScatterItems];       // the item ends its run
#pragma unroll
  for (int i = 0; i < kScatterItems; ++i) {
    const int p = p0 + i;
    start[i] = (p == 0 || sm.key[p - 1] != k[i]) ? p : 0;
    last[i] = p == kScatterTile - 1 || sm.key[p + 1] != k[i];
  }
  __syncthreads();
  Scan(sm.scan).InclusiveScan(start, start, cub::Max());
#pragma unroll
  for (int i = 0; i < kScatterItems; ++i)
    if (k[i] != none && last[i]) run_base[start[i]] = atomicAdd(&cursor[bin0 + k[i]], p0 + i - start[i] + 1);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < kScatterItems; ++i)
    if (k[i] != none) items[chunk_base[k[i] / kScanChunk] + run_base[start[i]] + (p0 + i - start[i])] = w[i];
}
#endif

}  // namespace elector
