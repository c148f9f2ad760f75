// Binned prediction <-> ground-truth matching for region- and slide-scale inputs (match_predictions(binned=True)).
//
// The all-pairs matchers (match.cu, match_masks.cu) test every (prediction, ground truth) pair and name a pair by the
// 32-bit index rank * G + j: O(P * G) work and P * G < 2^32.  Here the ground truth goes into a uniform grid and a
// prediction only meets the ground truth listed in the cells its box covers:
//   * bin_stats_kernel: extent, count and mean side of the valid ground truth (the host picks the cell size from it);
//   * bin_count / bin_emit: one entry per (cell, j) a ground-truth rectangle covers, counted, scanned and written as
//     keys cell << 32 | j in ascending j; the caller sorts them by cell (stable radix sort), so every cell lists its
//     ground truth in ascending j; bin_cells_kernel finds each cell's first entry by binary search;
//   * pairs_kernel<BOXES / WINDOWS>: one thread per prediction in score-rank order walks the cells its rectangle
//     covers.  A pair is tested only in the cell holding the top-left corner of its intersection, (max(x0_p, x0_g),
//     max(y0_p, y0_g)): that corner lies in both rectangles, so in both cell ranges (the cell function is monotone),
//     and every pair is seen exactly once.  A count pass and its scan size the per-prediction lists; the emit pass
//     writes each prediction's pairs and sorts them by j, so the lists are in row-major (rank, j) order;
//   * boxes: a pair is kept when ref_box_iou >= iou_min; masks: a pair is a candidate when window_pair_may_match, and
//     mask_exact_kernel counts each candidate's intersection (warp_window_intersection) before a stable compaction;
//   * order_keys_kernel: ~orderable(iou) << 32 | position; a stable sort of the high half gives IoU-descending order
//     with ties in (rank, j) order -- torch.where's order, the order the all-pairs keys rank * G + j give.
// iou_min > 0 everywhere: a pair that matches has a positive intersection, so its rectangles overlap (for finite fp32
// coordinates min(x1) - max(x0) > 0 exactly when min(x1) > max(x0); no flush-to-zero).  Rectangles that cannot overlap
// anything (non-finite coordinates, zero or negative extent, empty windows) are never binned and never walk.
#include <cmath>

#include "match_common.cuh"
#include "scan_common.cuh"

namespace hdy {

// Uniform grid over the ground truth's region: cell (cx, cy) covers [ox + cx / inv, ox + (cx + 1) / inv) in x.
// cell_of is monotone in v (each rounding is), and clamps: coordinates outside the region land in the border cells.
struct Grid {
  float ox, oy, inv;
  int nx, ny;
  __device__ __forceinline__ int cell_of(float v, float o, int n) const {
    float t = __fmul_rn(__fsub_rn(v, o), inv);
    t = fminf(fmaxf(t, 0.0f), (float)(n - 1));
    return (int)t;
  }
  __device__ __forceinline__ int cx(float x) const { return cell_of(x, ox, nx); }
  __device__ __forceinline__ int cy(float y) const { return cell_of(y, oy, ny); }
};

// The rectangle a prediction or ground truth occupies, as the corners (x0, y0) <= (x1, y1) both inside it.
//   boxes: xyxy fp32; valid when all four are finite and x1 > x0, y1 > y0 (anything else has no positive overlap);
//   windows {x0, y0, w, h}: the pixels x0 .. x0 + w - 1; valid when w > 0 and h > 0.
struct Rect {
  float x0, y0, x1, y1;
  bool valid;
};
__device__ __forceinline__ Rect box_rect(const float4 b) {
  const bool finite = isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w);
  return {b.x, b.y, b.z, b.w, finite && b.z > b.x && b.w > b.y};
}
__device__ __forceinline__ Rect window_rect(const int4 g) {
  return {__int2float_rn(g.x), __int2float_rn(g.y), __int2float_rn(g.x + g.z - 1), __int2float_rn(g.y + g.w - 1),
          g.z > 0 && g.w > 0};
}

enum Kind { BOXES = 0, WINDOWS = 1 };

template <int KIND>
__device__ __forceinline__ Rect gt_rect(const void* gt, long long j) {
  if (KIND == BOXES) return box_rect(reinterpret_cast<const float4*>(gt)[j]);
  return window_rect(reinterpret_cast<const int4*>(gt)[j]);
}

// ---------------------------------------------------------------------------------------------- binning
// stats [6] u64: orderable min x0, min y0, max x1, max y1 of the valid rectangles, their number, and the sum of
// max(width, height) in 1/16 px (each side clamped to 2^20 px).  Min / max / integer sums: the result does not depend
// on the order of the atomics.
constexpr int kBinThreads = 256;

__global__ void bin_stats_init_kernel(unsigned long long* stats) {
  if (threadIdx.x < 6) stats[threadIdx.x] = threadIdx.x < 2 ? ~0ull : 0ull;
}

template <int KIND>
__global__ void __launch_bounds__(kBinThreads) bin_stats_kernel(const void* __restrict__ gt, long long G,
                                                                unsigned long long* __restrict__ stats) {
  const long long j = (long long)blockIdx.x * kBinThreads + threadIdx.x;
  const Rect r = j < G ? gt_rect<KIND>(gt, j) : Rect{0.f, 0.f, 0.f, 0.f, false};
  unsigned v[4] = {0xffffffffu, 0xffffffffu, 0u, 0u};
  unsigned n = 0;
  unsigned long long side = 0;
  if (r.valid) {
    v[0] = orderable_u32(r.x0);
    v[1] = orderable_u32(r.y0);
    v[2] = orderable_u32(r.x1);
    v[3] = orderable_u32(r.y1);
    n = 1;
    const float s = KIND == BOXES ? fmaxf(__fsub_rn(r.x1, r.x0), __fsub_rn(r.y1, r.y0))
                                  : fmaxf(__fsub_rn(r.x1, r.x0), __fsub_rn(r.y1, r.y0)) + 1.0f;
    side = (unsigned long long)(fminf(s, 1048576.0f) * 16.0f);
  }
  v[0] = __reduce_min_sync(0xffffffffu, v[0]);
  v[1] = __reduce_min_sync(0xffffffffu, v[1]);
  v[2] = __reduce_max_sync(0xffffffffu, v[2]);
  v[3] = __reduce_max_sync(0xffffffffu, v[3]);
  n = __reduce_add_sync(0xffffffffu, n);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) side += __shfl_xor_sync(0xffffffffu, side, o);
  if ((threadIdx.x & 31) == 0 && n) {
    atomicMin(stats + 0, (unsigned long long)v[0]);
    atomicMin(stats + 1, (unsigned long long)v[1]);
    atomicMax(stats + 2, (unsigned long long)v[2]);
    atomicMax(stats + 3, (unsigned long long)v[3]);
    atomicAdd(stats + 4, (unsigned long long)n);
    atomicAdd(stats + 5, side);
  }
}

// cell ranges [c0, c1] of a rectangle
struct CellRange {
  int x0, y0, x1, y1;
};
__device__ __forceinline__ CellRange cell_range(const Grid& g, const Rect& r) {
  return {g.cx(r.x0), g.cy(r.y0), g.cx(r.x1), g.cy(r.y1)};
}

// words(j) of the entry scan: the cells ground truth j covers (0 when it is not valid)
template <int KIND>
struct EntryCount {
  const void* gt;
  Grid g;
  __device__ int64_t operator()(long long j) const {
    const Rect r = gt_rect<KIND>(gt, j);
    if (!r.valid) return 0;
    const CellRange c = cell_range(g, r);
    return (int64_t)(c.x1 - c.x0 + 1) * (c.y1 - c.y0 + 1);
  }
};

template <int KIND>
__global__ void __launch_bounds__(kBinThreads) bin_emit_kernel(const void* __restrict__ gt, long long G, Grid g,
                                                               const int64_t* __restrict__ ent_off,
                                                               unsigned long long* __restrict__ cell_keys) {
  const long long j = (long long)blockIdx.x * kBinThreads + threadIdx.x;
  if (j >= G) return;
  const Rect r = gt_rect<KIND>(gt, j);
  if (!r.valid) return;
  const CellRange c = cell_range(g, r);
  long long e = ent_off[j];
  for (int y = c.y0; y <= c.y1; ++y)
    for (int x = c.x0; x <= c.x1; ++x)
      cell_keys[e++] = ((unsigned long long)((long long)y * g.nx + x) << 32) | (unsigned long long)j;
}

// cell_start[c] = first entry of cell c in the sorted keys (c = 0 .. n_cells; cell_start[n_cells] = E)
__global__ void __launch_bounds__(kBinThreads) bin_cells_kernel(const unsigned long long* __restrict__ cell_keys,
                                                                long long E, long long n_cells,
                                                                int64_t* __restrict__ cell_start) {
  const long long c = (long long)blockIdx.x * kBinThreads + threadIdx.x;
  if (c > n_cells) return;
  long long lo = 0, hi = E;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if ((long long)(cell_keys[mid] >> 32) < c)
      lo = mid + 1;
    else
      hi = mid;
  }
  cell_start[c] = lo;
}

// ---------------------------------------------------------------------------------------------- pairs
struct PairOut {
  int32_t* rank;  // NULL: count pass
  int32_t* j;
  float* val;     // boxes: the IoU; masks: unused (candidates)
};

// Heap sort of one prediction's list by j (the j of one prediction are distinct: any sort gives the same order).
__device__ void sort_by_j(int32_t* __restrict__ js, float* __restrict__ vals, long long n) {
  auto sift = [&](long long root, long long end) {
    while (2 * root + 1 < end) {
      long long child = 2 * root + 1;
      if (child + 1 < end && js[child + 1] > js[child]) ++child;
      if (js[root] >= js[child]) return;
      const int32_t tj = js[root];
      js[root] = js[child];
      js[child] = tj;
      if (vals) {
        const float tv = vals[root];
        vals[root] = vals[child];
        vals[child] = tv;
      }
      root = child;
    }
  };
  for (long long s = n / 2 - 1; s >= 0; --s) sift(s, n);
  for (long long end = n - 1; end > 0; --end) {
    const int32_t tj = js[0];
    js[0] = js[end];
    js[end] = tj;
    if (vals) {
      const float tv = vals[0];
      vals[0] = vals[end];
      vals[end] = tv;
    }
    sift(0, end);
  }
}

constexpr int kPairThreads = 128;

// One thread per prediction rank r.  Count pass (out.rank == NULL): off[r] = the number of pairs of r.  Emit pass:
// off[] holds their exclusive scan; the pairs of r go to [off[r], off[r + 1]), sorted by j.
//   BOXES:   pred / gt float4 xyxy, kept when ref_box_iou >= iou_min (val = iou);
//   WINDOWS: pred / gt int4 windows + areas, kept when window_pair_may_match (candidates of mask_exact_kernel).
template <int KIND>
__global__ void __launch_bounds__(kPairThreads) pairs_kernel(
    const void* __restrict__ pred, const int32_t* __restrict__ pred_areas, const int32_t* __restrict__ pred_order,
    long long P, const void* __restrict__ gt, const int32_t* __restrict__ gt_areas, Grid g,
    const int64_t* __restrict__ cell_start, const unsigned long long* __restrict__ cell_keys, float iou_min,
    int64_t* __restrict__ off, PairOut out) {
  const long long r = (long long)blockIdx.x * kPairThreads + threadIdx.x;
  if (r >= P) return;
  const int row = pred_order ? pred_order[r] : (int)r;
  const float4 pb = KIND == BOXES ? reinterpret_cast<const float4*>(pred)[row] : make_float4(0.f, 0.f, 0.f, 0.f);
  const int4 pw = KIND == WINDOWS ? reinterpret_cast<const int4*>(pred)[row] : make_int4(0, 0, 0, 0);
  const Rect a = KIND == BOXES ? box_rect(pb) : window_rect(pw);
  long long n = 0;
  const long long base = out.rank ? off[r] : 0;
  if (a.valid) {
    const float area_pb = KIND == BOXES ? box_area(pb) : 0.0f;
    const int area_pw = KIND == WINDOWS ? pred_areas[row] : 0;
    const CellRange c = cell_range(g, a);
    for (int y = c.y0; y <= c.y1; ++y) {
      for (int x = c.x0; x <= c.x1; ++x) {
        const long long cell = (long long)y * g.nx + x;
        const long long e1 = cell_start[cell + 1];
        for (long long e = cell_start[cell]; e < e1; ++e) {
          const int j = (int)(uint32_t)__ldg(cell_keys + e);
          bool keep;
          float val = 0.0f;
          if (KIND == BOXES) {
            const float4 b = reinterpret_cast<const float4*>(gt)[j];
            if (g.cx(fmaxf(pb.x, b.x)) != x || g.cy(fmaxf(pb.y, b.y)) != y) continue;   // seen in another cell
            val = ref_box_iou(pb, area_pb, b, box_area(b));
            keep = val >= iou_min;
          } else {
            const int4 b = reinterpret_cast<const int4*>(gt)[j];
            if (g.cx(__int2float_rn(max(pw.x, b.x))) != x || g.cy(__int2float_rn(max(pw.y, b.y))) != y) continue;
            keep = window_pair_may_match(pw, area_pw, b, gt_areas[j], iou_min);
          }
          if (!keep) continue;
          if (out.rank) {
            out.rank[base + n] = (int32_t)r;
            out.j[base + n] = j;
            if (out.val) out.val[base + n] = val;
          }
          ++n;
        }
      }
    }
  }
  if (!out.rank)
    off[r] = n;
  else if (n > 1)
    sort_by_j(out.j + base, out.val ? out.val + base : nullptr, n);
}

// ---------------------------------------------------------------------------------------------- mask IoU
constexpr int kExactListThreads = 256;
constexpr int kExactListMaxBlocks = 8192;

// One warp per candidate c < n: iou[c] = mask_iou of its exact intersection (the all-pairs exact_kernel's count).
__global__ void __launch_bounds__(kExactListThreads) mask_exact_kernel(
    const int32_t* __restrict__ pred_geom, const int64_t* __restrict__ pred_offsets,
    const uint32_t* __restrict__ pred_bits, const int32_t* __restrict__ pred_areas,
    const int32_t* __restrict__ pred_order, const int32_t* __restrict__ gt_geom,
    const int64_t* __restrict__ gt_offsets, const uint32_t* __restrict__ gt_bits,
    const int32_t* __restrict__ gt_areas, const int32_t* __restrict__ cand_rank, const int32_t* __restrict__ cand_j,
    long long n, float* __restrict__ iou) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (kExactListThreads / 32);
  for (long long c = ((long long)blockIdx.x * kExactListThreads + threadIdx.x) >> 5; c < n; c += warps) {
    const int r = cand_rank[c], j = cand_j[c];
    const int row = pred_order ? pred_order[r] : r;
    const int4 a = reinterpret_cast<const int4*>(pred_geom)[row];
    const int4 b = reinterpret_cast<const int4*>(gt_geom)[j];
    const int inter = warp_window_intersection(a, pred_bits + pred_offsets[row], b, gt_bits + gt_offsets[j], lane);
    if (lane == 0) iou[c] = mask_iou(inter, pred_areas[row], gt_areas[j]);
  }
}

// Stable compaction of the candidates with iou >= iou_min (scan_common.cuh's launch_compaction)
struct KeepMatched {
  struct Shared {};
  const int32_t* cand_rank;
  const int32_t* cand_j;
  const float* cand_iou;
  long long n;
  float iou_min;
  int32_t* rank;
  int32_t* j;
  float* iou;
  __device__ void init(Shared&) const {}
  __device__ long long rows() const { return n; }
  __device__ bool keep(const Shared&, long long i) const { return cand_iou[i] >= iou_min; }
  __device__ void emit(const Shared&, long long i, long long slot) const {
    rank[slot] = cand_rank[i];
    j[slot] = cand_j[i];
    iou[slot] = cand_iou[i];
  }
};

// ---------------------------------------------------------------------------------------------- order
__global__ void __launch_bounds__(256) order_keys_kernel(const float* __restrict__ iou, long long n,
                                                         unsigned long long* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i < n) keys[i] = make_key(iou[i], (uint32_t)i);
}

static int grid_ok(float ox, float oy, float inv, int nx, int ny, const char* what) {
  HDY_REQUIRE(std::isfinite(ox) && std::isfinite(oy) && std::isfinite(inv) && inv > 0.0f, "%s: bad grid origin / cell size", what);
  HDY_REQUIRE(nx >= 1 && ny >= 1 && (long long)nx * ny < (1ll << 31), "%s: bad grid %d x %d", what, nx, ny);
  return HDY_OK;
}

static unsigned blocks_of(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_match_bin_stats(const float* gt_boxes, const int32_t* gt_geom, int G, uint64_t* stats, hdy_stream_t stream) {
  HDY_REQUIRE(G >= 0, "hdy_match_bin_stats: negative G");
  HDY_REQUIRE((gt_boxes == nullptr) != (gt_geom == nullptr), "hdy_match_bin_stats: pass gt_boxes or gt_geom");
  HDY_REQUIRE(stats != nullptr, "hdy_match_bin_stats: stats is NULL");
  const void* gt = gt_boxes ? (const void*)gt_boxes : (const void*)gt_geom;
  HDY_REQUIRE(((uintptr_t)gt & 15) == 0, "hdy_match_bin_stats: rectangles must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* s = reinterpret_cast<unsigned long long*>(stats);
  bin_stats_init_kernel<<<1, 32, 0, st>>>(s);
  if (G > 0) {
    if (gt_boxes)
      bin_stats_kernel<BOXES><<<blocks_of(G, kBinThreads), kBinThreads, 0, st>>>(gt, G, s);
    else
      bin_stats_kernel<WINDOWS><<<blocks_of(G, kBinThreads), kBinThreads, 0, st>>>(gt, G, s);
  }
  return check_launch("hdy_match_bin_stats");
}

int hdy_match_bin_entries(const float* gt_boxes, const int32_t* gt_geom, int G, float ox, float oy, float inv_cell,
                          int nx, int ny, int64_t* ent_off, uint64_t* cell_keys, hdy_stream_t stream) {
  HDY_REQUIRE(G >= 1, "hdy_match_bin_entries: G=%d", G);
  HDY_REQUIRE((gt_boxes == nullptr) != (gt_geom == nullptr), "hdy_match_bin_entries: pass gt_boxes or gt_geom");
  HDY_REQUIRE(ent_off != nullptr, "hdy_match_bin_entries: ent_off is NULL");
  const void* gt = gt_boxes ? (const void*)gt_boxes : (const void*)gt_geom;
  HDY_REQUIRE(((uintptr_t)gt & 15) == 0, "hdy_match_bin_entries: rectangles must be 16-byte aligned");
  int rc = grid_ok(ox, oy, inv_cell, nx, ny, "hdy_match_bin_entries");
  if (rc) return rc;
  const Grid g{ox, oy, inv_cell, nx, ny};
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* k = reinterpret_cast<unsigned long long*>(cell_keys);
  if (!cell_keys) {
    if (gt_boxes)
      device_exclusive_scan<int64_t, 4>(EntryCount<BOXES>{gt, g}, G, ent_off, ent_off + G, st);
    else
      device_exclusive_scan<int64_t, 4>(EntryCount<WINDOWS>{gt, g}, G, ent_off, ent_off + G, st);
  } else if (gt_boxes) {
    bin_emit_kernel<BOXES><<<blocks_of(G, kBinThreads), kBinThreads, 0, st>>>(gt, G, g, ent_off, k);
  } else {
    bin_emit_kernel<WINDOWS><<<blocks_of(G, kBinThreads), kBinThreads, 0, st>>>(gt, G, g, ent_off, k);
  }
  return check_launch("hdy_match_bin_entries");
}

int hdy_match_bin_cells(const uint64_t* cell_keys, int64_t E, int64_t n_cells, int64_t* cell_start,
                        hdy_stream_t stream) {
  HDY_REQUIRE(E >= 0 && n_cells >= 1 && n_cells < (1ll << 31), "hdy_match_bin_cells: E=%lld n_cells=%lld",
              (long long)E, (long long)n_cells);
  HDY_REQUIRE(cell_start && (cell_keys || E == 0), "hdy_match_bin_cells: NULL pointer");
  bin_cells_kernel<<<blocks_of(n_cells + 1, kBinThreads), kBinThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned long long*>(cell_keys), E, n_cells, cell_start);
  return check_launch("hdy_match_bin_cells");
}

static int pairs_args_ok(const void* pred, int P, const void* gt, int G, const int64_t* cell_start,
                         const uint64_t* cell_keys, float iou_min, const int64_t* off, const int32_t* rank,
                         const int32_t* j, const char* what) {
  HDY_REQUIRE(P >= 1 && G >= 1, "%s: P=%d G=%d", what, P, G);
  HDY_REQUIRE(iou_min > 0.0f, "%s: iou_min must be > 0 (the binning only finds pairs that overlap)", what);
  HDY_REQUIRE(pred && gt && cell_start && cell_keys && off, "%s: NULL pointer", what);
  HDY_REQUIRE((rank == nullptr) == (j == nullptr), "%s: pass both output lists or neither", what);
  HDY_REQUIRE((((uintptr_t)pred | (uintptr_t)gt) & 15) == 0, "%s: rectangles must be 16-byte aligned", what);
  return HDY_OK;
}

int hdy_match_boxes_binned(const float* pred_boxes, const int32_t* pred_order, int P, const float* gt_boxes, int G,
                           float ox, float oy, float inv_cell, int nx, int ny, const int64_t* cell_start,
                           const uint64_t* cell_keys, float iou_min, int64_t* pair_off, int32_t* pair_rank,
                           int32_t* pair_j, float* pair_iou, hdy_stream_t stream) {
  int rc = pairs_args_ok(pred_boxes, P, gt_boxes, G, cell_start, cell_keys, iou_min, pair_off, pair_rank, pair_j,
                         "hdy_match_boxes_binned");
  if (rc) return rc;
  HDY_REQUIRE((pair_rank == nullptr) == (pair_iou == nullptr), "hdy_match_boxes_binned: pair_iou with the lists");
  rc = grid_ok(ox, oy, inv_cell, nx, ny, "hdy_match_boxes_binned");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  pairs_kernel<BOXES><<<blocks_of(P, kPairThreads), kPairThreads, 0, st>>>(
      pred_boxes, nullptr, pred_order, P, gt_boxes, nullptr, Grid{ox, oy, inv_cell, nx, ny}, cell_start,
      reinterpret_cast<const unsigned long long*>(cell_keys), iou_min, pair_off, PairOut{pair_rank, pair_j, pair_iou});
  if (!pair_rank) device_exclusive_scan<int64_t, 4>(ArrayValues<int64_t>{pair_off}, P, pair_off, pair_off + P, st);
  return check_launch("hdy_match_boxes_binned");
}

int hdy_match_mask_candidates_binned(const int32_t* pred_geom, const int32_t* pred_areas, const int32_t* pred_order,
                                     int P, const int32_t* gt_geom, const int32_t* gt_areas, int G, float ox, float oy,
                                     float inv_cell, int nx, int ny, const int64_t* cell_start,
                                     const uint64_t* cell_keys, float iou_min, int64_t* cand_off, int32_t* cand_rank,
                                     int32_t* cand_j, hdy_stream_t stream) {
  int rc = pairs_args_ok(pred_geom, P, gt_geom, G, cell_start, cell_keys, iou_min, cand_off, cand_rank, cand_j,
                         "hdy_match_mask_candidates_binned");
  if (rc) return rc;
  HDY_REQUIRE(pred_areas && gt_areas, "hdy_match_mask_candidates_binned: NULL areas");
  rc = grid_ok(ox, oy, inv_cell, nx, ny, "hdy_match_mask_candidates_binned");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  pairs_kernel<WINDOWS><<<blocks_of(P, kPairThreads), kPairThreads, 0, st>>>(
      pred_geom, pred_areas, pred_order, P, gt_geom, gt_areas, Grid{ox, oy, inv_cell, nx, ny}, cell_start,
      reinterpret_cast<const unsigned long long*>(cell_keys), iou_min, cand_off, PairOut{cand_rank, cand_j, nullptr});
  if (!cand_rank) device_exclusive_scan<int64_t, 4>(ArrayValues<int64_t>{cand_off}, P, cand_off, cand_off + P, st);
  return check_launch("hdy_match_mask_candidates_binned");
}

int hdy_match_mask_exact_list(const int32_t* pred_geom, const int64_t* pred_offsets, const uint32_t* pred_bits,
                              const int32_t* pred_areas, const int32_t* pred_order, const int32_t* gt_geom,
                              const int64_t* gt_offsets, const uint32_t* gt_bits, const int32_t* gt_areas,
                              const int32_t* cand_rank, const int32_t* cand_j, int64_t n_cand, float iou_min,
                              float* cand_iou, int32_t* pair_rank, int32_t* pair_j, float* pair_iou,
                              int32_t* pair_count, int32_t* block_scratch, hdy_stream_t stream) {
  HDY_REQUIRE(n_cand >= 1 && n_cand < (1ll << 31), "hdy_match_mask_exact_list: n_cand=%lld", (long long)n_cand);
  HDY_REQUIRE(iou_min > 0.0f, "hdy_match_mask_exact_list: iou_min must be > 0");
  HDY_REQUIRE(pred_geom && pred_offsets && pred_bits && pred_areas && gt_geom && gt_offsets && gt_bits && gt_areas &&
                  cand_rank && cand_j && cand_iou && pair_rank && pair_j && pair_iou && pair_count && block_scratch,
              "hdy_match_mask_exact_list: NULL pointer");
  HDY_REQUIRE((((uintptr_t)pred_geom | (uintptr_t)gt_geom) & 15) == 0,
              "hdy_match_mask_exact_list: geom arrays must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const long long blocks = min((long long)kExactListMaxBlocks, ((long long)n_cand + 7) / 8);
  mask_exact_kernel<<<(unsigned)blocks, kExactListThreads, 0, st>>>(pred_geom, pred_offsets, pred_bits, pred_areas,
                                                                     pred_order, gt_geom, gt_offsets, gt_bits,
                                                                     gt_areas, cand_rank, cand_j, n_cand, cand_iou);
  launch_compaction(KeepMatched{cand_rank, cand_j, cand_iou, n_cand, iou_min, pair_rank, pair_j, pair_iou}, n_cand,
                    block_scratch, pair_count, st);
  return check_launch("hdy_match_mask_exact_list");
}

int hdy_match_order_keys(const float* ious, int64_t n, uint64_t* keys, hdy_stream_t stream) {
  HDY_REQUIRE(n >= 0 && n < (1ll << 31), "hdy_match_order_keys: n=%lld", (long long)n);
  if (n == 0) return HDY_OK;
  HDY_REQUIRE(ious && keys, "hdy_match_order_keys: NULL pointer");
  order_keys_kernel<<<blocks_of(n, 256), 256, 0, (cudaStream_t)stream>>>(
      ious, n, reinterpret_cast<unsigned long long*>(keys));
  return check_launch("hdy_match_order_keys");
}

}  // extern "C"
