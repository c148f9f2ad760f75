// Whole-slide tile merge: Detect.merge_outputs (T2) + Ensemble.merge (T3), sparse and exact.
//
// Reference: metayolo/models/yolo_head.py:450-471 (merge_outputs / rescale_outputs: shift tile-local boxes by the
// tile origin, concatenate, no NMS) and metayolo/models/yolo.py:165-204 (Ensemble.merge: keep scores > conf, one
// class-agnostic torchvision.ops.nms over ALL detections of the slide on their final scores, first max_det).
//
// torchvision's NMS is dense O(n^2) (338 s on the CPU at 2x10^5 boxes); a 100k x 100k px slide holds ~3x10^7
// detections.  The same result is produced here without ever forming a pair matrix:
//   * a detection can only be suppressed by a higher-scored box it intersects.  Boxes that survived the per-tile NMS
//     never suppress each other again when merge iou_thres >= tile iou_thres, so a detection whose box cannot reach
//     any other tile's detections ("interior": strictly inside its tile's core shrunk by the largest overhang of any
//     box over its tile) is KEPT outright; only the overlap-band detections enter the pairwise stage;
//   * band detections are binned by box centre into a torus hash grid (cell = 2 x mean box extent; boxes larger
//     than a cell go to one bucket everybody scans) and copied into cell order (box + 64-bit order key), so the 3x3
//     neighbourhood of a box is three contiguous runs;
//   * greedy NMS is resolved as a fixed point, in rounds: a box is KEPT once every intersecting (IoU > thr)
//     higher-ranked box is SUPPRESSED, SUPPRESSED as soon as one of them is KEPT.  Rank = (score desc, global index
//     asc), the order torchvision's stable sort visits boxes in; no global sort is needed for the verdicts;
//   * multi-GPU: entries [n_local, n) are replicas of seam detections owned by other ranks; they take part in every
//     test but their verdicts are imported from the owner between rounds (hdy_seam_export / hdy_seam_import).
// The IoU arithmetic is hdy_common.cuh's iou_gt (fp32, torchvision's operation order).  Binning only prunes pairs
// that cannot intersect, so it never changes a verdict.
//
// Also here: an LSD radix sort (8-bit digits, warp-private stable ranking) used to return survivors in the
// reference's score-descending order, and the small device-wide exclusive scan both need.
#include "hdy_common.cuh"

namespace hdy {

enum : uint8_t { MS_UNKNOWN = 0, MS_KEPT = 1, MS_SUPPRESSED = 2, MS_DROPPED = 3, MS_REMOTE_UNKNOWN = 4 };

constexpr int kMergeThreads = 256;
constexpr int kMaxRounds = 64;
constexpr float kMergeCellMargin = 1.01f;
constexpr float kMergeMaxScaled = 1.0e6f;

constexpr int kExtBins = 128;  // 8 bins per octave of max(w, h), 2^-2 .. 2^14 px
struct MergeStats {
  float ext_sum;
  unsigned ext_cnt;
  float cell_size;              // picked by merge_pick_cell_kernel
  unsigned ext_hist[kExtBins];
  int unknown[kMaxRounds + 1];  // unknown[r] = boxes still undecided after round r
  int rounds_run;
};

// ------------------------------------------------------------------------------------------------
// device-wide exclusive scan of int32 (in place), 3 phases, 4096 items per block
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ int block_scan_1024(int v, int* warp_tmp, int& total) {
  // inclusive scan over the block's `v`; returns this thread's exclusive prefix, total = block sum
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) warp_tmp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int s = warp_tmp[lane], t = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += u;
    }
    warp_tmp[lane] = t - s;
    if (lane == 31) warp_tmp[32] = t;
  }
  __syncthreads();
  const int excl = warp_tmp[warp] + incl - v;
  total = warp_tmp[32];
  __syncthreads();
  return excl;
}

__global__ void __launch_bounds__(kScanThreads) scan_reduce_kernel(const int* __restrict__ a, long long n,
                                                                    int* __restrict__ block_sums) {
  __shared__ int warp_tmp[33];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  int s = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k)
    if (base + k < n) s += a[base + k];
  int total;
  block_scan_1024(s, warp_tmp, total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) scan_sums_kernel(int* __restrict__ block_sums, int nblocks,
                                                                  int* __restrict__ total_out) {
  __shared__ int warp_tmp[33];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < nblocks; b0 += kScanThreads) {
    const int i = b0 + threadIdx.x;
    const int v = i < nblocks ? block_sums[i] : 0;
    int total;
    const int excl = block_scan_1024(v, warp_tmp, total);
    if (i < nblocks) block_sums[i] = carry + excl;
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0 && total_out) *total_out = carry;
}

__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(int* __restrict__ a, long long n,
                                                                   const int* __restrict__ block_sums) {
  __shared__ int warp_tmp[33];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  int v[kScanItems], s = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    v[k] = (base + k < n) ? a[base + k] : 0;
    s += v[k];
  }
  int total;
  int run = block_sums[blockIdx.x] + block_scan_1024(s, warp_tmp, total);
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    if (base + k < n) a[base + k] = run;
    run += v[k];
  }
}

static inline size_t scan_scratch_ints(long long n) { return (size_t)((n + kScanTile - 1) / kScanTile) + 1; }

// exclusive scan of a[0..n) in place; *total_out (device, may be NULL) receives the sum
static int device_exclusive_scan(int* a, long long n, int* scratch, int* total_out, cudaStream_t st) {
  if (n <= 0) return HDY_OK;
  const int nblocks = (int)((n + kScanTile - 1) / kScanTile);
  scan_reduce_kernel<<<nblocks, kScanThreads, 0, st>>>(a, n, scratch);
  scan_sums_kernel<<<1, kScanThreads, 0, st>>>(scratch, nblocks, total_out);
  scan_apply_kernel<<<nblocks, kScanThreads, 0, st>>>(a, n, scratch);
  return check_launch("device_exclusive_scan");
}

// ------------------------------------------------------------------------------------------------
// T2: tile-local detections -> slide coordinates, appended to flat arrays
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) append_offsets_kernel(const int32_t* __restrict__ counts, int bs,
                                                               long long* __restrict__ cursor,
                                                               long long* __restrict__ tile_offsets) {
  __shared__ int warp_tmp[33];
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = *cursor;
  __syncthreads();
  for (int b0 = 0; b0 < bs; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    const int v = i < bs ? max(counts[i], 0) : 0;
    int total;
    const int excl = block_scan_1024(v, warp_tmp, total);
    if (i < bs) tile_offsets[i] = carry + excl;
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    tile_offsets[bs] = carry;
    *cursor = carry;
  }
}

__global__ void append_tiles_kernel(const float4* __restrict__ boxes, const float* __restrict__ scores,
                                    const int64_t* __restrict__ labels, const uint8_t* __restrict__ fragile,
                                    const int32_t* __restrict__ counts,
                                    const float4* __restrict__ rois, int max_det, int tile_base, float scale,
                                    const long long* __restrict__ tile_offsets, long long capacity,
                                    float4* __restrict__ out_boxes, float* __restrict__ out_scores,
                                    int64_t* __restrict__ out_labels, int32_t* __restrict__ out_tile,
                                    int32_t* __restrict__ status) {
  const int tile = blockIdx.y;
  const int k = min(max(counts[tile], 0), max_det);
  const long long off = tile_offsets[tile];
  const float4 roi = rois[tile];
  for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < k; d += gridDim.x * blockDim.x) {
    const long long o = off + d;
    if (o >= capacity) {
      atomicOr(status, HDY_STATUS_OVERFLOW);
      continue;
    }
    const size_t s = (size_t)tile * max_det + d;
    float4 b = boxes[s];
    if (scale != 1.0f) {  // rescale_outputs: r['boxes'] *= scale          yolo_head.py:468-469
      b.x = __fmul_rn(b.x, scale);
      b.y = __fmul_rn(b.y, scale);
      b.z = __fmul_rn(b.z, scale);
      b.w = __fmul_rn(b.w, scale);
    }
    // boxes + [roi.x0, roi.y0, roi.x0, roi.y0]                             yolo_head.py:455
    b.x = __fadd_rn(b.x, roi.x);
    b.y = __fadd_rn(b.y, roi.y);
    b.z = __fadd_rn(b.z, roi.x);
    b.w = __fadd_rn(b.w, roi.y);
    out_boxes[o] = b;
    if (out_scores) out_scores[o] = scores[s];
    if (out_labels) out_labels[o] = labels[s];
    // fragile rows carry ~tile (negative): they still know their tile (overhang), but never take the shortcut
    if (out_tile) out_tile[o] = (fragile && fragile[s]) ? ~(tile_base + tile) : tile_base + tile;
  }
}

// ------------------------------------------------------------------------------------------------
// overhang of boxes over their own tile (slide coordinates)
// ------------------------------------------------------------------------------------------------
constexpr int kOverBins = 256;  // 1-px bins of ceil(overhang); the last one also takes everything beyond

__device__ __forceinline__ float box_overhang(const float4& b, const float4& r) {
  float o = fmaxf(fmaxf(r.x - b.x, r.y - b.y), fmaxf(b.z - r.z, b.w - r.w));
  if (!(o <= 3.0e38f)) o = 3.0e38f;  // NaN / inf coordinates: nothing is interior
  return o;
}

__global__ void overhang_hist_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ tile_id,
                                     const float4* __restrict__ tile_rois, const long long* __restrict__ n_dev,
                                     long long n_max, unsigned* __restrict__ hist) {
  __shared__ unsigned sh[kOverBins];
  for (int i = threadIdx.x; i < kOverBins; i += blockDim.x) sh[i] = 0u;
  __syncthreads();
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    int t = tile_id[i];
    if (t < 0) t = ~t;
    const float o = box_overhang(boxes[i], tile_rois[t]);
    if (o > 0.f) atomicAdd(&sh[o >= (float)(kOverBins - 1) ? kOverBins - 1 : (int)ceilf(o)], 1u);  // bin 0: inside
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kOverBins; i += blockDim.x)
    if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// The smallest whole-pixel cap in [min_cap, max_cap] that leaves at most max_far boxes sticking out further.  The
// margin every core is shrunk by is the largest overhang below the cap, so a handful of big false positives must not
// set it: at the 100k slide the largest overhang under a fixed 64 px cap is 63 px and 36 % of all rows stay active;
// nuclei themselves stick out by at most half their size.
__global__ void overhang_pick_kernel(const unsigned* __restrict__ hist, int max_far, float min_cap, float max_cap,
                                     float* __restrict__ cap_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int hi = (int)fminf(fmaxf(max_cap, 0.f), (float)(kOverBins - 2));
  int lo = (int)fminf(fmaxf(ceilf(min_cap), 0.f), (float)hi);
  unsigned long long above = 0;
  for (int b = kOverBins - 1; b > hi; --b) above += hist[b];
  int c = hi;
  while (c > lo && above + hist[c] <= (unsigned long long)max_far) above += hist[c--];
  *cap_out = (float)c;
}

__global__ void overhang_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ tile_id,
                                const float4* __restrict__ tile_rois, const long long* __restrict__ n_dev,
                                long long n_max, float far_cap, const float* __restrict__ far_cap_dev,
                                float* __restrict__ margin,
                                float4* __restrict__ far_boxes, int32_t* __restrict__ far_tile,
                                int32_t* __restrict__ far_count, int far_capacity) {
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  if (far_cap_dev) far_cap = *far_cap_dev;
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    int t = tile_id[i];
    if (t < 0) t = ~t;  // fragile row: ~tile
    const float4 b = boxes[i], r = tile_rois[t];
    const float o = box_overhang(b, r);
    if (far_count && o > far_cap) {
      // a box that reaches far beyond its tile (a rare, huge false positive) would shrink EVERY core through the
      // margin: list it instead, the tiles it touches lose the shortcut (dirty_tiles_kernel)
      const int k = atomicAdd(far_count, 1);
      if (k < far_capacity) {
        far_boxes[k] = b;
        far_tile[k] = t;
      }
    } else {
      m = fmaxf(m, o);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(reinterpret_cast<int*>(margin), __float_as_int(m));
}

// dirty[t] = 1 if a far-reaching box of ANOTHER tile intersects tile t's window (or the far list overflowed, or a far
// box is not finite): rows of dirty tiles never take the interior shortcut
__global__ void dirty_tiles_kernel(const float4* __restrict__ far_boxes, const int32_t* __restrict__ far_tile,
                                   const int32_t* __restrict__ far_count, int far_capacity,
                                   const float4* __restrict__ tile_rois, int n_tiles, uint8_t* __restrict__ dirty) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const int nf = *far_count;
  uint8_t d = nf > far_capacity ? 1 : 0;
  const float4 r = tile_rois[t];
  for (int k = 0; k < min(nf, far_capacity) && !d; ++k) {
    if (far_tile[k] == t) continue;
    const float4 b = far_boxes[k];
    const bool apart = (b.z < r.x) || (b.x > r.z) || (b.w < r.y) || (b.y > r.w);  // false for NaN: dirty
    if (!apart) d = 1;
  }
  dirty[t] = d;
}

// ------------------------------------------------------------------------------------------------
// merge NMS
// ------------------------------------------------------------------------------------------------
struct MergeWs {
  MergeStats* stats;
  int* cell;       // [G*G + 2] counts -> begin offsets -> end offsets
  int* scan_tmp;   // scan scratch
  float4* cbox;    // [n_max] boxes in cell order
  uint64_t* ckey;  // [n_max] order keys in cell order
  uint8_t* cstate; // [n_max]
  uint32_t* pos;   // [n_max] entry -> cell-order position (0xffffffff: not active)
  int32_t* ctile;     // per cell-ordered entry: tile of a local, non-fragile detection when the gray-zone flags are in
                      // force (tile_cores given), else negative
  uint32_t* blocked;  // per cell-ordered entry: round stamp of "a large dominator is still undecided"
  size_t bytes;
  int G;
};

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static int merge_grid_side(long long n_max) {
  // The torus only has to keep aliasing rare: with the interior shortcut a fifth of the rows is active, and a grid of
  // n_max / 2 buckets (16.8 M at the 100k slide: 67 MB, resident in L2 during the rounds) clears and scans four times
  // faster than one of 2 * n_max.  Any size is exact.
  int G = 64;
  while (G < 8192 && (long long)G * G < n_max / 2) G <<= 1;
  return G;
}

static MergeWs merge_layout(void* base, long long n_max) {
  MergeWs w;
  w.G = merge_grid_side(n_max);
  const size_t nb = (size_t)w.G * w.G + 2;
  size_t o = 0;
  unsigned char* p = static_cast<unsigned char*>(base);
  w.stats = reinterpret_cast<MergeStats*>(p + o);
  o += align256(sizeof(MergeStats));
  w.cell = reinterpret_cast<int*>(p + o);
  o += align256(nb * 4);
  w.scan_tmp = reinterpret_cast<int*>(p + o);
  o += align256(scan_scratch_ints((long long)nb) * 4);
  w.cbox = reinterpret_cast<float4*>(p + o);
  o += align256((size_t)n_max * 16);
  w.ckey = reinterpret_cast<uint64_t*>(p + o);
  o += align256((size_t)n_max * 8);
  w.pos = reinterpret_cast<uint32_t*>(p + o);
  o += align256((size_t)n_max * 4);
  w.cstate = reinterpret_cast<uint8_t*>(p + o);
  o += align256((size_t)n_max);
  w.blocked = reinterpret_cast<uint32_t*>(p + o);
  o += align256((size_t)n_max * 4);
  w.ctile = reinterpret_cast<int32_t*>(p + o);
  o += align256((size_t)n_max * 4);
  w.bytes = o;
  return w;
}

struct CellGeom {
  float cell_size, inv_cell, max_center;
};

__device__ __forceinline__ int ext_bin(float e) {
  const int b = (int)floorf(8.0f * log2f(e)) + 16;
  return min(max(b, 0), kExtBins - 1);
}
__device__ __forceinline__ float ext_bin_upper(int b) { return exp2f((float)(b - 16 + 1) * 0.125f) * 1.0001f; }

__device__ __forceinline__ CellGeom cell_geom(const MergeStats* s) {
  CellGeom g;
  float cs = s->cell_size;
  if (!(cs > 1e-20f) || !(cs < 1e30f)) cs = 1.0f;
  g.cell_size = cs;
  g.inv_cell = 1.0f / (cs * kMergeCellMargin);
  g.max_center = cs * kMergeMaxScaled;
  return g;
}

// 0: degenerate (never intersects anything), 1: small (bucket = torus cell), 2: large (bucket = G*G)
__device__ __forceinline__ int merge_classify_box(const float4& b, const CellGeom& g, int G, int& bucket, int& ix,
                                                  int& iy) {
  const float w = b.z - b.x, h = b.w - b.y;
  if (w <= 0.f || h <= 0.f) return 0;
  const float cx = (b.x + b.z) * 0.5f, cy = (b.y + b.w) * 0.5f;
  if (w <= g.cell_size && h <= g.cell_size && fabsf(cx) <= g.max_center && fabsf(cy) <= g.max_center) {
    ix = (int)floorf(cx * g.inv_cell);
    iy = (int)floorf(cy * g.inv_cell);
    bucket = (ix & (G - 1)) + (iy & (G - 1)) * G;
    return 1;
  }
  bucket = G * G;
  return 2;  // also NaN / inf coordinates
}

__global__ void merge_stats_kernel(const float4* __restrict__ boxes, const float* __restrict__ scores,
                                   const long long* __restrict__ n_dev, long long n_max, float conf,
                                   MergeStats* __restrict__ stats) {
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  __shared__ unsigned hist[kExtBins];
  for (int i = threadIdx.x; i < kExtBins; i += blockDim.x) hist[i] = 0u;
  __syncthreads();
  float sum = 0.f;
  unsigned cnt = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (!(scores[i] > conf)) continue;
    const float4 b = boxes[i];
    const float w = b.z - b.x, h = b.w - b.y;
    if (w > 0.f && h > 0.f && w < 3.0e38f && h < 3.0e38f) {
      sum += fmaxf(w, h);
      ++cnt;
      atomicAdd(&hist[ext_bin(fmaxf(w, h))], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kExtBins; i += blockDim.x)
    if (hist[i]) atomicAdd(&stats->ext_hist[i], hist[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0 && cnt) {
    atomicAdd(&stats->ext_sum, sum);
    atomicAdd(&stats->ext_cnt, cnt);
  }
}

// Cell size of the spatial hash: the smallest bin edge that leaves at most max(64, 0.05 %) of the boxes in the "large"
// bucket (one warp each), but never more than twice the mean extent.  A box is tested against the 3x3 cells around
// its centre, so the pair tests per box grow with the square of the cell size: for nuclei (12-36 px) this picks ~38 px
// where twice the mean is 48 px (-35 % pair tests).  Any value is exact; it only moves work between the two paths.
__global__ void merge_pick_cell_kernel(MergeStats* __restrict__ stats) {
  if (threadIdx.x != 0) return;
  const unsigned c = stats->ext_cnt;
  float cs = c ? 2.0f * (stats->ext_sum / (float)c) : 1.0f;
  if (c) {
    const unsigned allowed = max(64u, c / 2000u);
    unsigned above = 0;
    int b = kExtBins - 1;
    // walk down while the boxes in bins above b still fit the allowance
    while (b > 0 && above + stats->ext_hist[b] <= allowed) above += stats->ext_hist[b--];
    if (b < kExtBins - 1) cs = fminf(cs, ext_bin_upper(b));
  }
  stats->cell_size = cs;
}

struct MergeIn {
  const float4* boxes;
  const float* scores;
  const uint32_t* rep_gidx;   // optional global index of the replicas (entry n_local + k -> rep_gidx[k])
  const uint32_t* gidx_base_dev;  // optional device global index of entry 0: own entry i ranks as *gidx_base_dev + i
                                  // in score ties (NULL: i)
  int tile_base;              // tile_id[i] + tile_base indexes tile_cores / tile_dirty (ranks hold local tile ids)
  const int32_t* tile_id;     // optional
  const float4* tile_cores;   // optional [n_tiles] core rectangles (slide coordinates)
  const uint8_t* tile_dirty;  // optional [n_tiles]: tiles reached by another tile's far-reaching box (no shortcut)
  const float* margin;        // device float: largest overhang of any (not far-reaching) box over its tile
  const long long* n_dev;     // optional device count
  long long n_max, n_local;   // entries >= n_local are remote replicas
  float conf, thr;
};

// pass 1: initial verdicts, cell histogram.  state[i]: KEPT (interior / degenerate), DROPPED (<= conf), UNKNOWN (active)
__global__ void merge_classify_kernel(const MergeIn in, const MergeStats* __restrict__ stats, int G,
                                      int* __restrict__ cell, uint8_t* __restrict__ state) {
  const long long n = in.n_dev ? min(*in.n_dev, in.n_max) : in.n_max;
  const CellGeom g = cell_geom(stats);
  const float m = (in.tile_cores && in.margin) ? *in.margin : 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint8_t st = MS_UNKNOWN;
    const float4 b = in.boxes[i];
    if (!(in.scores[i] > in.conf)) {  // keep = scores > conf_thres                    yolo.py:189
      st = MS_DROPPED;
    } else {
      int bucket = 0, ix, iy;
      const int cls = merge_classify_box(b, g, G, bucket, ix, iy);
      const bool remote = i >= in.n_local;
      if (cls == 0 && !remote) {
        st = MS_KEPT;
      } else {
        bool interior = false;
        if (!remote && in.tile_cores && in.tile_id && in.tile_id[i] >= 0) {
          const int tg = in.tile_id[i] + in.tile_base;
          const float4 c = in.tile_cores[tg];
          interior = (b.x > c.x + m) && (b.y > c.y + m) && (b.z < c.z - m) && (b.w < c.w - m) &&
                     !(in.tile_dirty && in.tile_dirty[tg]);
        }
        if (interior)
          st = MS_KEPT;
        else
          atomicAdd(&cell[bucket], 1);
      }
    }
    state[i] = st;
  }
}

// pass 2: copy active entries into cell order
__global__ void merge_fill_kernel(const MergeIn in, const MergeStats* __restrict__ stats, int G,
                                  int* __restrict__ cell, const uint8_t* __restrict__ state,
                                  float4* __restrict__ cbox, uint64_t* __restrict__ ckey,
                                  uint8_t* __restrict__ cstate, uint32_t* __restrict__ pos,
                                  uint32_t* __restrict__ blocked, int32_t* __restrict__ ctile) {
  const long long n = in.n_dev ? min(*in.n_dev, in.n_max) : in.n_max;
  const CellGeom g = cell_geom(stats);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint32_t p = 0xffffffffu;
    if (state[i] == MS_UNKNOWN) {
      const float4 b = in.boxes[i];
      int bucket = 0, ix, iy;
      const int cls = merge_classify_box(b, g, G, bucket, ix, iy);
      p = (uint32_t)atomicAdd(&cell[bucket], 1);
      cbox[p] = b;
      const bool remote = i >= in.n_local;
      const uint32_t gi = (remote && in.rep_gidx) ? in.rep_gidx[i - in.n_local]
                                                  : (in.gidx_base_dev ? *in.gidx_base_dev : 0u) + (uint32_t)i;
      ckey[p] = make_key(in.scores[i], gi);
      cstate[p] = remote ? (uint8_t)MS_REMOTE_UNKNOWN : (cls == 0 ? (uint8_t)MS_KEPT : (uint8_t)MS_UNKNOWN);
      blocked[p] = 0u;
      ctile[p] = (!remote && in.tile_cores && in.tile_id) ? in.tile_id[i] : -1;
    }
    pos[i] = p;
  }
}

// One round of the fixed point over cell-ordered positions.  The two read-only directions of a round are kernels of
// their own.  (Round 2 tried them as ONE launch -- block ranges of a fused kernel -- to save a dependent launch per
// round at small per-rank sizes: no gain at N = 8, rounds 1.06 ms either way, and 5.8 -> 7.7 ms on one GPU, the
// small-box part inheriting the large part's register count.)
__global__ void __launch_bounds__(kMergeThreads) merge_round_kernel(const float4* __restrict__ cbox,
                                                                    const uint64_t* __restrict__ ckey, uint8_t* cstate,
                                                                    const int* __restrict__ cell, MergeStats* stats,
                                                                    int G, float thr, int round,
                                                                    const uint32_t* __restrict__ blocked,
                                                                    const int32_t* __restrict__ ctile) {
  if (round > 0 && stats->unknown[round - 1] == 0) {
    if (blockIdx.x == 0 && threadIdx.x == 0) stats->unknown[round] = 0;
    return;
  }
  const int NB = G * G + 1;
  const int large_begin = cell[NB - 2];
  const CellGeom g = cell_geom(stats);
  volatile uint8_t* vstate = cstate;
  int unknown = 0;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < large_begin; p += gridDim.x * blockDim.x) {
    if (vstate[p] != MS_UNKNOWN) continue;
    const float4 bi = cbox[p];
    const uint64_t ki = ckey[p];
    // Two survivors of the same tile's NMS that are not flagged fragile have IoU <= thr in slide coordinates too (the
    // gray-zone bound of hdy_nms_tiles, DESIGN.md 3.5): such a pair is never tested.  Fragile rows carry ~tile (< 0).
    const int ti = ctile[p];
    int decided = MS_KEPT;
    auto visit = [&](int q) -> bool {
      if (ckey[q] < ki && !(ti >= 0 && ctile[q] == ti) && iou_gt(cbox[q], bi, thr)) {
        const uint8_t sq = vstate[q];
        if (sq == MS_KEPT) {
          decided = MS_SUPPRESSED;
          return true;
        }
        if (sq == MS_UNKNOWN || sq == MS_REMOTE_UNKNOWN) decided = MS_UNKNOWN;
      }
      return false;
    };
    bool done = false;
    {
      const float cx = (bi.x + bi.z) * 0.5f, cy = (bi.y + bi.w) * 0.5f;
      const int ix = (int)floorf(cx * g.inv_cell), iy = (int)floorf(cy * g.inv_cell);
#pragma unroll 1
      for (int dy = -1; dy <= 1 && !done; ++dy) {
        const int rowb = ((iy + dy) & (G - 1)) * G;
#pragma unroll 1
        for (int dx = -1; dx <= 1 && !done; ++dx) {
          const int b = ((ix + dx) & (G - 1)) + rowb;
          const int beg = b ? cell[b - 1] : 0, end = cell[b];
          for (int q = beg; q < end; ++q)
            if (visit(q)) {
              done = true;
              break;
            }
        }
      }
    }
    // boxes of the large bucket that outrank this one are not scanned here (every small box would walk the whole
    // bucket): merge_large_push_kernel visits the small boxes under each large box instead -- it has already marked
    // this box SUPPRESSED if such a box is KEPT, and stamped it for this round if one is still undecided
    if (decided == MS_KEPT && blocked[p] == (uint32_t)round + 1u) decided = MS_UNKNOWN;
    if (decided != MS_UNKNOWN)
      vstate[p] = (uint8_t)decided;
    else
      unknown = 1;
  }
  unknown = __syncthreads_count(unknown);
  if (threadIdx.x == 0 && unknown) atomicAdd(&stats->unknown[round], unknown);
}

// Same round for the entries of the "large" bucket (boxes wider than a cell, or numerically awkward ones): ONE WARP
// per entry.  A large box can intersect small boxes whose centre lies within half a cell of it, i.e. the cells
// [floor((x1 - c/2) / cell), floor((x2 + c/2) / cell)] x [same in y]; the lanes share those cells (the whole grid if
// the range wraps around the torus, the whole array if the coordinates are not finite) and the large bucket.
__global__ void __launch_bounds__(kMergeThreads) merge_round_large_kernel(const float4* __restrict__ cbox,
                                                                          const uint64_t* __restrict__ ckey,
                                                                          uint8_t* cstate, const int* __restrict__ cell,
                                                                          MergeStats* stats, int G, float thr,
                                                                          int round) {
  if (round > 0 && stats->unknown[round - 1] == 0) return;
  const int NB = G * G + 1;
  const int n_active = cell[NB - 1];
  const int large_begin = cell[NB - 2];
  const CellGeom g = cell_geom(stats);
  volatile uint8_t* vstate = cstate;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int p = large_begin + warp; p < n_active; p += n_warps) {
    if (vstate[p] != MS_UNKNOWN) continue;  // warp-uniform
    const float4 bi = cbox[p];
    const uint64_t ki = ckey[p];
    int kept_dom = 0, unk_dom = 0;
    auto visit = [&](int q) {
      if (ckey[q] < ki && iou_gt(cbox[q], bi, thr)) {
        const uint8_t sq = vstate[q];
        if (sq == MS_KEPT) kept_dom = 1;
        if (sq == MS_UNKNOWN || sq == MS_REMOTE_UNKNOWN) unk_dom = 1;
      }
    };
    const float half = 0.5f * g.cell_size;
    const float fx0 = floorf((bi.x - half) * g.inv_cell), fx1 = floorf((bi.z + half) * g.inv_cell);
    const float fy0 = floorf((bi.y - half) * g.inv_cell), fy1 = floorf((bi.w + half) * g.inv_cell);
    const bool finite = fabsf(fx0) < 1.0e9f && fabsf(fx1) < 1.0e9f && fabsf(fy0) < 1.0e9f && fabsf(fy1) < 1.0e9f &&
                        fx1 >= fx0 && fy1 >= fy0;
    if (!finite) {
      for (int q = lane; q < large_begin; q += 32) visit(q);
    } else {
      const int ix0 = (int)fx0, iy0 = (int)fy0;
      const int nx = (int)fminf(fx1 - fx0 + 1.0f, (float)G), ny = (int)fminf(fy1 - fy0 + 1.0f, (float)G);
      const long long cells = (long long)nx * ny;
      for (long long c = lane; c < cells; c += 32) {
        const int cy = (int)(c / nx), cx = (int)(c - (long long)cy * nx);
        const int b = ((ix0 + cx) & (G - 1)) + ((iy0 + cy) & (G - 1)) * G;
        const int beg = b ? cell[b - 1] : 0, end = cell[b];
        for (int q = beg; q < end; ++q) visit(q);
      }
    }
    for (int q = large_begin + lane; q < n_active; q += 32) visit(q);
    kept_dom = __any_sync(0xffffffffu, kept_dom);
    unk_dom = __any_sync(0xffffffffu, unk_dom);
    if (lane == 0) {
      if (kept_dom)
        vstate[p] = (uint8_t)MS_SUPPRESSED;
      else if (!unk_dom)
        vstate[p] = (uint8_t)MS_KEPT;
      else
        atomicAdd(&stats->unknown[round], 1);
    }
  }
}

// Large -> small direction of a round: ONE WARP per entry of the large bucket that is not SUPPRESSED walks the small
// boxes it can intersect (same cell range as above).  A small box it outranks and overlaps (IoU > thr) is marked
// SUPPRESSED at once if the large box is KEPT, and stamped "blocked in this round" if the large box is still
// undecided, so merge_round_kernel never has to scan the large bucket (n_small x n_large pair tests otherwise: 7.5 of
// the 10.8 ms of the 100k slide's merge).  Runs before merge_round_kernel of the same round.
__global__ void __launch_bounds__(kMergeThreads) merge_large_push_kernel(const float4* __restrict__ cbox,
                                                                         const uint64_t* __restrict__ ckey,
                                                                         uint8_t* cstate, const int* __restrict__ cell,
                                                                         const MergeStats* stats, int G, float thr,
                                                                         int round, uint32_t* __restrict__ blocked) {
  if (round > 0 && stats->unknown[round - 1] == 0) return;
  const int NB = G * G + 1;
  const int n_active = cell[NB - 1];
  const int large_begin = cell[NB - 2];
  const CellGeom g = cell_geom(stats);
  volatile uint8_t* vstate = cstate;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t stamp = (uint32_t)round + 1u;
  for (int q = large_begin + warp; q < n_active; q += n_warps) {
    const uint8_t sq = vstate[q];  // warp-uniform
    if (sq != MS_KEPT && sq != MS_UNKNOWN && sq != MS_REMOTE_UNKNOWN) continue;
    const float4 bq = cbox[q];
    const uint64_t kq = ckey[q];
    auto visit = [&](int p) {
      if (kq < ckey[p] && vstate[p] == MS_UNKNOWN && iou_gt(bq, cbox[p], thr)) {
        if (sq == MS_KEPT)
          vstate[p] = (uint8_t)MS_SUPPRESSED;
        else
          blocked[p] = stamp;
      }
    };
    const float half = 0.5f * g.cell_size;
    const float fx0 = floorf((bq.x - half) * g.inv_cell), fx1 = floorf((bq.z + half) * g.inv_cell);
    const float fy0 = floorf((bq.y - half) * g.inv_cell), fy1 = floorf((bq.w + half) * g.inv_cell);
    const bool finite = fabsf(fx0) < 1.0e9f && fabsf(fx1) < 1.0e9f && fabsf(fy0) < 1.0e9f && fabsf(fy1) < 1.0e9f &&
                        fx1 >= fx0 && fy1 >= fy0;
    if (!finite) {
      for (int p = lane; p < large_begin; p += 32) visit(p);
    } else {
      const int ix0 = (int)fx0, iy0 = (int)fy0;
      const int nx = (int)fminf(fx1 - fx0 + 1.0f, (float)G), ny = (int)fminf(fy1 - fy0 + 1.0f, (float)G);
      const long long cells = (long long)nx * ny;
      for (long long c = lane; c < cells; c += 32) {
        const int cy = (int)(c / nx), cx = (int)(c - (long long)cy * nx);
        const int b = ((ix0 + cx) & (G - 1)) + ((iy0 + cy) & (G - 1)) * G;
        const int beg = b ? cell[b - 1] : 0, end = cell[b];
        for (int p = beg; p < end; ++p) visit(p);
      }
    }
  }
}

__global__ void merge_finish_kernel(const uint32_t* __restrict__ pos, const uint8_t* __restrict__ cstate,
                                    const long long* __restrict__ n_dev, long long n_max,
                                    uint8_t* __restrict__ state, int32_t* __restrict__ status) {
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  bool bad = false;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t p = pos[i];
    if (p == 0xffffffffu) continue;
    uint8_t s = cstate[p];
    if (s == MS_UNKNOWN || s == MS_REMOTE_UNKNOWN) {
      s = MS_UNKNOWN;
      bad = true;
    }
    state[i] = s;
  }
  if (bad && status) atomicOr(status, HDY_STATUS_ROUNDS);
}

// ------------------------------------------------------------------------------------------------
// survivors -> keys in row order, LSD radix sort, gather
// ------------------------------------------------------------------------------------------------
// Keys leave in ROW order, so that a stable sort on the score half alone (4 radix passes instead of 8) already breaks
// ties by the lower row.  Blocks own contiguous row ranges: count -> scan of the block counts -> write.
constexpr int kSelThreads = 256;
constexpr int kSelMaxBlocks = 4096;

__global__ void __launch_bounds__(kSelThreads) select_count_kernel(const uint8_t* __restrict__ state,
                                                                   const long long* __restrict__ n_dev,
                                                                   long long n_max, long long chunk,
                                                                   int* __restrict__ block_counts) {
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, n);
  int c = 0;
  for (long long i = lo + threadIdx.x; i < hi; i += kSelThreads) c += state[i] == MS_KEPT;
  __shared__ int part[kSelThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < kSelThreads / 32; ++w) t += part[w];
    block_counts[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(1024) select_scan_kernel(int* __restrict__ block_counts, int nblocks,
                                                           int* __restrict__ count_out) {
  __shared__ int warp_tmp[33];
  // nblocks <= kSelMaxBlocks = 4 x 1024: four consecutive entries per thread
  int v[4], s = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int i = threadIdx.x * 4 + j;
    v[j] = i < nblocks ? block_counts[i] : 0;
    s += v[j];
  }
  int total;
  int excl = block_scan_1024(s, warp_tmp, total);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int i = threadIdx.x * 4 + j;
    if (i < nblocks) block_counts[i] = excl;
    excl += v[j];
  }
  if (threadIdx.x == 0) *count_out = total;
}

__global__ void __launch_bounds__(kSelThreads) select_write_kernel(const uint8_t* __restrict__ state,
                                                                   const float* __restrict__ scores,
                                                                   const long long* __restrict__ n_dev,
                                                                   long long n_max, long long chunk,
                                                                   const int* __restrict__ block_offsets,
                                                                   uint64_t* __restrict__ keys) {
  __shared__ int wcount[kSelThreads / 32];
  const long long n = n_dev ? min(*n_dev, n_max) : n_max;
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, n);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long running = block_offsets[blockIdx.x];
  for (long long i0 = lo; i0 < hi; i0 += kSelThreads) {
    const long long i = i0 + threadIdx.x;
    const bool k = i < hi && state[i] == MS_KEPT;
    const unsigned m = __ballot_sync(0xffffffffu, k);
    if (lane == 0) wcount[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kSelThreads / 32; ++w) {
      const int c = wcount[w];
      if (w < warp) before += c;
      total += c;
    }
    if (k) keys[running + before + __popc(m & ((1u << lane) - 1u))] = make_key(scores[i], (uint32_t)i);
    running += total;
    __syncthreads();
  }
}

constexpr int kSortThreads = 256;                         // 8 warps
constexpr int kSortPerWarp = 1024;                        // keys per warp sub-tile
constexpr int kSortWarps = kSortThreads / 32;

// histogram of one digit per warp sub-tile: hist[digit * n_sub + sub]
__global__ void __launch_bounds__(kSortThreads) sort_hist_kernel(const uint64_t* __restrict__ keys,
                                                                  const int* __restrict__ n_dev, int n_max, int shift,
                                                                  int n_sub, int* __restrict__ hist) {
  __shared__ int h[kSortWarps][256];
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = blockIdx.x * kSortWarps + warp;
  for (int d = lane; d < 256; d += 32) h[warp][d] = 0;
  __syncwarp();
  const long long b = (long long)sub * kSortPerWarp;
  for (int k = lane; k < kSortPerWarp; k += 32)
    if (b + k < n) atomicAdd(&h[warp][(int)((keys[b + k] >> shift) & 255)], 1);
  __syncwarp();
  if (sub < n_sub)
    for (int d = lane; d < 256; d += 32) hist[(size_t)d * n_sub + sub] = h[warp][d];
}

__global__ void __launch_bounds__(kSortThreads) sort_scatter_kernel(const uint64_t* __restrict__ keys,
                                                                     const int* __restrict__ n_dev, int n_max,
                                                                     int shift, int n_sub, const int* __restrict__ hist,
                                                                     uint64_t* __restrict__ out) {
  __shared__ int base[kSortWarps][256];
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = blockIdx.x * kSortWarps + warp;
  if (sub >= n_sub) return;
  for (int d = lane; d < 256; d += 32) base[warp][d] = hist[(size_t)d * n_sub + sub];
  __syncwarp();
  const long long b = (long long)sub * kSortPerWarp;
  for (int k0 = 0; k0 < kSortPerWarp; k0 += 32) {
    const long long i = b + k0 + lane;
    const bool valid = i < n;
    const uint64_t key = valid ? keys[i] : 0;
    const int d = valid ? (int)((key >> shift) & 255) : 256 + lane;  // invalid lanes match nobody
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    int dst = 0;
    if (valid) dst = base[warp][d] + rank;
    __syncwarp();
    if (valid && rank == 0) base[warp][d] += __popc(peers);
    __syncwarp();
    if (valid) out[dst] = key;
  }
}

__global__ void merge_gather_kernel(const uint64_t* __restrict__ keys, const int* __restrict__ count, int max_det,
                                    const float4* __restrict__ boxes, const float* __restrict__ scores,
                                    const int64_t* __restrict__ labels, int64_t* __restrict__ out_idx,
                                    float4* __restrict__ out_boxes, float* __restrict__ out_scores,
                                    int64_t* __restrict__ out_labels, int* __restrict__ out_count) {
  const int k = min(*count, max_det);
  if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = k;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x) {
    const uint32_t i = key_index(keys[j]);
    if (out_idx) out_idx[j] = (int64_t)i;
    if (out_boxes) out_boxes[j] = boxes[i];
    if (out_scores) out_scores[j] = scores[i];  // (a random 4-byte read; key_score would canonicalise -0.0)
    if (out_labels && labels) out_labels[j] = labels[i];
  }
}

static inline unsigned blocks_for(long long n, int threads, int max_blocks = 148 * 16) {
  long long b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (unsigned)b;
}

// ------------------------------------------------------------------------------------------------
// multi-GPU seam exchange: fixed-size blocks, every size stays on the device (include/hd_yolo_b200.h)
// ------------------------------------------------------------------------------------------------
constexpr int kSeamHdr = HDY_SEAM_HDR_WORDS, kSeamFar = HDY_SEAM_FAR_WORDS, kSeamRow = HDY_SEAM_ROW_WORDS;
constexpr int kSeamMaxWorld = HDY_SEAM_MAX_WORLD;
// meta words (int32): see hdy_seam_scatter in the header
enum { SM_NTOTAL = 0, SM_MARGIN = 2, SM_GBASE = 3, SM_FLAGS = 4, SM_FAR_TOTAL = 5, SM_UNDECIDED = 8, SM_REP_OFF = 16,
       SM_OWN_SEAM = 88 };

__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  if (v >= 0.f)
    atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else
    atomicMax(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  if (v >= 0.f)
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else
    atomicMin(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}

// header + far list of this rank's summary block (the rectangle starts inverted; seam_rect_kernel folds the boxes in)
__global__ void seam_summary_pack_kernel(long long n_local, const float* __restrict__ margin,
                                         const float4* __restrict__ far_boxes, const int32_t* __restrict__ far_tile,
                                         const int32_t* __restrict__ far_count, int far_list_capacity, int tile_base,
                                         int far_cap, int32_t* __restrict__ block) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int nf = far_count ? *far_count : 0;
  if (k == 0) {
    float* f = reinterpret_cast<float*>(block);
    const float big = 3.0e38f;
    f[0] = big, f[1] = big, f[2] = -big, f[3] = -big;
    f[4] = margin ? *margin : 0.f;
    // a list that overflowed on the way here is reported as "more than far_cap": every tile turns dirty
    block[5] = nf > far_list_capacity ? far_cap + 1 : nf;
    *reinterpret_cast<long long*>(block + 6) = n_local;
    for (int i = 8; i < kSeamHdr; ++i) block[i] = 0;
  }
  if (k < far_cap) {
    int32_t* e = block + kSeamHdr + k * kSeamFar;
    if (k < min(nf, far_list_capacity)) {
      const float4 b = far_boxes[k];
      e[0] = __float_as_int(b.x), e[1] = __float_as_int(b.y), e[2] = __float_as_int(b.z), e[3] = __float_as_int(b.w);
      e[4] = far_tile[k] + tile_base;
    } else {
      e[0] = e[1] = e[2] = e[3] = 0, e[4] = -1;
    }
    e[5] = e[6] = e[7] = 0;
  }
}

__global__ void seam_rect_kernel(const float4* __restrict__ boxes, long long n, float* __restrict__ rect) {
  const float big = 3.0e38f;
  float x1 = big, y1 = big, x2 = -big, y2 = -big;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float4 b = boxes[i];  // fminf / fmaxf skip NaN coordinates: such a box intersects nothing anyway
    x1 = fminf(x1, fmaxf(b.x, -big)), y1 = fminf(y1, fmaxf(b.y, -big));
    x2 = fmaxf(x2, fminf(b.z, big)), y2 = fmaxf(y2, fminf(b.w, big));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    x1 = fminf(x1, __shfl_xor_sync(0xffffffffu, x1, o)), y1 = fminf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
    x2 = fmaxf(x2, __shfl_xor_sync(0xffffffffu, x2, o)), y2 = fmaxf(y2, __shfl_xor_sync(0xffffffffu, y2, o));
  }
  if ((threadIdx.x & 31) == 0 && x2 >= x1) {
    atomic_min_float(rect + 0, x1), atomic_min_float(rect + 1, y1);
    atomic_max_float(rect + 2, x2), atomic_max_float(rect + 3, y2);
  }
}

struct SeamRects {
  float4 r[kSeamMaxWorld];
  int live[kSeamMaxWorld];
};
__device__ __forceinline__ void seam_load_rects(SeamRects& S, const int32_t* summaries, int world, int rank, int hb) {
  for (int q = threadIdx.x; q < world; q += blockDim.x) {
    const int32_t* h = summaries + (size_t)q * hb;
    S.r[q] = make_float4(__int_as_float(h[0]), __int_as_float(h[1]), __int_as_float(h[2]), __int_as_float(h[3]));
    S.live[q] = (q != rank) && (*reinterpret_cast<const long long*>(h + 6) > 0);
  }
  __syncthreads();
}
// closed-interval test against every other rank's rectangle: a superset of "the boxes intersect", which is all
// exactness needs (hd_yolo_b200/dist.py)
__device__ __forceinline__ bool seam_row(const float4& b, const SeamRects& S, int world) {
  bool s = false;
  for (int q = 0; q < world; ++q)
    s |= S.live[q] && (b.z >= S.r[q].x) && (b.x <= S.r[q].z) && (b.w >= S.r[q].y) && (b.y <= S.r[q].w);
  return s;
}

__global__ void __launch_bounds__(kSelThreads) seam_count_kernel(const float4* __restrict__ boxes, long long n,
                                                                 long long chunk, const int32_t* __restrict__ summaries,
                                                                 int world, int rank, int hb,
                                                                 int* __restrict__ block_counts) {
  __shared__ SeamRects S;
  __shared__ int part[kSelThreads / 32];
  seam_load_rects(S, summaries, world, rank, hb);
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, n);
  int c = 0;
  for (long long i = lo + threadIdx.x; i < hi; i += kSelThreads) c += seam_row(boxes[i], S, world);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < kSelThreads / 32; ++w) t += part[w];
    block_counts[blockIdx.x] = t;
  }
}

// rows leave in ascending row order: payload row k = (box bits, score bits, global index) of own row sel[k]
__global__ void __launch_bounds__(kSelThreads) seam_write_kernel(const float4* __restrict__ boxes,
                                                                 const float* __restrict__ scores, long long n,
                                                                 long long chunk, const int32_t* __restrict__ summaries,
                                                                 int world, int rank, int hb,
                                                                 const int* __restrict__ block_offsets, int seam_cap,
                                                                 int32_t* __restrict__ sel, int32_t* __restrict__ block) {
  __shared__ SeamRects S;
  __shared__ int wcount[kSelThreads / 32];
  seam_load_rects(S, summaries, world, rank, hb);
  long long gbase = 0;  // rows owned by lower ranks
  for (int q = 0; q < rank; ++q) gbase += *reinterpret_cast<const long long*>(summaries + (size_t)q * hb + 6);
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, n);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long running = block_offsets[blockIdx.x];
  for (long long i0 = lo; i0 < hi; i0 += kSelThreads) {
    const long long i = i0 + threadIdx.x;
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    bool k = false;
    if (i < hi) {
      b = boxes[i];
      k = seam_row(b, S, world);
    }
    const unsigned m = __ballot_sync(0xffffffffu, k);
    if (lane == 0) wcount[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kSelThreads / 32; ++w) {
      const int c = wcount[w];
      if (w < warp) before += c;
      total += c;
    }
    const long long slot = running + before + __popc(m & ((1u << lane) - 1u));
    if (k && slot < seam_cap) {
      sel[slot] = (int32_t)i;
      int32_t* e = block + kSeamHdr + slot * kSeamRow;
      e[0] = __float_as_int(b.x), e[1] = __float_as_int(b.y), e[2] = __float_as_int(b.z), e[3] = __float_as_int(b.w);
      e[4] = __float_as_int(scores[i]);
      e[5] = (int32_t)(uint32_t)(gbase + i);
    }
    running += total;
    __syncthreads();
  }
}

__global__ void seam_block_header_kernel(const int* __restrict__ count, int32_t* __restrict__ block) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    block[0] = *count;
    for (int i = 1; i < kSeamHdr; ++i) block[i] = 0;
  }
}

// replicas: the other ranks' seam rows, rank by rank, appended behind the own rows; meta for the later steps
__global__ void seam_scatter_kernel(const int32_t* __restrict__ payloads, const int32_t* __restrict__ summaries,
                                    int world, int rank, int hb, int pb, int far_cap, int seam_cap, long long n_local,
                                    long long rep_cap, float4* __restrict__ boxes, float* __restrict__ scores,
                                    uint32_t* __restrict__ rep_gidx, int32_t* __restrict__ meta) {
  __shared__ int off[kSeamMaxWorld + 1];
  if (threadIdx.x == 0) {
    int run = 0, fl = 0, far_total = 0;
    float m = 0.f;
    long long gbase = 0, rows_all = 0;
    for (int q = 0; q < world; ++q) {
      off[q] = run;
      const int32_t* h = summaries + (size_t)q * hb;
      const int cnt = payloads[(size_t)q * pb];
      if (cnt > seam_cap) fl |= 1;
      if (q != rank) run += min(max(cnt, 0), seam_cap);
      m = fmaxf(m, __int_as_float(h[4]));
      if (h[5] > far_cap) fl |= 4;
      far_total += min(max(h[5], 0), far_cap);
      if (q < rank) gbase += *reinterpret_cast<const long long*>(h + 6);
      rows_all += *reinterpret_cast<const long long*>(h + 6);
    }
    off[world] = run;
    if (run > rep_cap) fl |= 2;
    if (rows_all >= (1ll << 32)) fl |= 8;  // global indices are 32-bit
    if (blockIdx.x == 0 && blockIdx.y == 0) {
      *reinterpret_cast<long long*>(meta + SM_NTOTAL) = n_local + min((long long)run, rep_cap);
      meta[SM_MARGIN] = __float_as_int(m);
      meta[SM_GBASE] = (int32_t)(uint32_t)gbase;
      meta[SM_FLAGS] = fl;
      meta[SM_FAR_TOTAL] = far_total;
      for (int e = 0; e < 8; ++e) meta[SM_UNDECIDED + e] = 0;
      for (int q = 0; q <= world; ++q) meta[SM_REP_OFF + q] = off[q];
      meta[SM_OWN_SEAM] = min(max(payloads[(size_t)rank * pb], 0), seam_cap);
    }
  }
  __syncthreads();
  const int q = blockIdx.y;
  if (q == rank) return;
  const int cnt = min(max(payloads[(size_t)q * pb], 0), seam_cap);
  const int32_t* src = payloads + (size_t)q * pb + kSeamHdr;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < cnt; j += gridDim.x * blockDim.x) {
    const long long r = (long long)off[q] + j;
    if (r >= rep_cap) break;
    const int32_t* e = src + (size_t)j * kSeamRow;
    boxes[n_local + r] = make_float4(__int_as_float(e[0]), __int_as_float(e[1]), __int_as_float(e[2]),
                                     __int_as_float(e[3]));
    scores[n_local + r] = __int_as_float(e[4]);
    rep_gidx[r] = (uint32_t)e[5];
  }
}

// dirty tiles from every rank's far list (global tile ids); all dirty when a list overflowed
__global__ void seam_dirty_tiles_kernel(const int32_t* __restrict__ summaries, int world, int hb, int far_cap,
                                        const float4* __restrict__ tile_rois, int n_tiles,
                                        uint8_t* __restrict__ dirty) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const float4 r = tile_rois[t];
  uint8_t d = 0;
  for (int q = 0; q < world && !d; ++q) {
    const int32_t* h = summaries + (size_t)q * hb;
    const int nf = h[5];
    if (nf > far_cap) d = 1;
    for (int k = 0; k < min(nf, far_cap) && !d; ++k) {
      const int32_t* e = h + kSeamHdr + k * kSeamFar;
      if (e[4] == t) continue;
      const float4 b = make_float4(__int_as_float(e[0]), __int_as_float(e[1]), __int_as_float(e[2]),
                                   __int_as_float(e[3]));
      const bool apart = (b.z < r.x) || (b.x > r.z) || (b.w < r.y) || (b.y > r.w);  // false for NaN: dirty
      if (!apart) d = 1;
    }
  }
  dirty[t] = d;
}

__global__ void seam_export_kernel(const uint32_t* __restrict__ pos, const uint8_t* __restrict__ cstate,
                                   const uint8_t* __restrict__ state, const int32_t* __restrict__ sel,
                                   const int32_t* __restrict__ my_block, int seam_cap, uint8_t* __restrict__ out) {
  const int m = min(max(my_block[0], 0), seam_cap);
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < m; k += gridDim.x * blockDim.x) {
    const int32_t i = sel[k];
    const uint32_t p = pos[i];
    out[k] = (p == 0xffffffffu) ? state[i] : cstate[p];
  }
}

// verdicts of the replicas from their owners; undecided[exchange] != 0 while any seam row anywhere is still open
__global__ void seam_import_kernel(const uint32_t* __restrict__ pos, uint8_t* __restrict__ cstate, long long n_local,
                                   const uint8_t* __restrict__ states, const int32_t* __restrict__ payloads, int pb,
                                   int32_t* __restrict__ meta, int world, int rank, int seam_cap, int exchange) {
  const int q = blockIdx.y;
  const int cnt = min(max(payloads[(size_t)q * pb], 0), seam_cap);
  const long long first = n_local + meta[SM_REP_OFF + q];
  const long long n_total = *reinterpret_cast<const long long*>(meta + SM_NTOTAL);
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) meta[SM_UNDECIDED + ((exchange + 1) & 7)] = 0;
  int open = 0;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < cnt; j += gridDim.x * blockDim.x) {
    const uint8_t s = states[(size_t)q * seam_cap + j];
    const bool decided = (s == MS_KEPT || s == MS_SUPPRESSED || s == MS_DROPPED);
    open |= !decided;
    if (q == rank || first + j >= n_total) continue;
    const uint32_t p = pos[first + j];
    if (p == 0xffffffffu) continue;
    cstate[p] = decided ? s : (uint8_t)MS_REMOTE_UNKNOWN;
  }
  if (__syncthreads_or(open) && threadIdx.x == 0) atomicOr(meta + SM_UNDECIDED + (exchange & 7), 1);
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_merge_append(const float* boxes, const float* scores, const int64_t* labels, const uint8_t* fragile,
                     const int32_t* counts, const float* rois, int bs, int max_det, int tile_base, float scale,
                     int64_t capacity,
                     float* out_boxes, float* out_scores, int64_t* out_labels, int32_t* out_tile, int64_t* cursor,
                     int64_t* tile_offsets, int32_t* status, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det > 0 && capacity >= 0, "hdy_merge_append: bad sizes");
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "hdy_merge_append: bs > 65535 (split the batch)");
  HDY_REQUIRE(boxes && counts && rois && out_boxes && cursor && tile_offsets && status, "hdy_merge_append: NULL pointer");
  HDY_REQUIRE((((uintptr_t)boxes | (uintptr_t)rois | (uintptr_t)out_boxes) & 15) == 0,
              "hdy_merge_append: box arrays must be 16-byte aligned");
  HDY_REQUIRE(!out_scores || scores, "hdy_merge_append: out_scores without scores");
  HDY_REQUIRE(!out_labels || labels, "hdy_merge_append: out_labels without labels");
  cudaStream_t st = (cudaStream_t)stream;
  append_offsets_kernel<<<1, 1024, 0, st>>>(counts, bs, reinterpret_cast<long long*>(cursor),
                                            reinterpret_cast<long long*>(tile_offsets));
  dim3 grid((unsigned)((max_det + 127) / 128), (unsigned)bs);
  append_tiles_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const float4*>(boxes), scores, labels, fragile, counts,
                                            reinterpret_cast<const float4*>(rois), max_det, tile_base, scale,
                                            reinterpret_cast<const long long*>(tile_offsets), capacity,
                                            reinterpret_cast<float4*>(out_boxes), out_scores, out_labels, out_tile,
                                            status);
  return check_launch("hdy_merge_append");
}

int hdy_merge_overhang_cap(const float* boxes, const int32_t* tile_id, const float* tile_rois, const int64_t* n_dev,
                           int64_t n_max, int max_far, float min_cap, float max_cap, uint32_t* hist, float* cap_out,
                           hdy_stream_t stream) {
  HDY_REQUIRE(n_max >= 0 && hist && cap_out && max_far >= 0, "hdy_merge_overhang_cap: bad arguments");
  HDY_REQUIRE(min_cap >= 0.f && max_cap >= min_cap, "hdy_merge_overhang_cap: need 0 <= min_cap <= max_cap");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(hist, 0, kOverBins * sizeof(uint32_t), st);
  if (e != cudaSuccess) {
    set_error("hdy_merge_overhang_cap: cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  if (n_max > 0) {
    HDY_REQUIRE(boxes && tile_id && tile_rois && (((uintptr_t)boxes | (uintptr_t)tile_rois) & 15) == 0,
                "hdy_merge_overhang_cap: NULL or misaligned pointer");
    overhang_hist_kernel<<<blocks_for(n_max, 256, 148 * 8), 256, 0, st>>>(
        reinterpret_cast<const float4*>(boxes), tile_id, reinterpret_cast<const float4*>(tile_rois),
        reinterpret_cast<const long long*>(n_dev), n_max, hist);
  }
  overhang_pick_kernel<<<1, 32, 0, st>>>(hist, max_far, min_cap, max_cap, cap_out);
  return check_launch("hdy_merge_overhang_cap");
}

int hdy_merge_overhang(const float* boxes, const int32_t* tile_id, const float* tile_rois, const int64_t* n_dev,
                       int64_t n_max, float far_cap, const float* far_cap_dev, float* margin, float* far_boxes,
                       int32_t* far_tile, int32_t* far_count, int far_capacity, hdy_stream_t stream) {
  HDY_REQUIRE(n_max >= 0 && margin, "hdy_merge_overhang: bad arguments");
  HDY_REQUIRE(!far_count || (far_boxes && far_tile && far_capacity >= 0 && ((uintptr_t)far_boxes & 15) == 0),
              "hdy_merge_overhang: far_count needs far_boxes (16-byte aligned) and far_tile");
  if (n_max == 0) return HDY_OK;
  HDY_REQUIRE(boxes && tile_id && tile_rois && (((uintptr_t)boxes | (uintptr_t)tile_rois) & 15) == 0,
              "hdy_merge_overhang: NULL or misaligned pointer");
  overhang_kernel<<<blocks_for(n_max, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(boxes), tile_id, reinterpret_cast<const float4*>(tile_rois),
      reinterpret_cast<const long long*>(n_dev), n_max, far_cap, far_cap_dev, margin,
      reinterpret_cast<float4*>(far_boxes), far_tile, far_count, far_capacity);
  return check_launch("hdy_merge_overhang");
}

int hdy_merge_dirty_tiles(const float* far_boxes, const int32_t* far_tile, const int32_t* far_count, int far_capacity,
                          const float* tile_rois, int n_tiles, uint8_t* dirty, hdy_stream_t stream) {
  HDY_REQUIRE(n_tiles >= 0 && far_capacity >= 0, "hdy_merge_dirty_tiles: bad sizes");
  if (n_tiles == 0) return HDY_OK;
  HDY_REQUIRE(far_boxes && far_tile && far_count && tile_rois && dirty &&
                  (((uintptr_t)far_boxes | (uintptr_t)tile_rois) & 15) == 0,
              "hdy_merge_dirty_tiles: NULL or misaligned pointer");
  dirty_tiles_kernel<<<(unsigned)((n_tiles + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(far_boxes), far_tile, far_count, far_capacity,
      reinterpret_cast<const float4*>(tile_rois), n_tiles, dirty);
  return check_launch("hdy_merge_dirty_tiles");
}

size_t hdy_merge_workspace_bytes(int64_t n_max) {
  if (n_max <= 0) return 256;
  return merge_layout(nullptr, n_max).bytes;
}

// The build step of hdy_merge_nms and hdy_seam_build (`what` names the call in error messages): initial verdicts,
// then the active entries copied into cell order.
static int merge_build_common(const char* what, MergeIn in, const float* tile_cores, uint8_t* state, void* workspace,
                              size_t workspace_bytes, cudaStream_t st) {
  const int64_t n_max = in.n_max, n_local = in.n_local;
  HDY_REQUIRE(n_max >= 0 && n_local >= 0 && n_local <= n_max, "%s: bad sizes", what);
  HDY_REQUIRE(n_max < (1ll << 31), "%s: at most 2^31-1 detections per call", what);
  HDY_REQUIRE(in.thr >= 0.f, "%s: iou_thres must be >= 0", what);
  HDY_REQUIRE(workspace && workspace_bytes >= hdy_merge_workspace_bytes(n_max), "%s: workspace too small", what);
  HDY_REQUIRE(!tile_cores || (in.tile_id && in.margin), "%s: tile_cores needs tile_id and margin", what);
  MergeWs w = merge_layout(workspace, n_max > 0 ? n_max : 1);
  const size_t nb = (size_t)w.G * w.G + 2;
  cudaError_t e = cudaMemsetAsync(w.stats, 0, sizeof(MergeStats), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(w.cell, 0, nb * 4, st);
  if (e != cudaSuccess) {
    set_error("%s: cudaMemsetAsync: %s", what, cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  if (n_max == 0) return HDY_OK;
  HDY_REQUIRE(in.boxes && in.scores && state && (((uintptr_t)in.boxes | (uintptr_t)tile_cores) & 15) == 0,
              "%s: NULL or misaligned pointer", what);
  const unsigned blocks = blocks_for(n_max, kMergeThreads);
  merge_stats_kernel<<<blocks, kMergeThreads, 0, st>>>(in.boxes, in.scores, in.n_dev, n_max, in.conf, w.stats);
  merge_pick_cell_kernel<<<1, 32, 0, st>>>(w.stats);
  merge_classify_kernel<<<blocks, kMergeThreads, 0, st>>>(in, w.stats, w.G, w.cell, state);
  int rc = device_exclusive_scan(w.cell, (long long)nb - 1, w.scan_tmp, nullptr, st);
  if (rc) return rc;
  merge_fill_kernel<<<blocks, kMergeThreads, 0, st>>>(in, w.stats, w.G, w.cell, state, w.cbox, w.ckey, w.cstate,
                                                      w.pos, w.blocked, w.ctile);
  return check_launch(what);
}

// ---- multi-GPU seam exchange -------------------------------------------------------------------
static inline int seam_hb(int far_cap) { return kSeamHdr + far_cap * kSeamFar; }
static inline int seam_pb(int seam_cap) { return kSeamHdr + seam_cap * kSeamRow; }

int hdy_seam_summary(const float* boxes, int64_t n_local, const float* margin, const float* far_boxes,
                     const int32_t* far_tile, const int32_t* far_count, int far_list_capacity, int tile_base,
                     int far_cap, int32_t* block, hdy_stream_t stream) {
  HDY_REQUIRE(n_local >= 0 && far_cap >= 0 && block, "hdy_seam_summary: bad arguments");
  HDY_REQUIRE(!far_count || (far_boxes && far_tile && far_list_capacity >= 0 && ((uintptr_t)far_boxes & 15) == 0),
              "hdy_seam_summary: far_count needs far_boxes (16-byte aligned) and far_tile");
  HDY_REQUIRE(n_local == 0 || (boxes && ((uintptr_t)boxes & 15) == 0), "hdy_seam_summary: NULL or misaligned boxes");
  cudaStream_t st = (cudaStream_t)stream;
  seam_summary_pack_kernel<<<(unsigned)(far_cap / 256 + 1), 256, 0, st>>>(
      n_local, margin, reinterpret_cast<const float4*>(far_boxes), far_tile, far_count, far_list_capacity, tile_base,
      far_cap, block);
  if (n_local > 0)
    seam_rect_kernel<<<blocks_for(n_local, 256, 148 * 4), 256, 0, st>>>(reinterpret_cast<const float4*>(boxes),
                                                                      n_local, reinterpret_cast<float*>(block));
  return check_launch("hdy_seam_summary");
}

int hdy_seam_select(const float* boxes, const float* scores, int64_t n_local, const int32_t* summaries, int world,
                    int rank, int far_cap, int seam_cap, int32_t* sel, int32_t* block, int32_t* block_scratch,
                    hdy_stream_t stream) {
  HDY_REQUIRE(n_local >= 0 && n_local < (1ll << 31) && world >= 1 && world <= kSeamMaxWorld && rank >= 0 &&
                  rank < world && far_cap >= 0 && seam_cap >= 0,
              "hdy_seam_select: bad arguments (world <= %d)", kSeamMaxWorld);
  HDY_REQUIRE(summaries && sel && block && block_scratch, "hdy_seam_select: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_local == 0) {
    cudaError_t e = cudaMemsetAsync(block, 0, kSeamHdr * 4, st);
    if (e != cudaSuccess) {
      set_error("hdy_seam_select: %s", cudaGetErrorString(e));
      return HDY_ERR_CUDA;
    }
    return HDY_OK;
  }
  HDY_REQUIRE(boxes && scores && ((uintptr_t)boxes & 15) == 0, "hdy_seam_select: NULL or misaligned pointer");
  long long chunk = (n_local + kSelMaxBlocks - 1) / kSelMaxBlocks;
  chunk = ((chunk + kSelThreads - 1) / kSelThreads) * kSelThreads;
  if (chunk < 4 * kSelThreads) chunk = 4 * kSelThreads;
  const int nblocks = (int)((n_local + chunk - 1) / chunk);
  const float4* b4 = reinterpret_cast<const float4*>(boxes);
  const int hb = seam_hb(far_cap);
  // block_scratch: [kSelMaxBlocks] block counts -> offsets, then the total
  seam_count_kernel<<<nblocks, kSelThreads, 0, st>>>(b4, n_local, chunk, summaries, world, rank, hb, block_scratch);
  select_scan_kernel<<<1, 1024, 0, st>>>(block_scratch, nblocks, block_scratch + kSelMaxBlocks);
  seam_block_header_kernel<<<1, 32, 0, st>>>(block_scratch + kSelMaxBlocks, block);
  seam_write_kernel<<<nblocks, kSelThreads, 0, st>>>(b4, scores, n_local, chunk, summaries, world, rank, hb,
                                                     block_scratch, seam_cap, sel, block);
  return check_launch("hdy_seam_select");
}

int hdy_seam_scatter(const int32_t* payloads, const int32_t* summaries, int world, int rank, int far_cap, int seam_cap,
                     int64_t n_local, int64_t rep_cap, float* boxes, float* scores, uint32_t* rep_gidx, int32_t* meta,
                     hdy_stream_t stream) {
  HDY_REQUIRE(world >= 1 && world <= kSeamMaxWorld && rank >= 0 && rank < world && far_cap >= 0 && seam_cap >= 0 &&
                  n_local >= 0 && rep_cap >= 0,
              "hdy_seam_scatter: bad arguments");
  HDY_REQUIRE(payloads && summaries && boxes && scores && rep_gidx && meta && ((uintptr_t)boxes & 15) == 0,
              "hdy_seam_scatter: NULL or misaligned pointer");
  dim3 grid((unsigned)(seam_cap / 1024 + 1), (unsigned)world);
  if (grid.x > 64) grid.x = 64;
  seam_scatter_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(payloads, summaries, world, rank, seam_hb(far_cap),
                                                            seam_pb(seam_cap), far_cap, seam_cap, n_local, rep_cap,
                                                            reinterpret_cast<float4*>(boxes), scores, rep_gidx, meta);
  return check_launch("hdy_seam_scatter");
}

int hdy_seam_dirty_tiles(const int32_t* summaries, int world, int far_cap, const float* tile_rois, int n_tiles,
                         uint8_t* dirty, hdy_stream_t stream) {
  HDY_REQUIRE(world >= 1 && far_cap >= 0 && n_tiles >= 0, "hdy_seam_dirty_tiles: bad sizes");
  if (n_tiles == 0) return HDY_OK;
  HDY_REQUIRE(summaries && tile_rois && dirty && ((uintptr_t)tile_rois & 15) == 0,
              "hdy_seam_dirty_tiles: NULL or misaligned pointer");
  seam_dirty_tiles_kernel<<<(unsigned)((n_tiles + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      summaries, world, seam_hb(far_cap), far_cap, reinterpret_cast<const float4*>(tile_rois), n_tiles, dirty);
  return check_launch("hdy_seam_dirty_tiles");
}

int hdy_seam_build(const float* boxes, const float* scores, const uint32_t* rep_gidx, const int32_t* meta,
                   const int32_t* tile_id, int tile_base, const float* tile_cores, const uint8_t* tile_dirty,
                   int64_t n_max, int64_t n_local, float conf_thres, float iou_thres, uint8_t* state, void* workspace,
                   size_t workspace_bytes, hdy_stream_t stream) {
  HDY_REQUIRE(meta && rep_gidx, "hdy_seam_build: NULL pointer");
  MergeIn in;
  in.boxes = reinterpret_cast<const float4*>(boxes);
  in.scores = scores;
  in.rep_gidx = rep_gidx;
  in.gidx_base_dev = reinterpret_cast<const uint32_t*>(meta + SM_GBASE);
  in.tile_base = tile_base;
  in.tile_id = tile_id;
  in.tile_cores = reinterpret_cast<const float4*>(tile_cores);
  in.tile_dirty = tile_dirty;
  in.margin = reinterpret_cast<const float*>(meta + SM_MARGIN);
  in.n_dev = reinterpret_cast<const long long*>(meta + SM_NTOTAL);
  in.n_max = n_max;
  in.n_local = n_local;
  in.conf = conf_thres;
  in.thr = iou_thres;
  return merge_build_common("hdy_seam_build", in, tile_cores, state, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hdy_seam_export(void* workspace, int64_t n_max, const uint8_t* state, const int32_t* sel, const int32_t* my_block,
                    int seam_cap, uint8_t* out, hdy_stream_t stream) {
  HDY_REQUIRE(workspace && n_max >= 0 && seam_cap >= 0, "hdy_seam_export: bad arguments");
  if (seam_cap == 0 || n_max == 0) return HDY_OK;
  HDY_REQUIRE(state && sel && my_block && out, "hdy_seam_export: NULL pointer");
  MergeWs w = merge_layout(workspace, n_max);
  seam_export_kernel<<<blocks_for(seam_cap, 256, 148), 256, 0, (cudaStream_t)stream>>>(w.pos, w.cstate, state, sel,
                                                                                    my_block, seam_cap, out);
  return check_launch("hdy_seam_export");
}

int hdy_seam_import(void* workspace, int64_t n_max, int64_t n_local, const uint8_t* states, const int32_t* payloads,
                    int32_t* meta, int world, int rank, int seam_cap, int exchange, hdy_stream_t stream) {
  HDY_REQUIRE(workspace && n_max >= 0 && n_local >= 0 && world >= 1 && world <= kSeamMaxWorld && rank >= 0 &&
                  rank < world && seam_cap >= 0 && exchange >= 0,
              "hdy_seam_import: bad arguments");
  HDY_REQUIRE(states && payloads && meta, "hdy_seam_import: NULL pointer");
  MergeWs w = merge_layout(workspace, n_max > 0 ? n_max : 1);
  dim3 grid((unsigned)(seam_cap / 1024 + 1), (unsigned)world);
  if (grid.x > 64) grid.x = 64;
  seam_import_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w.pos, w.cstate, n_local, states, payloads,
                                                           seam_pb(seam_cap), meta, world, rank, seam_cap, exchange);
  return check_launch("hdy_seam_import");
}

int hdy_merge_rounds(void* workspace, int64_t n_max, float iou_thres, int first_round, int n_rounds,
                     hdy_stream_t stream) {
  HDY_REQUIRE(workspace && n_max >= 0, "hdy_merge_rounds: bad arguments");
  HDY_REQUIRE(first_round >= 0 && n_rounds >= 0 && first_round + n_rounds <= kMaxRounds,
              "hdy_merge_rounds: at most %d rounds in total", kMaxRounds);
  if (n_max == 0) return HDY_OK;
  MergeWs w = merge_layout(workspace, n_max);
  const unsigned blocks = blocks_for(n_max, kMergeThreads, 148 * 8);
  for (int r = first_round; r < first_round + n_rounds; ++r) {
    merge_large_push_kernel<<<148 * 2, kMergeThreads, 0, (cudaStream_t)stream>>>(w.cbox, w.ckey, w.cstate, w.cell,
                                                                                 w.stats, w.G, iou_thres, r, w.blocked);
    merge_round_kernel<<<blocks, kMergeThreads, 0, (cudaStream_t)stream>>>(w.cbox, w.ckey, w.cstate, w.cell, w.stats,
                                                                           w.G, iou_thres, r, w.blocked, w.ctile);
    merge_round_large_kernel<<<148 * 2, kMergeThreads, 0, (cudaStream_t)stream>>>(w.cbox, w.ckey, w.cstate, w.cell,
                                                                                  w.stats, w.G, iou_thres, r);
  }
  return check_launch("hdy_merge_rounds");
}

int hdy_merge_finish(void* workspace, const int64_t* n_dev, int64_t n_max, uint8_t* state, int32_t* status,
                     hdy_stream_t stream) {
  HDY_REQUIRE(workspace && n_max >= 0, "hdy_merge_finish: bad arguments");
  if (n_max == 0) return HDY_OK;
  HDY_REQUIRE(state != nullptr, "hdy_merge_finish: state is NULL");
  MergeWs w = merge_layout(workspace, n_max);
  merge_finish_kernel<<<blocks_for(n_max, 256), 256, 0, (cudaStream_t)stream>>>(
      w.pos, w.cstate, reinterpret_cast<const long long*>(n_dev), n_max, state, status);
  return check_launch("hdy_merge_finish");
}

int hdy_merge_nms(const float* boxes, const float* scores, const int32_t* tile_id, const float* tile_cores,
                  const uint8_t* tile_dirty, const float* margin, const int64_t* n_dev, int64_t n_max, float conf_thres,
                  float iou_thres,
                  int max_rounds, uint8_t* state, int32_t* status, void* workspace, size_t workspace_bytes,
                  hdy_stream_t stream) {
  HDY_REQUIRE(max_rounds >= 1 && max_rounds <= kMaxRounds, "hdy_merge_nms: max_rounds out of range [1,%d]", kMaxRounds);
  MergeIn in;
  in.boxes = reinterpret_cast<const float4*>(boxes);
  in.scores = scores;
  in.rep_gidx = nullptr;
  in.gidx_base_dev = nullptr;
  in.tile_base = 0;
  in.tile_id = tile_id;
  in.tile_cores = reinterpret_cast<const float4*>(tile_cores);
  in.tile_dirty = tile_dirty;
  in.margin = margin;
  in.n_dev = reinterpret_cast<const long long*>(n_dev);
  in.n_max = n_max;
  in.n_local = n_max;
  in.conf = conf_thres;
  in.thr = iou_thres;
  int rc = merge_build_common("hdy_merge_nms", in, tile_cores, state, workspace, workspace_bytes, (cudaStream_t)stream);
  if (rc) return rc;
  rc = hdy_merge_rounds(workspace, n_max, iou_thres, 0, max_rounds, stream);
  if (rc) return rc;
  return hdy_merge_finish(workspace, n_dev, n_max, state, status, stream);
}

size_t hdy_sort_workspace_bytes(int64_t n_max) {
  if (n_max <= 0) return 256;
  const long long n_sub = (n_max + kSortPerWarp - 1) / kSortPerWarp;
  const long long hist = 256 * n_sub;
  return align256((size_t)hist * 4) + align256(scan_scratch_ints(hist) * 4);
}

int hdy_sort_keys_bytes(uint64_t* keys, uint64_t* tmp, const int32_t* n_dev, int64_t n_max, int first_byte,
                        int n_bytes, void* workspace, size_t workspace_bytes, hdy_stream_t stream) {
  HDY_REQUIRE(first_byte >= 0 && n_bytes >= 0 && first_byte + n_bytes <= 8 && (n_bytes & 1) == 0,
              "hdy_sort_keys_bytes: bytes [%d, %d) -- an even number of bytes inside the key", first_byte,
              first_byte + n_bytes);
  HDY_REQUIRE(n_max >= 0 && n_max < (1ll << 31), "hdy_sort_keys_bytes: bad size");
  if (n_max == 0) return HDY_OK;
  HDY_REQUIRE(keys && tmp && workspace && workspace_bytes >= hdy_sort_workspace_bytes(n_max),
              "hdy_sort_keys_bytes: NULL pointer or workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_sub = (int)((n_max + kSortPerWarp - 1) / kSortPerWarp);
  const long long hist_n = 256ll * n_sub;
  int* hist = static_cast<int*>(workspace);
  int* scratch = reinterpret_cast<int*>(static_cast<unsigned char*>(workspace) + align256((size_t)hist_n * 4));
  const unsigned blocks = (unsigned)((n_sub + kSortWarps - 1) / kSortWarps);
  uint64_t* src = keys;
  uint64_t* dst = tmp;
  for (int pass = first_byte; pass < first_byte + n_bytes; ++pass) {
    sort_hist_kernel<<<blocks, kSortThreads, 0, st>>>(src, n_dev, (int)n_max, pass * 8, n_sub, hist);
    int rc = device_exclusive_scan(hist, hist_n, scratch, nullptr, st);
    if (rc) return rc;
    sort_scatter_kernel<<<blocks, kSortThreads, 0, st>>>(src, n_dev, (int)n_max, pass * 8, n_sub, hist, dst);
    uint64_t* t = src;
    src = dst;
    dst = t;
  }
  return check_launch("hdy_sort_keys_bytes");  // an even number of passes: the result is back in `keys`
}

int hdy_merge_select_ordered(const uint8_t* state, const float* scores, const int64_t* n_dev, int64_t n_max,
                             uint64_t* keys, int32_t* count, int32_t* block_scratch, hdy_stream_t stream) {
  HDY_REQUIRE(n_max >= 0 && n_max < (1ll << 31) && count && block_scratch, "hdy_merge_select_ordered: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_max == 0) {
    cudaError_t e = cudaMemsetAsync(count, 0, 4, st);
    if (e != cudaSuccess) {
      set_error("hdy_merge_select_ordered: %s", cudaGetErrorString(e));
      return HDY_ERR_CUDA;
    }
    return HDY_OK;
  }
  HDY_REQUIRE(state && scores && keys, "hdy_merge_select_ordered: NULL pointer");
  // contiguous row ranges, a multiple of the block size, at most kSelMaxBlocks of them
  long long chunk = (n_max + kSelMaxBlocks - 1) / kSelMaxBlocks;
  chunk = ((chunk + kSelThreads - 1) / kSelThreads) * kSelThreads;
  if (chunk < 4 * kSelThreads) chunk = 4 * kSelThreads;
  const int nblocks = (int)((n_max + chunk - 1) / chunk);
  const long long* nd = reinterpret_cast<const long long*>(n_dev);
  select_count_kernel<<<nblocks, kSelThreads, 0, st>>>(state, nd, n_max, chunk, block_scratch);
  select_scan_kernel<<<1, 1024, 0, st>>>(block_scratch, nblocks, count);
  select_write_kernel<<<nblocks, kSelThreads, 0, st>>>(state, scores, nd, n_max, chunk, block_scratch, keys);
  return check_launch("hdy_merge_select_ordered");
}

int hdy_merge_gather(const uint64_t* keys, const int32_t* count, int64_t max_det, const float* boxes,
                     const float* scores, const int64_t* labels, int64_t* out_idx, float* out_boxes,
                     float* out_scores, int64_t* out_labels, int32_t* out_count, hdy_stream_t stream) {
  HDY_REQUIRE(max_det >= 0 && max_det < (1ll << 31) && keys && count && out_count, "hdy_merge_gather: bad arguments");
  HDY_REQUIRE((!out_boxes || boxes) && (!out_scores || scores), "hdy_merge_gather: output without its source");
  HDY_REQUIRE((((uintptr_t)boxes | (uintptr_t)out_boxes) & 15) == 0, "hdy_merge_gather: box arrays must be 16-byte aligned");
  merge_gather_kernel<<<blocks_for(max_det > 0 ? max_det : 1, 256), 256, 0, (cudaStream_t)stream>>>(
      keys, count, (int)max_det, reinterpret_cast<const float4*>(boxes), scores, labels, out_idx,
      reinterpret_cast<float4*>(out_boxes), out_scores, out_labels, out_count);
  return check_launch("hdy_merge_gather");
}

}  // extern "C"
