// Prediction <-> ground-truth matching by MASK IoU, over the cropped bit-packed layout (PackedMasks): the
// iou_type='masks' branch of APMeter.add (metayolo/models/metrics.py:270-303).
//
// The reference builds dense [k,1,H,W] fp32 masks (paste_masks_in_image) and a dense k x g overlap matrix -- 12.6 GB
// of predicted masks per 1024 px image at k = 3 000.  Here a mask is its tight window plus its bit plane (~100-300 B
// per nucleus), two windows that do not overlap cannot intersect, and only the few pairs whose windows overlap are
// counted, exactly:
//   * bounds_kernel + pack_kernel (hdy_pack_masks_geometry / hdy_pack_masks): dense [K,H,W] masks -> tight windows
//     (bounding rectangle of the set pixels; empty mask: w = h = 0) -> word offsets (device_exclusive_scan) -> bits;
//   * areas_kernel (hdy_mask_areas): popcount per mask, padding bits of each row's last word masked off;
//   * candidates_kernel: one thread per prediction in score rank order against every ground-truth window, keeps the
//     pairs whose windows overlap and whose IoU UPPER BOUND reaches iou_min;
//   * exact_kernel: one warp per candidate counts the intersection over the overlap rectangle and appends the pairs
//     with iou >= iou_min as order keys ~orderable(iou) << 32 | (rank * g + j), the box path's keys (match.cu).
// A pixel is set iff its value is > 0.5 (fp32 / fp16) or nonzero (uint8 / bool).  iou = float(inter) / float(union),
// both conversions and the division rounded to nearest: what `inter.float() / union.float()` gives in torch.
#include "match_common.cuh"
#include "scan_common.cuh"

namespace hdy {

// ---------------------------------------------------------------------------------------------- dense -> windows
// Element i of a dense mask is set?
template <int DT>
__device__ __forceinline__ bool elem_set(const void* p, size_t i) {
  if (DT == HDY_F32) return reinterpret_cast<const float*>(p)[i] > 0.5f;
  if (DT == HDY_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]) > 0.5f;
  return reinterpret_cast<const uint8_t*>(p)[i] != 0;
}

// Set flags of the elements of one 16-byte vector, bit e for element e (4, 8 or 16 elements).
template <int DT>
__device__ __forceinline__ uint32_t vec_set_bits(const int4 v) {
  const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (DT == HDY_F32) {
      m |= (uint32_t)(__uint_as_float(w[k]) > 0.5f) << k;
    } else if (DT == HDY_F16) {
      const __half2 h = *reinterpret_cast<const __half2*>(&w[k]);
      m |= ((uint32_t)(__low2float(h) > 0.5f) | ((uint32_t)(__high2float(h) > 0.5f) << 1)) << (2 * k);
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b) m |= (uint32_t)(((w[k] >> (8 * b)) & 0xffu) != 0) << (4 * k + b);
    }
  }
  return m;
}

constexpr int kBoundsThreads = 256;
constexpr int kBoundsUnroll = 4;       // 16-byte vectors in flight per thread
constexpr int kBoundsIters = 4;        // rounds per CTA: a CTA covers 256 * 4 * 4 * 16 B = 64 KB of one mask
constexpr long long kBoundsScalarChunk = 16384;

struct Bounds {
  int x0, y0, x1, y1;  // inclusive pixel bounds of the set pixels seen so far (x0 > x1 while none)
  __device__ void add(int e, int W) {  // e: element index inside the mask (H * W < 2^31)
    const int y = e / W, x = e - y * W;
    x0 = min(x0, x);
    x1 = max(x1, x);
    y0 = min(y0, y);
    y1 = max(y1, y);
  }
};

// Pass 1: the bounding rectangle of every mask's set pixels, reduced into geom4[i] as four atomicMax targets that start
// at zero (the caller clears geom4): (W - min x, H - min y, max x + 1, max y + 1), all four > 0 iff a pixel is set.
// CTA b takes slice b % slices of mask b / slices.  Every dense byte is read once (streaming, no L1 allocation).
template <int DT, bool VEC>
__global__ void __launch_bounds__(kBoundsThreads) bounds_kernel(const void* __restrict__ masks, int H, int W,
                                                                int slices, int32_t* __restrict__ geom4) {
  constexpr int kEsz = DT == HDY_F32 ? 4 : DT == HDY_F16 ? 2 : 1;
  constexpr int kElems = 16 / kEsz;
  const long long i = blockIdx.x / slices;
  const int slice = (int)(blockIdx.x - i * slices);
  const long long N = (long long)H * W;
  Bounds b{W, H, -1, -1};
  if (VEC) {
    const int4* v = reinterpret_cast<const int4*>(reinterpret_cast<const char*>(masks) + (size_t)i * N * kEsz);
    const long long nv = N / kElems;
    constexpr long long kSlice = (long long)kBoundsThreads * kBoundsUnroll * kBoundsIters;
    const long long lo = (long long)slice * kSlice, hi = min(lo + kSlice, nv);
    for (long long r = lo + threadIdx.x; r < hi; r += (long long)kBoundsThreads * kBoundsUnroll) {
      int4 x[kBoundsUnroll];
#pragma unroll
      for (int u = 0; u < kBoundsUnroll; ++u) {
        const long long q = r + (long long)u * kBoundsThreads;
        x[u] = q < hi ? __ldcs(v + q) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < kBoundsUnroll; ++u) {
        // rare for nuclei: a few hundred set pixels in a 10^6-pixel canvas
        const int e0 = (int)((r + (long long)u * kBoundsThreads) * kElems);
        for (uint32_t m = vec_set_bits<DT>(x[u]); m; m &= m - 1) b.add(e0 + __ffs(m) - 1, W);
      }
    }
  } else {
    const long long lo = (long long)slice * kBoundsScalarChunk, hi = min(lo + kBoundsScalarChunk, N);
    const size_t base = (size_t)i * N;
    for (long long e = lo + threadIdx.x; e < hi; e += kBoundsThreads)
      if (elem_set<DT>(masks, base + e)) b.add((int)e, W);
  }
  // CTA reduction of the four extrema, then one set of atomics per CTA that saw a set pixel
  int v4[4] = {W - b.x0, H - b.y0, b.x1 + 1, b.y1 + 1};  // all 0 when nothing was set
  __shared__ int red[kBoundsThreads / 32][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v4[k] = __reduce_max_sync(0xffffffffu, v4[k]);
    if (lane == 0) red[warp][k] = v4[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    int m = 0;
    for (int w = 0; w < kBoundsThreads / 32; ++w) m = max(m, red[w][threadIdx.x]);
    if (m > 0) atomicMax(geom4 + 4 * i + threadIdx.x, m);
  }
}

// words(i) of the scan: turns geom4[i] from the reduced bounds into the window {x0, y0, w, h} on the way
struct BoundsWindowWords {
  int32_t* geom4;
  int H, W;
  __device__ int64_t operator()(long long i) const {
    const int4 b = reinterpret_cast<const int4*>(geom4)[i];
    int4 g = make_int4(0, 0, 0, 0);
    if (b.z > 0) {
      g.x = W - b.x;
      g.y = H - b.y;
      g.z = b.z - g.x;
      g.w = b.w - g.y;
    }
    reinterpret_cast<int4*>(geom4)[i] = g;
    return (int64_t)((g.z + 31) >> 5) * g.w;
  }
};

// Pass 2: one CTA per mask; a warp takes a (row, 32-pixel word) item of the window: lane b reads pixel x0 + 32 word + b
// (one coalesced load per item), the ballot is the word.  Lanes beyond the window's width vote 0: padding bits are
// zero.
constexpr int kPackThreads = 256;
template <int DT>
__global__ void __launch_bounds__(kPackThreads) pack_kernel(const void* __restrict__ masks, int H, int W,
                                                            const int32_t* __restrict__ geom4,
                                                            const int64_t* __restrict__ offsets,
                                                            uint32_t* __restrict__ bits, long long capacity_words,
                                                            int32_t* __restrict__ status) {
  const long long i = blockIdx.x;
  const int4 g = reinterpret_cast<const int4*>(geom4)[i];
  if (g.z <= 0 || g.w <= 0) return;
  const int wpr = (g.z + 31) >> 5;
  const long long off = offsets[i];
  if (off + (long long)wpr * g.w > capacity_words) {
    if (threadIdx.x == 0) atomicOr(status, HDY_STATUS_OVERFLOW);
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t base = (size_t)i * H * W;
  for (int item = warp; item < g.w * wpr; item += kPackThreads / 32) {
    const int r = item / wpr, wd = item - r * wpr;
    const int x = (wd << 5) + lane;
    const bool s = x < g.z && elem_set<DT>(masks, base + (size_t)(g.y + r) * W + g.x + x);
    const uint32_t word = __ballot_sync(0xffffffffu, s);
    if (lane == 0) bits[off + (long long)r * wpr + wd] = word;
  }
}

// ---------------------------------------------------------------------------------------------- areas
// One warp per mask.  Bits beyond w in a row's last word are masked off rather than trusted to be zero: PackedMasks
// also arrive from files and from four producers.
constexpr int kAreaThreads = 256;
__global__ void __launch_bounds__(kAreaThreads) areas_kernel(const int32_t* __restrict__ geom4,
                                                             const int64_t* __restrict__ offsets,
                                                             const uint32_t* __restrict__ bits, long long K,
                                                             int32_t* __restrict__ areas) {
  const long long i = ((long long)blockIdx.x * kAreaThreads + threadIdx.x) >> 5;
  if (i >= K) return;  // uniform per warp
  const int lane = threadIdx.x & 31;
  const int4 g = reinterpret_cast<const int4*>(geom4)[i];
  int c = 0;
  if (g.z > 0 && g.w > 0) {
    const int wpr = (g.z + 31) >> 5;
    const uint32_t last = (g.z & 31) ? (1u << (g.z & 31)) - 1u : 0xffffffffu;
    const uint32_t* p = bits + offsets[i];
    const int n = wpr * g.w;  // < 2^31: the window lies in a canvas of fewer than 2^31 pixels
    for (int t = lane; t < n; t += 32) {
      const uint32_t m = t % wpr == wpr - 1 ? last : 0xffffffffu;
      c += __popc(__ldg(p + t) & m);
    }
  }
  c = __reduce_add_sync(0xffffffffu, c);
  if (lane == 0) areas[i] = c;
}

// ---------------------------------------------------------------------------------------------- matching
constexpr int kCandThreads = 256;

// One thread per prediction (rank r in score order), the ground-truth windows and areas staged through shared memory
// in chunks (as match_pairs_kernel does with boxes).  A pair is a candidate when its windows overlap and its IoU upper
// bound reaches iou_min (window_pair_may_match, match_common.cuh): no pair whose exact IoU reaches iou_min is dropped.
__global__ void __launch_bounds__(kCandThreads) candidates_kernel(
    const int32_t* __restrict__ pred_geom, const int32_t* __restrict__ pred_areas,
    const int32_t* __restrict__ pred_order, int P, const int32_t* __restrict__ gt_geom,
    const int32_t* __restrict__ gt_areas, int G, float iou_min, int cand_cap, uint32_t* __restrict__ cand,
    int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  __shared__ int4 gw[kCandThreads];
  __shared__ int ga[kCandThreads];
  const int r = blockIdx.x * kCandThreads + threadIdx.x;
  const bool have = r < P;
  int4 a = make_int4(0, 0, 0, 0);
  int area_a = 0;
  if (have) {
    const int row = pred_order ? pred_order[r] : r;
    a = reinterpret_cast<const int4*>(pred_geom)[row];
    area_a = pred_areas[row];
  }
  const bool live = have && a.z > 0 && a.w > 0;
  for (int j0 = 0; j0 < G; j0 += kCandThreads) {
    __syncthreads();
    if (j0 + threadIdx.x < G) {
      gw[threadIdx.x] = reinterpret_cast<const int4*>(gt_geom)[j0 + threadIdx.x];
      ga[threadIdx.x] = gt_areas[j0 + threadIdx.x];
    }
    __syncthreads();
    if (!live) continue;
    const int lim = min(kCandThreads, G - j0);
    for (int j = 0; j < lim; ++j) {
      if (window_pair_may_match(a, area_a, gw[j], ga[j], iou_min)) {
        const int pos = atomicAdd(&counts[1], 1);
        if (pos < cand_cap)
          cand[pos] = (uint32_t)r * (uint32_t)G + (uint32_t)(j0 + j);
        else
          atomicOr(status, HDY_STATUS_OVERFLOW);
      }
    }
  }
}

constexpr int kExactThreads = 256;
constexpr int kExactMaxBlocks = 4096;

// One warp per candidate (grid-stride over the candidates found, up to cand_cap) counts the intersection
// (warp_window_intersection, match_common.cuh).  Pairs with iou >= iou_min are appended as make_key(iou, rank * G + j).
__global__ void __launch_bounds__(kExactThreads) exact_kernel(
    const int32_t* __restrict__ pred_geom, const int64_t* __restrict__ pred_offsets,
    const uint32_t* __restrict__ pred_bits, const int32_t* __restrict__ pred_areas,
    const int32_t* __restrict__ pred_order, const int32_t* __restrict__ gt_geom,
    const int64_t* __restrict__ gt_offsets, const uint32_t* __restrict__ gt_bits,
    const int32_t* __restrict__ gt_areas, int G, float iou_min, int cand_cap, const uint32_t* __restrict__ cand,
    int cap, uint64_t* __restrict__ pair_keys, int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const long long n = min(counts[1], cand_cap);  // candidates_kernel ran before on the stream
  const long long warps = (long long)gridDim.x * (kExactThreads / 32);
  for (long long c = ((long long)blockIdx.x * kExactThreads + threadIdx.x) >> 5; c < n; c += warps) {
    const uint32_t idx = cand[c];
    const int r = (int)(idx / (uint32_t)G), j = (int)(idx - (uint32_t)r * (uint32_t)G);
    const int row = pred_order ? pred_order[r] : r;
    const int4 a = reinterpret_cast<const int4*>(pred_geom)[row];
    const int4 b = reinterpret_cast<const int4*>(gt_geom)[j];
    const int inter = warp_window_intersection(a, pred_bits + pred_offsets[row], b, gt_bits + gt_offsets[j], lane);
    if (lane == 0) {
      const float iou = mask_iou(inter, pred_areas[row], gt_areas[j]);
      if (iou >= iou_min) {
        const int pos = atomicAdd(&counts[0], 1);
        if (pos < cap)
          pair_keys[pos] = make_key(iou, idx);
        else
          atomicOr(status, HDY_STATUS_OVERFLOW);
      }
    }
  }
}

template <int DT>
static void launch_bounds_pass(const void* masks, int K, int H, int W, int32_t* geom, cudaStream_t st) {
  constexpr int kEsz = DT == HDY_F32 ? 4 : DT == HDY_F16 ? 2 : 1;
  const long long N = (long long)H * W;
  const bool vec = ((uintptr_t)masks & 15) == 0 && (N * kEsz) % 16 == 0;
  long long slices;
  if (vec) {
    const long long per = (long long)kBoundsThreads * kBoundsUnroll * kBoundsIters;
    slices = (N / (16 / kEsz) + per - 1) / per;
    bounds_kernel<DT, true><<<(unsigned)(K * slices), kBoundsThreads, 0, st>>>(masks, H, W, (int)slices, geom);
  } else {
    slices = (N + kBoundsScalarChunk - 1) / kBoundsScalarChunk;
    bounds_kernel<DT, false><<<(unsigned)(K * slices), kBoundsThreads, 0, st>>>(masks, H, W, (int)slices, geom);
  }
}

static int pack_args_ok(const void* masks, int dtype, int K, int H, int W, const int32_t* geom, const char* what) {
  HDY_REQUIRE(K >= 0 && H >= 1 && W >= 1, "%s: bad sizes K=%d H=%d W=%d", what, K, H, W);
  HDY_REQUIRE(dtype == HDY_F32 || dtype == HDY_F16 || dtype == HDY_U8, "%s: dtype must be HDY_F32, HDY_F16 or HDY_U8",
              what);
  HDY_REQUIRE((long long)H * W < (1ll << 31), "%s: H*W must be below 2^31", what);
  if (K > 0) {
    HDY_REQUIRE(masks && geom, "%s: NULL pointer", what);
    HDY_REQUIRE(((uintptr_t)geom & 15) == 0, "%s: geom must be 16-byte aligned", what);
  }
  return HDY_OK;
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_pack_masks_geometry(const void* masks, int dtype, int K, int H, int W, int32_t* geom, int64_t* offsets,
                            hdy_stream_t stream) {
  int rc = pack_args_ok(masks, dtype, K, H, W, geom, "hdy_pack_masks_geometry");
  if (rc) return rc;
  HDY_REQUIRE(offsets != nullptr, "hdy_pack_masks_geometry: offsets is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (K == 0) {
    cudaMemsetAsync(offsets, 0, sizeof(int64_t), st);
    return check_launch("hdy_pack_masks_geometry");
  }
  const long long N = (long long)H * W;
  const long long esz = dtype == HDY_F32 ? 4 : dtype == HDY_F16 ? 2 : 1;
  const long long blocks = (long long)K * ((N + kBoundsScalarChunk - 1) / kBoundsScalarChunk);  // the larger grid
  HDY_REQUIRE(blocks < (1ll << 31), "hdy_pack_masks_geometry: %lld bytes of masks are too many for one call",
              (long long)K * N * esz);
  cudaError_t e = cudaMemsetAsync(geom, 0, (size_t)K * 16, st);
  if (e != cudaSuccess) {
    set_error("cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  if (dtype == HDY_F32)
    launch_bounds_pass<HDY_F32>(masks, K, H, W, geom, st);
  else if (dtype == HDY_F16)
    launch_bounds_pass<HDY_F16>(masks, K, H, W, geom, st);
  else
    launch_bounds_pass<HDY_U8>(masks, K, H, W, geom, st);
  device_exclusive_scan<int64_t, 1>(BoundsWindowWords{geom, H, W}, K, offsets, offsets + K, st);
  return check_launch("hdy_pack_masks_geometry");
}

int hdy_pack_masks(const void* masks, int dtype, int K, int H, int W, const int32_t* geom, const int64_t* offsets,
                   uint32_t* bits, int64_t capacity_words, int32_t* status, hdy_stream_t stream) {
  int rc = pack_args_ok(masks, dtype, K, H, W, geom, "hdy_pack_masks");
  if (rc) return rc;
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(offsets && bits && status && capacity_words >= 0, "hdy_pack_masks: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == HDY_F32)
    pack_kernel<HDY_F32><<<(unsigned)K, kPackThreads, 0, st>>>(masks, H, W, geom, offsets, bits, capacity_words, status);
  else if (dtype == HDY_F16)
    pack_kernel<HDY_F16><<<(unsigned)K, kPackThreads, 0, st>>>(masks, H, W, geom, offsets, bits, capacity_words, status);
  else
    pack_kernel<HDY_U8><<<(unsigned)K, kPackThreads, 0, st>>>(masks, H, W, geom, offsets, bits, capacity_words, status);
  return check_launch("hdy_pack_masks");
}

int hdy_mask_areas(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int32_t* areas,
                   hdy_stream_t stream) {
  HDY_REQUIRE(K >= 0, "hdy_mask_areas: negative K");
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(geom && offsets && bits && areas, "hdy_mask_areas: NULL pointer");
  HDY_REQUIRE(((uintptr_t)geom & 15) == 0, "hdy_mask_areas: geom must be 16-byte aligned");
  const long long blocks = ((long long)K * 32 + kAreaThreads - 1) / kAreaThreads;
  areas_kernel<<<(unsigned)blocks, kAreaThreads, 0, (cudaStream_t)stream>>>(geom, offsets, bits, K, areas);
  return check_launch("hdy_mask_areas");
}

int hdy_match_mask_pairs(const int32_t* pred_geom, const int64_t* pred_offsets, const uint32_t* pred_bits,
                         const int32_t* pred_areas, const int32_t* pred_order, int P, const int32_t* gt_geom,
                         const int64_t* gt_offsets, const uint32_t* gt_bits, const int32_t* gt_areas, int G,
                         float iou_min, int cand_cap, uint32_t* cand, int cap, uint64_t* pair_keys, int32_t* counts,
                         int32_t* status, hdy_stream_t stream) {
  HDY_REQUIRE(P >= 0 && G >= 0 && cand_cap >= 1 && cap >= 1, "match_mask_pairs: P=%d G=%d cand_cap=%d cap=%d", P, G,
              cand_cap, cap);
  HDY_REQUIRE(iou_min > 0.0f, "match_mask_pairs: iou_min must be > 0 (disjoint masks have IoU 0)");
  if (P == 0 || G == 0) return HDY_OK;
  HDY_REQUIRE((long long)P * G < (1ll << 32), "match_mask_pairs: P*G must fit 32 bits (the row-major pair index)");
  HDY_REQUIRE(pred_geom && pred_offsets && pred_bits && pred_areas && gt_geom && gt_offsets && gt_bits && gt_areas &&
                  cand && pair_keys && counts && status,
              "match_mask_pairs: NULL pointer");
  HDY_REQUIRE((((uintptr_t)pred_geom | (uintptr_t)gt_geom) & 15) == 0,
              "match_mask_pairs: geom arrays must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  candidates_kernel<<<(unsigned)((P + kCandThreads - 1) / kCandThreads), kCandThreads, 0, st>>>(
      pred_geom, pred_areas, pred_order, P, gt_geom, gt_areas, G, iou_min, cand_cap, cand, counts, status);
  const long long blocks = min((long long)kExactMaxBlocks, ((long long)cand_cap + 7) / 8);
  exact_kernel<<<(unsigned)blocks, kExactThreads, 0, st>>>(pred_geom, pred_offsets, pred_bits, pred_areas, pred_order,
                                                           gt_geom, gt_offsets, gt_bits, gt_areas, G, iou_min,
                                                           cand_cap, cand, cap, pair_keys, counts, status);
  return check_launch("hdy_match_mask_pairs");
}

}  // extern "C"
