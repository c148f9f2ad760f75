// Per-pair arithmetic of prediction <-> ground-truth matching, shared by the all-pairs matchers (match.cu,
// match_masks.cu) and the binned ones (match_binned.cu): both must give every pair the same IoU bits.
#pragma once
#include "hdy_common.cuh"

namespace hdy {

// box_iou of the reference (utils_general.py:247-265): inter = clamp(min(a2,b2) - max(a1,b1), 0).prod();
// iou = inter / (area1 + area2 - inter), fp32, one rounding per operation; 0/0 = NaN fails `>=`.
__device__ __forceinline__ float ref_box_iou(const float4& a, float area_a, const float4& b, float area_b) {
  const float w = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.0f);
  const float h = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.0f);
  const float inter = __fmul_rn(w, h);
  return __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
}

// iou = float(inter) / float(union), each step rounded to nearest (torch: inter.float() / union.float())
__device__ __forceinline__ float mask_iou(int inter, int area_a, int area_b) {
  const long long uni = (long long)area_a + area_b - inter;
  return __fdiv_rn(__int2float_rn(inter), __ll2float_rn(uni));
}

// The IoU upper bound of two mask windows {x0, y0, w, h}: float(min(overlap area, area_a, area_b)) over the union it
// implies.  The intersection can be at most that, the IoU increases with the intersection, and the round-to-nearest
// conversions and division are monotone, so the fp32 IoU of the pair is <= the bound.  Windows that do not overlap
// return false (their intersection is 0, their IoU 0 or NaN, and iou_min > 0).
__device__ __forceinline__ bool window_pair_may_match(const int4& a, int area_a, const int4& b, int area_b,
                                                      float iou_min) {
  const int ow = min(a.x + a.z, b.x + b.z) - max(a.x, b.x);
  const int oh = min(a.y + a.w, b.y + b.w) - max(a.y, b.y);
  if (ow <= 0 || oh <= 0) return false;
  const int inter_max = (int)min((long long)ow * oh, (long long)min(area_a, area_b));
  return mask_iou(inter_max, area_a, area_b) >= iou_min;
}

// 32 bits of a row of a bit plane starting at bit `dx` (>= 0) of the row; the word after the one holding `dx` is only
// read when the shift needs it and it belongs to the row.
__device__ __forceinline__ uint32_t row_bits(const uint32_t* __restrict__ row, int wpr, int dx) {
  const int k = dx >> 5, s = dx & 31;
  const uint32_t lo = __ldg(row + k);
  const uint32_t hi = (s && k + 1 < wpr) ? __ldg(row + k + 1) : 0u;
  return __funnelshift_r(lo, hi, s);
}

// Exact intersection of two overlapping windows a, b (bit planes at pa, pb), counted by a whole warp; every lane
// returns the sum.  The lanes split the overlap rectangle into (row, 32-pixel chunk) items; both planes are aligned to
// the chunk's first pixel with a funnel shift and the chunk's pixels beyond the overlap are masked off, so padding bits
// never count.
__device__ __forceinline__ int warp_window_intersection(const int4& a, const uint32_t* __restrict__ pa_plane,
                                                        const int4& b, const uint32_t* __restrict__ pb_plane,
                                                        int lane) {
  const int ox0 = max(a.x, b.x), ox1 = min(a.x + a.z, b.x + b.z);
  const int oy0 = max(a.y, b.y), oy1 = min(a.y + a.w, b.y + b.w);
  const int wa = (a.z + 31) >> 5, wb = (b.z + 31) >> 5;
  const uint32_t* pa = pa_plane + (long long)(oy0 - a.y) * wa;
  const uint32_t* pb = pb_plane + (long long)(oy0 - b.y) * wb;
  const int nch = (ox1 - ox0 + 31) >> 5;
  const int items = (oy1 - oy0) * nch;
  int inter = 0;
  for (int t = lane; t < items; t += 32) {
    const int y = t / nch, ch = t - y * nch;
    const int x = ox0 + (ch << 5);
    const int nv = min(32, ox1 - x);
    const uint32_t m = nv == 32 ? 0xffffffffu : (1u << nv) - 1u;
    const uint32_t va = row_bits(pa + (long long)y * wa, wa, x - a.x);
    const uint32_t vb = row_bits(pb + (long long)y * wb, wb, x - b.x);
    inter += __popc(va & vb & m);
  }
  return __reduce_add_sync(0xffffffffu, inter);
}

}  // namespace hdy
