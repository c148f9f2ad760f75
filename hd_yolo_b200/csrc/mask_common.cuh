// Shared device helpers of the mask kernels (mask.cu, mask_regions.cu).
#pragma once
#include "hdy_common.cuh"

namespace hdy {

// ATen's bilinear (align_corners=False): scale = in/out (fp32); src = scale*(dst+0.5)-0.5, clamped at 0;
// i0 = (int)src; i1 = min(i0+1, in-1); l1 = src-i0; l0 = 1-l1; v = l0y*(l0x*v00 + l1x*v01) + l1y*(l0x*v10 + l1x*v11).
struct Lerp {
  int i0, i1;
  float l0, l1;
};

__device__ __forceinline__ Lerp lerp_coord(int dst, float scale, int in_size) {
  float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  if (src < 0.f) src = 0.f;
  Lerp L;
  L.i0 = min((int)src, in_size - 1);
  L.i1 = min(L.i0 + 1, in_size - 1);
  L.l1 = fminf(fmaxf(__fsub_rn(src, (float)L.i0), 0.f), 1.f);
  L.l0 = __fsub_rn(1.0f, L.l1);
  return L;
}

__device__ __forceinline__ float bilerp(float v00, float v01, float v10, float v11, const Lerp& X, const Lerp& Y) {
  const float top = __fadd_rn(__fmul_rn(X.l0, v00), __fmul_rn(X.l1, v01));
  const float bot = __fadd_rn(__fmul_rn(X.l0, v10), __fmul_rn(X.l1, v11));
  return __fadd_rn(__fmul_rn(Y.l0, top), __fmul_rn(Y.l1, bot));
}

// ------------------------------------------------------------------------------------- (B) process_mask
__device__ __forceinline__ int ceil_to_int_clamped(float v, int lo, int hi) {
  if (!(v > (float)lo)) return lo;  // also NaN
  if (v >= (float)hi) return hi;
  return (int)ceilf(v);
}

// The proto pixels crop_mask keeps: x1d <= col < x2d, y1d <= row < y2d (float compares against arange).
struct KeptRange {
  float x1d, y1d, x2d, y2d;  // down-scaled box (fp32, as the reference computes it)
  int px0, py0, px1, py1;    // kept proto pixel range [p0, p1)
};
__device__ __forceinline__ KeptRange kept_range(const float4 b, float rx, float ry, int mw, int mh) {
  KeptRange k;
  k.x1d = __fmul_rn(b.x, rx);  // downsampled_bboxes[:, 0] *= mw / iw ...
  k.x2d = __fmul_rn(b.z, rx);
  k.y1d = __fmul_rn(b.y, ry);
  k.y2d = __fmul_rn(b.w, ry);
  // r >= x1 & r < x2 over integers r: [ceil(x1), ceil(x2))
  k.px0 = ceil_to_int_clamped(k.x1d, 0, mw);
  k.px1 = ceil_to_int_clamped(k.x2d, 0, mw);
  k.py0 = ceil_to_int_clamped(k.y1d, 0, mh);
  k.py1 = ceil_to_int_clamped(k.y2d, 0, mh);
  // a NaN coordinate fails every crop comparison of the reference: nothing is kept.  For finite coordinates the crop
  // test x1d <= col < x2d over integer columns IS col in [px0, px1), so the two-phase kernels walk the integer range
  // and never compare against the floats again.
  if (!(k.x1d == k.x1d) || !(k.x2d == k.x2d) || !(k.y1d == k.y1d) || !(k.y2d == k.y2d)) k.px1 = k.px0, k.py1 = k.py0;
  return k;
}

// Window of mask i in output pixels.  With upsample the bilinear taps spread every kept pixel over its neighbours, so
// the output window is the pre-image of [p0-1, p1) under i0 = floor(src).
struct PMGeom : KeptRange {
  int x0, y0, w, h;  // output window
};

// Source coordinate of output pixel `dst` exactly as lerp_coord (ATen) computes it.
__device__ __forceinline__ float pm_src(int dst, float scale) {
  const float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  return src < 0.f ? 0.f : src;
}

// Shrinks the window [o0, o1) of one axis to the output pixels whose value can exceed 0.5.  Proto pixels outside
// [p0, p1) are cropped to zero and the kept ones are at most 1, so an output pixel left of the kept range is worth at
// most its weight on pixel p0: with i0 = p0 - 1 that weight is l1 = src - i0, i.e. the pixel is dead while
// src <= p0 - 0.5 (and it is exactly zero while i1 < p0).  Symmetrically on the right, where pixel p1 exists (p1 < in):
// dead once src >= p1 - 0.5 (l0 = 1 - l1 <= 0.5).  Rounding cannot lift such a value over 0.5: every product and sum
// in bilerp is monotone in its operands and 0.5 * (l0 + l1) rounds to 0.5.  src is monotone in the pixel index, so
// both ends are found from an estimate and a short walk.  At 4x a nucleus' window shrinks by 6 pixels per axis
// (36 -> 30: one 32-bit word per row instead of two).
__device__ __forceinline__ void pm_trim(int& o0, int& o1, int p0, int p1, int in_size, float scale) {
  if (o1 <= o0) return;
  if (p0 > 0) {
    const float tl = (float)p0 - 0.5f;
    int c = (int)floorf((float)p0 / scale - 0.5f) - 1;
    c = min(max(c, o0), o1);
    while (c < o1 && !(pm_src(c, scale) > tl)) ++c;
    while (c > o0 && pm_src(c - 1, scale) > tl) --c;
    o0 = c;
  }
  if (p1 < in_size && o1 > o0) {
    const float tr = (float)p1 - 0.5f;
    int c = (int)floorf((float)p1 / scale - 0.5f) - 1;
    c = min(max(c, o0), o1);
    while (c < o1 && !(pm_src(c, scale) >= tr)) ++c;
    while (c > o0 && pm_src(c - 1, scale) >= tr) --c;
    o1 = c;
  }
}

__device__ __forceinline__ PMGeom pm_geometry(const float4 b, int mh, int mw, int ih, int iw, int upsample,
                                              float rx, float ry) {
  PMGeom g;
  static_cast<KeptRange&>(g) = kept_range(b, rx, ry, mw, mh);
  if (g.px1 <= g.px0 || g.py1 <= g.py0) {
    g.x0 = g.y0 = g.w = g.h = 0;
    return g;
  }
  if (!upsample) {
    g.x0 = g.px0;
    g.y0 = g.py0;
    g.w = g.px1 - g.px0;
    g.h = g.py1 - g.py0;
  } else {
    // conservative superset: src = s*(dst+0.5)-0.5 with s = mw/iw; i0 in [p0-1, p1-1]  <=>  src in [p0-1, p1)
    const float sx = (float)mw / (float)iw, sy = (float)mh / (float)ih;
    int ox0 = (int)floorf(((float)g.px0 - 0.5f) / sx - 0.5f) - 1, ox1 = (int)ceilf(((float)g.px1 + 0.5f) / sx - 0.5f) + 1;
    int oy0 = (int)floorf(((float)g.py0 - 0.5f) / sy - 0.5f) - 1, oy1 = (int)ceilf(((float)g.py1 + 0.5f) / sy - 0.5f) + 1;
    ox0 = max(ox0, 0);
    oy0 = max(oy0, 0);
    ox1 = min(ox1, iw);
    oy1 = min(oy1, ih);
    // ... trimmed to the pixels that CAN exceed 0.5 (exact, see pm_trim)
    pm_trim(ox0, ox1, g.px0, g.px1, mw, sx);
    pm_trim(oy0, oy1, g.py0, g.py1, mh, sy);
    g.x0 = ox0;
    g.y0 = oy0;
    g.w = max(ox1 - ox0, 0);
    g.h = max(oy1 - oy0, 0);
    if (g.w == 0 || g.h == 0) g.x0 = g.y0 = g.w = g.h = 0;
  }
  return g;
}


// smallest dst in [lo, hi) whose first tap lerp_coord(dst).i0 is >= target (hi if there is none)
__device__ __forceinline__ int first_dst_i0_ge(int target, int lo, int hi, float scale, int in_size) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (lerp_coord(mid, scale, in_size).i0 >= target)
      hi = mid;
    else
      lo = mid + 1;
  }
  return lo;
}

constexpr int kPmTile = 32;               // proto pixels per staged tile side
constexpr int kPmStage = kPmTile + 1;     // + 1 halo for the second bilinear tap

// One CTA per detection slot.  For every kPmTile^2 block of proto pixels touching the mask's window the
// cropped sigmoid(coef . proto) values are staged in shared memory (32 FFMA per pixel, channel-strided
// coalesced reads that hit L2 after the first detection of a tile), then the output pixels whose first tap
// falls into the block are emitted.
// `stage` [kPmStage^2] and `cf` [64] floats of shared memory are the caller's (static in process_mask_kernel, a corner of
// the region buffer when the listed detections ride in proto_patch_kernel's launch); every thread of the CTA calls it.
// Items item_first, item_first + item_step, ... < n_items; of each item the proto tiles tile_first, + tile_step, ...
template <bool PACKED, bool HALF>
__device__ __forceinline__ void process_mask_body(
    const void* __restrict__ protos, const float* __restrict__ coef, const float4* __restrict__ boxes,
    const int32_t* __restrict__ counts, int max_det, int nm, int mh, int mw, int ih, int iw, int upsample,
    float rx, float ry, float* __restrict__ out_dense, const int32_t* __restrict__ geom4,
    const int64_t* __restrict__ offsets,
    uint32_t* __restrict__ bits, long long capacity_words, int32_t* __restrict__ status,
    const int32_t* __restrict__ slot_list, long long n_items, long long item_first, long long item_step,
    int tile_first, int tile_step, float* __restrict__ stage, float* __restrict__ cf) {
  const int nthreads = blockDim.x;
  for (long long item = item_first; item < n_items; item += item_step) {
  const long long slot = slot_list ? (long long)slot_list[item] : item;
  const int tile = (int)(slot / max_det), d = (int)(slot - (long long)tile * max_det);
  __syncthreads();  // cf / stage of the previous item are free
  if (d >= counts[tile]) continue;
  if (geom4 && (geom4[4 * slot + 2] <= 0 || geom4[4 * slot + 3] <= 0)) continue;  // empty, or not KEPT (slide form)
  const PMGeom g = pm_geometry(boxes[slot], mh, mw, ih, iw, upsample, rx, ry);
  if (g.w <= 0 || g.h <= 0) continue;
  const int oh = upsample ? ih : mh, ow = upsample ? iw : mw;
  const int wpr = (g.w + 31) >> 5;
  long long off = 0;
  if (PACKED) {
    off = offsets[slot];
    if (off + (long long)wpr * g.h > capacity_words) {
      if (threadIdx.x == 0) atomicOr(status, HDY_STATUS_OVERFLOW);
      continue;
    }
  }
  for (int c = threadIdx.x; c < nm; c += nthreads) cf[c] = coef[slot * nm + c];
  const size_t P0 = (size_t)tile * nm * mh * mw;  // first element of the tile's prototypes
  const size_t plane = (size_t)mh * mw;
  const float sxs = (float)mw / (float)iw, sys = (float)mh / (float)ih;  // ATen: scale = in / out (fp32)
  // proto range that can contribute: the kept pixels, plus one pixel before (their second-tap neighbours)
  const int ty_begin = upsample ? max(g.py0 - 1, 0) : g.py0, tx_begin = upsample ? max(g.px0 - 1, 0) : g.px0;
  const int nty = (g.py1 - ty_begin + kPmTile - 1) / kPmTile, ntx = (g.px1 - tx_begin + kPmTile - 1) / kPmTile;
  for (int tt = tile_first; tt < nty * ntx; tt += tile_step) {
    {
      const int ty = ty_begin + (tt / ntx) * kPmTile, tx = tx_begin + (tt % ntx) * kPmTile;
      __syncthreads();
      // ---- stage cropped sigmoid values for proto pixels [ty, ty+33) x [tx, tx+33)
      for (int e = threadIdx.x; e < kPmStage * kPmStage; e += nthreads) {
        const int yy = ty + e / kPmStage, xx = tx + e % kPmStage;
        float v = 0.f;
        if (yy < mh && xx < mw && (float)xx >= g.x1d && (float)xx < g.x2d && (float)yy >= g.y1d &&
            (float)yy < g.y2d) {
          const size_t p = P0 + (size_t)yy * mw + xx;
          // (the listed form runs a handful of CTAs: its duration is this latency chain, so all the channel loads of a
          // pixel are issued before the first FMA -- with 8 in flight the kernel took 4 DRAM round trips per pixel)
          float acc = 0.f;
          int c = 0;
          for (; c + 32 <= nm; c += 32) {
            float pv[32];
#pragma unroll
            for (int j = 0; j < 32; ++j)
              pv[j] = HALF ? __half2float(__ldg(static_cast<const __half*>(protos) + p + (c + j) * plane))
                           : __ldg(static_cast<const float*>(protos) + p + (c + j) * plane);
#pragma unroll
            for (int j = 0; j < 32; ++j) acc = fmaf(cf[c + j], pv[j], acc);
          }
          for (; c < nm; ++c) {
            const float pv = HALF ? __half2float(__ldg(static_cast<const __half*>(protos) + p + c * plane))
                                  : __ldg(static_cast<const float*>(protos) + p + c * plane);
            acc = fmaf(cf[c], pv, acc);
          }
          v = sigmoidf_ref(acc);
        }
        stage[e] = v;
      }
      __syncthreads();
      if (!upsample) {
        // output pixel == proto pixel
        const int y_lo = max(ty, g.y0), y_hi = min(ty + kPmTile, g.y0 + g.h);
        const int x_lo = max(tx, g.x0), x_hi = min(tx + kPmTile, g.x0 + g.w);
        const int tw = x_hi - x_lo, th = y_hi - y_lo;
        for (int e = threadIdx.x; e < tw * th; e += nthreads) {
          const int yy = y_lo + e / tw, xx = x_lo + e % tw;
          const bool bit = stage[(yy - ty) * kPmStage + (xx - tx)] > 0.5f;
          if (PACKED) {
            if (bit) atomicOr(&bits[off + (long long)(yy - g.y0) * wpr + ((xx - g.x0) >> 5)], 1u << ((xx - g.x0) & 31));
          } else {
            out_dense[(size_t)slot * oh * ow + (size_t)yy * ow + xx] = bit ? 1.f : 0.f;
          }
        }
      } else {
        // output pixels of the window whose first taps (i0) fall into [ty, ty+32) x [tx, tx+32): i0 is monotone in the
        // output coordinate, so they form a rectangle whose edges are found by bisection (scanning the whole window
        // for every tile made a large box quadratic in its tile count)
        const int oy_lo = first_dst_i0_ge(ty, g.y0, g.y0 + g.h, sys, mh);
        const int oy_hi = first_dst_i0_ge(ty + kPmTile, oy_lo, g.y0 + g.h, sys, mh);
        const int ox_lo = first_dst_i0_ge(tx, g.x0, g.x0 + g.w, sxs, mw);
        const int ox_hi = first_dst_i0_ge(tx + kPmTile, ox_lo, g.x0 + g.w, sxs, mw);
        const int tw = ox_hi - ox_lo, th = oy_hi - oy_lo;
        for (int e = threadIdx.x; e < tw * th; e += nthreads) {
          const int oy = oy_lo + e / tw, ox = ox_lo + e % tw;
          const Lerp Y = lerp_coord(oy, sys, mh), X = lerp_coord(ox, sxs, mw);
          const int sy0 = Y.i0 - ty, sx0 = X.i0 - tx, sy1 = Y.i1 - ty, sx1 = X.i1 - tx;
          const float v = bilerp(stage[sy0 * kPmStage + sx0], stage[sy0 * kPmStage + sx1],
                                 stage[sy1 * kPmStage + sx0], stage[sy1 * kPmStage + sx1], X, Y);
          const bool bit = v > 0.5f;
          if (PACKED) {
            if (bit) atomicOr(&bits[off + (long long)(oy - g.y0) * wpr + ((ox - g.x0) >> 5)], 1u << ((ox - g.x0) & 31));
          } else {
            out_dense[(size_t)slot * oh * ow + (size_t)oy * ow + ox] = bit ? 1.f : 0.f;
          }
        }
      }
    }
  }
  }
}


// mask_regions.cu: two-phase process_mask (TMA-staged prototypes -> sigmoid patches -> upsample + pack).  Returns 1
// when the shapes / workspace / windows do not meet its requirements (the caller then uses the per-detection kernel in
// mask.cu).
constexpr int kPatchPitch = 16;  // sigmoid patches of up to 16 x 16 proto pixels go through the workspace
size_t process_mask_workspace_bytes(long long bs, long long max_det);
int launch_process_mask_regions(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                                const int32_t* counts, int bs, int max_det, int nm, int mh, int mw, int ih, int iw, int upsample, float rx,
                                float ry, float* out_dense, const int32_t* geom, const int64_t* offsets, uint32_t* bits,
                                long long capacity_words, int32_t* status, void* workspace, size_t workspace_bytes,
                                cudaStream_t stream);

}  // namespace hdy
