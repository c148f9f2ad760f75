// Mask post-processing.
//
// (A) reference parity  -- M1: sigmoid + per-label channel gather (yolo_head.py:332, 346-353)
//                          M2: torchvision paste_masks_in_image(masks, boxes, (H,W), padding=1) as called at
//                              val_nuclei.py:169-176 / evaluation.py:122-123
//                          M3: > 0.5 (the reference only thresholds for display, image_utils.py:331-340)
// (B) north-star        -- process_mask (ultralytics/yolov5 v7 utils/segment/general.py): K=32 prototype x
//                          coefficient contraction in fp32 FFMA, sigmoid, box crop, optional bilinear upsample,
//                          > 0.5.
//
// Output layouts:
//   dense   : exactly the reference tensors ([K,H,W] fp32), for drop-in parity; the canvas is cleared with
//             one memset and only the paste window is computed.
//   packed  : box-cropped bit planes.  geom[i] = {x0, y0, w, h} (window in output pixels), offsets[i] = first
//             32-bit word of mask i; row r of mask i occupies ceil(w/32) words, bit (x - x0) & 31 of word
//             (x - x0) >> 5, set iff value > 0.5.  This is the layout the throughput numbers use: a nucleus
//             costs ~100-300 bytes instead of H*W*4.
//
// ATen's bilinear (align_corners=False): scale = in/out (fp32); src = scale*(dst+0.5)-0.5, clamped at 0;
// i0 = (int)src; i1 = min(i0+1, in-1); l1 = src-i0; l0 = 1-l1; v = l0y*(l0x*v00 + l1x*v01) + l1y*(l0x*v10 + l1x*v11).
#include <stdlib.h>
#include "mask_common.cuh"
#include "scan_common.cuh"

namespace hdy {

// ---------------------------------------------------------------------------------------------- M1
__global__ void mask_select_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                   const int64_t* __restrict__ mask_indices, int K, int C, int MM,
                                   float* __restrict__ out) {
  const int i = blockIdx.x;
  if (i >= K) return;
  // mask_labels = mask_indices[labels.clamp(min=0)]; masks[mask_labels < 0] = 0       yolo_head.py:348-353
  const int64_t lab = labels[i] < 0 ? 0 : labels[i];
  const int64_t ch = mask_indices[lab];
  const float* src = logits + ((size_t)i * C + (ch < 0 ? 0 : ch)) * MM;
  float* dst = out + (size_t)i * MM;
  for (int e = threadIdx.x; e < MM; e += blockDim.x) dst[e] = ch < 0 ? 0.f : sigmoidf_ref(src[e]);
}

// ------------------------------------------------------------------------------------------ M2 geometry
struct PasteGeom {
  int bx0, by0;  // expanded integer box origin (may be negative)
  int rw, rh;    // resize target (>= 1)
  int x0, y0;    // paste window origin inside the image
  int w, h;      // paste window size (0 if nothing lands in the image)
};

__device__ __forceinline__ PasteGeom paste_geometry(const float4 b, float scale, int H, int W) {
  // expand_boxes (torchvision roi_heads.py): half extents scaled about the centre, then .to(int64) (truncation)
  float w_half = __fmul_rn(__fmul_rn(__fsub_rn(b.z, b.x), 0.5f), scale);
  float h_half = __fmul_rn(__fmul_rn(__fsub_rn(b.w, b.y), 0.5f), scale);
  const float xc = __fmul_rn(__fadd_rn(b.z, b.x), 0.5f), yc = __fmul_rn(__fadd_rn(b.w, b.y), 0.5f);
  const long long x0 = (long long)__fsub_rn(xc, w_half), x1 = (long long)__fadd_rn(xc, w_half);
  const long long y0 = (long long)__fsub_rn(yc, h_half), y1 = (long long)__fadd_rn(yc, h_half);
  PasteGeom g;
  long long rw = x1 - x0 + 1, rh = y1 - y0 + 1;  // TO_REMOVE = 1
  rw = rw < 1 ? 1 : rw;
  rh = rh < 1 ? 1 : rh;
  const long long px0 = x0 > 0 ? x0 : 0, px1 = (x1 + 1 < W) ? x1 + 1 : W;
  const long long py0 = y0 > 0 ? y0 : 0, py1 = (y1 + 1 < H) ? y1 + 1 : H;
  const long long big = 1ll << 30;
  g.bx0 = (int)max(-big, min(big, x0));
  g.by0 = (int)max(-big, min(big, y0));
  g.rw = (int)min(big, rw);
  g.rh = (int)min(big, rh);
  if (px1 > px0 && py1 > py0 && x0 > -big && y0 > -big) {
    g.x0 = (int)px0;
    g.y0 = (int)py0;
    g.w = (int)(px1 - px0);
    g.h = (int)(py1 - py0);
  } else {
    g.x0 = g.y0 = g.w = g.h = 0;
  }
  return g;
}

// offsets[0..K] of the packed layout: an exclusive scan of the words of every mask's cropped bit plane (words(i)),
// offsets[K] = the total.  One launch up to 1 024 masks, three beyond (device_exclusive_scan, no scratch).
template <class Words>
static void scan_words(Words words, long long K, int64_t* offsets, cudaStream_t st) {
  if (K <= 0)
    cudaMemsetAsync(offsets, 0, sizeof(int64_t), st);
  else
    device_exclusive_scan<int64_t, 1>(words, K, offsets, offsets + K, st);
}

struct GeomWords {
  const int32_t* geom4;
  __device__ int64_t operator()(long long i) const {
    return (int64_t)((__ldg(geom4 + 4 * i + 2) + 31) >> 5) * __ldg(geom4 + 4 * i + 3);
  }
};

__global__ void paste_geometry_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ channel, int K,
                                      float scale, int H, int W, int32_t* __restrict__ geom4) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K) return;
  int4 out = make_int4(0, 0, 0, 0);
  if (!channel || channel[i] >= 0) {  // channel < 0: empty mask (no words)
    const PasteGeom g = paste_geometry(boxes[i], scale, H, W);
    out = make_int4(g.x0, g.y0, g.w, g.h);
  }
  reinterpret_cast<int4*>(geom4)[i] = out;
}

// One CTA (4 warps) per mask.  The (M+2p)^2 zero-padded mask is staged in shared memory (sigmoid applied on the way
// if the source holds logits).  The paste window is cut into items of (32-pixel word, quarter of the rows); a warp
// takes an item, interpolates its lanes' columns along x for the source rows the item touches (ATen's `top`/`bot`
// terms, once per source row instead of once per pixel), then every output row is one 2-tap blend from that column
// buffer, a compare and a ballot.  Narrow tail words (4 columns of a 36-px window) are processed several rows at a
// time.  Every word of the mask is stored exactly once.
constexpr int kPasteThreads = 128;
constexpr int kPasteWarps = kPasteThreads / 32;
constexpr int kPasteRows = 64;  // output rows per pass
struct PasteRow {
  int i0, i1;
  float l0, l1;
};
static inline size_t paste_smem_bytes(int Mp) {
  return (size_t)Mp * Mp * 4 + kPasteRows * sizeof(PasteRow) + (size_t)kPasteWarps * Mp * 32 * 4;
}

template <bool PACKED>
__global__ void __launch_bounds__(kPasteThreads) paste_masks_kernel(
    const float* __restrict__ src, const int32_t* __restrict__ channel, const float4* __restrict__ boxes, int K,
    int C, int M, int pad, int apply_sigmoid, int H, int W, float scale, float* __restrict__ out_dense,
    const int64_t* __restrict__ offsets, uint32_t* __restrict__ bits, long long capacity_words,
    int32_t* __restrict__ status) {
  extern __shared__ __align__(16) float sm[];
  const int i = blockIdx.x;
  const int Mp = M + 2 * pad;
  const int ch = channel ? channel[i] : 0;
  if (ch < 0) return;  // empty mask: no words in the packed layout, the dense canvas is already zero
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* P = sm;                                                   // [Mp][Mp]
  PasteRow* rowtab = reinterpret_cast<PasteRow*>(sm + Mp * Mp);    // [kPasteRows]  (Mp*Mp*4 is a multiple of 16)
  float* col = reinterpret_cast<float*>(rowtab + kPasteRows) + (size_t)warp * Mp * 32;  // [Mp][32] per warp
  {
    // stage the padded mask: zero everything, then the M x M interior with 8 independent (coalesced) loads in flight
    // per thread before the first sigmoid needs its operand
    for (int e = threadIdx.x; e < Mp * Mp; e += kPasteThreads) P[e] = 0.f;
    __syncthreads();
    const float* m = src + ((size_t)i * C + ch) * M * M;
    const int MM = M * M;
    for (int e0 = 0; e0 < MM; e0 += kPasteThreads * 8) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int e = e0 + k * kPasteThreads + (int)threadIdx.x;
        v[k] = e < MM ? m[e] : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int e = e0 + k * kPasteThreads + (int)threadIdx.x;
        if (e < MM) {
          const int y = e / M, x = e - y * M;
          P[(y + pad) * Mp + x + pad] = apply_sigmoid ? sigmoidf_ref(v[k]) : v[k];
        }
      }
    }
  }
  const PasteGeom g = paste_geometry(boxes[i], scale, H, W);
  if (g.w <= 0 || g.h <= 0) return;  // uniform
  const int wpr = (g.w + 31) >> 5;
  long long off = 0;
  if (PACKED) {
    off = offsets[i];
    if (off + (long long)wpr * g.h > capacity_words) {
      if (threadIdx.x == 0) atomicOr(status, HDY_STATUS_OVERFLOW);
      return;
    }
  }
  const float sx = __fdiv_rn((float)Mp, (float)g.rw), sy = __fdiv_rn((float)Mp, (float)g.rh);
  for (int r0 = 0; r0 < g.h; r0 += kPasteRows) {
    const int nr = min(kPasteRows, g.h - r0);
    __syncthreads();  // P is complete / the previous pass is done with rowtab
    if ((int)threadIdx.x < nr) {
      const Lerp Y = lerp_coord(g.y0 + r0 + (int)threadIdx.x - g.by0, sy, Mp);
      PasteRow T;
      T.i0 = Y.i0;
      T.i1 = Y.i1;
      T.l0 = Y.l0;
      T.l1 = Y.l1;
      rowtab[threadIdx.x] = T;
    }
    __syncthreads();
    const int quarter = (nr + kPasteWarps - 1) / kPasteWarps;
    for (int item = warp; item < wpr * kPasteWarps; item += kPasteWarps) {
      // items of one word go to the four warps: (word, q) -> warp q handles rows [q*quarter, (q+1)*quarter)
      const int w = item / kPasteWarps;
      const int ra = min(warp * quarter, nr), rb = min(ra + quarter, nr);
      if (rb <= ra) continue;
      const int s_lo = rowtab[ra].i0, s_hi = rowtab[rb - 1].i1;  // source rows touched (lerp is monotone)
      const int vw = min(32, g.w - (w << 5));
      __syncwarp();
      if (vw <= 16) {
        const int rows_per = 32 / vw;
        const int lr = lane / vw, lc = lane - lr * vw;
        const bool active = lr < rows_per;
        const Lerp X = lerp_coord(g.x0 + (w << 5) + lc - g.bx0, sx, Mp);
        if (active)
          for (int s_ = s_lo + lr; s_ <= s_hi; s_ += rows_per)
            col[s_ * 32 + lc] = __fadd_rn(__fmul_rn(X.l0, P[s_ * Mp + X.i0]), __fmul_rn(X.l1, P[s_ * Mp + X.i1]));
        __syncwarp();
        const unsigned row_mask = (1u << vw) - 1u;
        for (int rbase = ra; rbase < rb; rbase += rows_per) {
          const int r = rbase + lr;
          bool bit = false;
          if (active && r < rb) {
            const float4 rt = *reinterpret_cast<const float4*>(&rowtab[r]);
            const float v = __fadd_rn(__fmul_rn(rt.z, col[__float_as_int(rt.x) * 32 + lc]),
                                      __fmul_rn(rt.w, col[__float_as_int(rt.y) * 32 + lc]));
            bit = v > 0.5f;
            if (!PACKED) out_dense[(size_t)i * H * W + (size_t)(g.y0 + r0 + r) * W + g.x0 + (w << 5) + lc] = v;
          }
          if (PACKED) {
            const unsigned mm = __ballot_sync(0xffffffffu, bit);
            if (active && lc == 0 && r < rb) bits[off + (long long)(r0 + r) * wpr + w] = (mm >> (lr * vw)) & row_mask;
          }
        }
        continue;
      }
      const int c = (w << 5) + lane;
      const bool valid = c < g.w;
      const Lerp X = lerp_coord(g.x0 + (valid ? c : 0) - g.bx0, sx, Mp);
      for (int s_ = s_lo; s_ <= s_hi; ++s_)
        col[s_ * 32 + lane] = __fadd_rn(__fmul_rn(X.l0, P[s_ * Mp + X.i0]), __fmul_rn(X.l1, P[s_ * Mp + X.i1]));
      __syncwarp();
      unsigned myword = 0;
      for (int r = ra; r < rb; ++r) {  // rb - ra <= 16
        const float4 rt = *reinterpret_cast<const float4*>(&rowtab[r]);
        const float v = __fadd_rn(__fmul_rn(rt.z, col[__float_as_int(rt.x) * 32 + lane]),
                                  __fmul_rn(rt.w, col[__float_as_int(rt.y) * 32 + lane]));
        if (PACKED) {
          const unsigned word = __ballot_sync(0xffffffffu, valid && v > 0.5f);
          if (r - ra == lane) myword = word;
        } else if (valid) {
          out_dense[(size_t)i * H * W + (size_t)(g.y0 + r0 + r) * W + g.x0 + c] = v;
        }
      }
      if (PACKED && lane < rb - ra) bits[off + (long long)(r0 + ra + lane) * wpr + w] = myword;
    }
  }
}

__global__ void unpack_masks_kernel(const int32_t* __restrict__ geom4, const int64_t* __restrict__ offsets,
                                    const uint32_t* __restrict__ bits, int H, int W, uint8_t* __restrict__ out) {
  const int i = blockIdx.x;
  const int4 g = reinterpret_cast<const int4*>(geom4)[i];
  const int wpr = (g.z + 31) >> 5;
  const long long off = offsets[i];
  uint8_t* o = out + (size_t)i * H * W;
  for (int e = threadIdx.x; e < g.z * g.w; e += blockDim.x) {
    const int yy = e / g.z, xx = e - yy * g.z;
    const uint32_t wd = bits[off + (long long)yy * wpr + (xx >> 5)];
    if (g.y + yy < H && g.x + xx < W && g.y + yy >= 0 && g.x + xx >= 0)   // windows are inside the canvas by
      o[(size_t)(g.y + yy) * W + g.x + xx] = (wd >> (xx & 31)) & 1u;      // construction; never write beyond it
  }
}

// words(i) of hdy_process_mask_geometry: the window of slot i, stored to geom4 on the way, so that the geometry and the
// first pass of the scan are one launch (the step is a chain of small dependent kernels)
struct PmWindowWords {
  const float4* boxes;
  const int32_t* counts;
  int max_det, mh, mw, ih, iw, upsample;
  float rx, ry;
  const uint8_t* row_state;
  const int64_t* tile_offsets;
  int32_t* geom4;
  __device__ int64_t operator()(long long i) const {
    const int tile = (int)(i / max_det), d = (int)(i - (long long)tile * max_det);
    int4 out = make_int4(0, 0, 0, 0);
    // row_state: the slot is row tile_offsets[tile] + d of the slide; only rows the slide-level merge KEPT get a mask
    if (d < __ldg(counts + tile) &&
        (!row_state || __ldg(row_state + __ldg(tile_offsets + tile) + d) == HDY_STATE_KEPT)) {
      const PMGeom g = pm_geometry(__ldg(boxes + i), mh, mw, ih, iw, upsample, rx, ry);
      out = make_int4(g.x0, g.y0, g.w, g.h);
    }
    reinterpret_cast<int4*>(geom4)[i] = out;
    return (int64_t)((out.z + 31) >> 5) * out.w;
  }
};

// Slide form of the packed layout: the batch's word offsets move behind the words of the earlier batches (device
// cursor, ping-pong so that one launch both reads and advances it) and every live slot's window / offset is copied to
// its slide row, the window shifted to slide pixels (x0 + roi.x0: bit positions inside the words do not change).
__global__ void pm_rows_kernel(int32_t* __restrict__ geom4, int64_t* __restrict__ offsets,
                               const int32_t* __restrict__ counts, const int64_t* __restrict__ tile_offsets,
                               const float4* __restrict__ rois, long long K, int max_det,
                               int64_t* __restrict__ cursor2, int parity, int32_t* __restrict__ geom_rows,
                               int64_t* __restrict__ off_rows) {
  const long long base = cursor2[parity & 1];
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > K) return;
  const long long o = offsets[i] + base;
  offsets[i] = o;
  if (i == K) {
    cursor2[(parity + 1) & 1] = o;
    return;
  }
  const int tile = (int)(i / max_det), d = (int)(i - (long long)tile * max_det);
  if (d >= counts[tile]) return;
  const long long row = tile_offsets[tile] + d;
  int4 g = reinterpret_cast<const int4*>(geom4)[i];
  if (g.z > 0 && g.w > 0) {
    const float4 r = rois[tile];
    g.x += (int)r.x;
    g.y += (int)r.y;
  }
  reinterpret_cast<int4*>(geom_rows)[row] = g;
  off_rows[row] = o;
}

constexpr int kPmThreads = 128;

// One CTA per detection slot, all of its proto tiles: the path of the shapes, workspaces and (packed) missing windows
// that mask_regions.cu does not take
template <bool PACKED, bool HALF>
__global__ void __launch_bounds__(kPmThreads) process_mask_kernel(
    const void* __restrict__ protos, const float* __restrict__ coef, const float4* __restrict__ boxes,
    const int32_t* __restrict__ counts, int max_det, int nm, int mh, int mw, int ih, int iw, int upsample,
    float rx, float ry, float* __restrict__ out_dense, const int32_t* __restrict__ geom4,
    const int64_t* __restrict__ offsets,
    uint32_t* __restrict__ bits, long long capacity_words, int32_t* __restrict__ status) {
  __shared__ float stage[kPmStage * kPmStage];
  __shared__ float cf[64];
  process_mask_body<PACKED, HALF>(protos, coef, boxes, counts, max_det, nm, mh, mw, ih, iw, upsample, rx, ry, out_dense,
                                  geom4, offsets, bits, capacity_words, status, nullptr, gridDim.x, blockIdx.x,
                                  gridDim.x, 0, 1, stage, cf);
}

template <bool PACKED>
static int launch_process_mask_kernel(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                                      const int32_t* counts, int bs, int max_det, int nm, int mh, int mw, int ih,
                                      int iw, int upsample, float rx, float ry, float* out_dense,
                                      const int32_t* geom, const int64_t* offsets, uint32_t* bits,
                                      long long capacity_words, int32_t* status, cudaStream_t st, const char* what) {
  const auto kernel = proto_dtype == HDY_F16 ? process_mask_kernel<PACKED, true> : process_mask_kernel<PACKED, false>;
  kernel<<<(unsigned)((size_t)bs * max_det), kPmThreads, 0, st>>>(protos, coef, reinterpret_cast<const float4*>(boxes),
                                                                   counts, max_det, nm, mh, mw, ih, iw, upsample, rx,
                                                                   ry, out_dense, geom, offsets, bits, capacity_words,
                                                                   status);
  return check_launch(what);
}

static int paste_args_ok(const float* src, const float* boxes, int K, int C, int M, int pad, int H, int W) {
  HDY_REQUIRE(K >= 0 && C >= 1 && M >= 1 && pad >= 0 && H >= 1 && W >= 1, "paste: bad sizes");
  HDY_REQUIRE(paste_smem_bytes(M + 2 * pad) <= 200 * 1024, "paste: mask too large for shared memory");
  if (K > 0) HDY_REQUIRE(src && boxes && ((uintptr_t)boxes & 15) == 0, "paste: NULL or misaligned pointer");
  return HDY_OK;
}

template <bool PACKED>
static int launch_paste(const float* src, const int32_t* channel, const float* boxes, int K, int C, int M, int pad,
                        int apply_sigmoid, int H, int W, float* out, const int64_t* offsets, uint32_t* bits,
                        long long cap, int32_t* status, cudaStream_t st) {
  const int Mp = M + 2 * pad;
  const size_t smem = paste_smem_bytes(Mp);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(paste_masks_kernel<PACKED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return HDY_ERR_CUDA;
    }
  }
  const float scale = (float)((double)(M + 2 * pad) / (double)M);  // expand_masks: float(M + 2p) / M
  paste_masks_kernel<PACKED><<<(unsigned)K, kPasteThreads, smem, st>>>(src, channel,
                                                                       reinterpret_cast<const float4*>(boxes), K, C, M,
                                                                       pad, apply_sigmoid, H, W, scale, out, offsets,
                                                                       bits, cap, status);
  return check_launch("hdy_paste_masks");
}

static int pm_args_ok(const void* protos, int proto_dtype, const float* coef, const float* boxes, const int32_t* counts, int bs,
                      int max_det, int nm, int mh, int mw, int ih, int iw) {
  HDY_REQUIRE(bs >= 0 && max_det >= 1 && nm >= 1 && nm <= 64 && mh >= 1 && mw >= 1 && ih >= 1 && iw >= 1,
              "process_mask: bad sizes (nm must be <= 64)");
  HDY_REQUIRE(proto_dtype == HDY_F32 || proto_dtype == HDY_F16, "process_mask: proto_dtype must be HDY_F32 or HDY_F16");
  if (bs > 0)
    HDY_REQUIRE(protos && coef && boxes && counts && ((uintptr_t)boxes & 15) == 0,
                "process_mask: NULL or misaligned pointer");
  return HDY_OK;
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_mask_select(const float* logits, const int64_t* labels, const int64_t* mask_indices, int K, int C, int M,
                    float* out, hdy_stream_t stream) {
  HDY_REQUIRE(K >= 0 && C >= 1 && M >= 1, "hdy_mask_select: bad sizes");
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(logits && labels && mask_indices && out, "hdy_mask_select: NULL pointer");
  mask_select_kernel<<<(unsigned)K, 128, 0, (cudaStream_t)stream>>>(logits, labels, mask_indices, K, C, M * M, out);
  return check_launch("hdy_mask_select");
}

int hdy_paste_masks(const float* src, const int32_t* channel, const float* boxes, int K, int C, int M, int padding,
                    int apply_sigmoid, int H, int W, float* out, hdy_stream_t stream) {
  int rc = paste_args_ok(src, boxes, K, C, M, padding, H, W);
  if (rc) return rc;
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(out != nullptr, "hdy_paste_masks: out is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)K * H * W * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  return launch_paste<false>(src, channel, boxes, K, C, M, padding, apply_sigmoid, H, W, out, nullptr, nullptr, 0,
                             nullptr, st);
}

int hdy_paste_geometry(const float* boxes, const int32_t* channel, int K, int M, int padding, int H, int W,
                       int32_t* geom, int64_t* offsets, hdy_stream_t stream) {
  HDY_REQUIRE(K >= 0 && M >= 1 && padding >= 0 && H >= 1 && W >= 1, "hdy_paste_geometry: bad sizes");
  HDY_REQUIRE(offsets != nullptr, "hdy_paste_geometry: offsets is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (K > 0) {
    HDY_REQUIRE(boxes && geom && ((uintptr_t)boxes & 15) == 0 && ((uintptr_t)geom & 15) == 0,
                "hdy_paste_geometry: NULL or misaligned pointer");
    const float scale = (float)((double)(M + 2 * padding) / (double)M);
    paste_geometry_kernel<<<(unsigned)((K + 127) / 128), 128, 0, st>>>(reinterpret_cast<const float4*>(boxes), channel,
                                                                       K, scale, H, W, geom);
  }
  scan_words(GeomWords{geom}, K, offsets, st);
  return check_launch("hdy_paste_geometry");
}

int hdy_paste_masks_packed(const float* src, const int32_t* channel, const float* boxes, const int64_t* offsets,
                           int K, int C, int M, int padding, int apply_sigmoid, int H, int W, uint32_t* bits,
                           int64_t capacity_words, int32_t* status, hdy_stream_t stream) {
  int rc = paste_args_ok(src, boxes, K, C, M, padding, H, W);
  if (rc) return rc;
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(offsets && bits && status && capacity_words >= 0, "hdy_paste_masks_packed: NULL pointer");
  return launch_paste<true>(src, channel, boxes, K, C, M, padding, apply_sigmoid, H, W, nullptr, offsets, bits,
                            capacity_words, status, (cudaStream_t)stream);
}

int hdy_unpack_masks(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int H, int W,
                     uint8_t* out, hdy_stream_t stream) {
  HDY_REQUIRE(K >= 0 && H >= 1 && W >= 1, "hdy_unpack_masks: bad sizes");
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(geom && offsets && bits && out && ((uintptr_t)geom & 15) == 0, "hdy_unpack_masks: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)K * H * W, st);
  if (e != cudaSuccess) {
    set_error("cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  unpack_masks_kernel<<<(unsigned)K, 128, 0, st>>>(geom, offsets, bits, H, W, out);
  return check_launch("hdy_unpack_masks");
}

size_t hdy_process_mask_workspace_bytes(int bs, int max_det) {
  return process_mask_workspace_bytes(bs > 0 ? bs : 0, max_det > 0 ? max_det : 0);
}

int hdy_process_mask(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                     const int32_t* counts, int bs, int max_det, int nm, int mh, int mw, int ih, int iw, int upsample,
                     float* out, void* workspace, size_t workspace_bytes, hdy_stream_t stream) {
  int rc = pm_args_ok(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw);
  if (rc) return rc;
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(out != nullptr, "hdy_process_mask: out is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t oh = upsample ? ih : mh, ow = upsample ? iw : mw;
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)bs * max_det * oh * ow * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  const float rx = (float)((double)mw / (double)iw), ry = (float)((double)mh / (double)ih);
  rc = launch_process_mask_regions(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw, upsample,
                                   rx, ry, out, nullptr, nullptr, nullptr, 0, nullptr, workspace, workspace_bytes, st);
  if (rc != 1) return rc;
  return launch_process_mask_kernel<false>(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw,
                                           upsample, rx, ry, out, nullptr, nullptr, nullptr, 0, nullptr, st,
                                           "hdy_process_mask");
}

int hdy_process_mask_geometry(const float* boxes, const int32_t* counts, int bs, int max_det, int mh, int mw, int ih,
                              int iw, int upsample, const uint8_t* row_state, const int64_t* tile_offsets,
                              int32_t* geom, int64_t* offsets, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det >= 1 && mh >= 1 && mw >= 1 && ih >= 1 && iw >= 1, "process_mask_geometry: bad sizes");
  HDY_REQUIRE(offsets != nullptr, "process_mask_geometry: offsets is NULL");
  HDY_REQUIRE(!row_state || tile_offsets, "process_mask_geometry: row_state needs tile_offsets");
  cudaStream_t st = (cudaStream_t)stream;
  const long long K = (long long)bs * max_det;
  if (K > 0)
    HDY_REQUIRE(boxes && counts && geom && ((uintptr_t)boxes & 15) == 0 && ((uintptr_t)geom & 15) == 0,
                "process_mask_geometry: NULL or misaligned pointer");
  const float rx = (float)((double)mw / (double)iw), ry = (float)((double)mh / (double)ih);
  scan_words(PmWindowWords{reinterpret_cast<const float4*>(boxes), counts, max_det, mh, mw, ih, iw, upsample, rx, ry,
                           row_state, tile_offsets, geom},
             K, offsets, st);
  return check_launch("hdy_process_mask_geometry");
}

int hdy_process_mask_rows(int32_t* geom, int64_t* offsets, const int32_t* counts, const int64_t* tile_offsets,
                          const float* rois, int bs, int max_det, int64_t* cursor2, int parity, int32_t* geom_rows,
                          int64_t* off_rows, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det >= 1, "hdy_process_mask_rows: bad sizes");
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(geom && offsets && counts && tile_offsets && rois && cursor2 && geom_rows && off_rows,
              "hdy_process_mask_rows: NULL pointer");
  HDY_REQUIRE((((uintptr_t)geom | (uintptr_t)geom_rows | (uintptr_t)rois) & 15) == 0,
              "hdy_process_mask_rows: geom / geom_rows / rois must be 16-byte aligned");
  const long long K = (long long)bs * max_det;
  pm_rows_kernel<<<(unsigned)((K + 1 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      geom, offsets, counts, tile_offsets, reinterpret_cast<const float4*>(rois), K, max_det, cursor2, parity,
      geom_rows, off_rows);
  return check_launch("hdy_process_mask_rows");
}

int hdy_process_mask_packed(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                            const int32_t* counts, const int32_t* geom, const int64_t* offsets, int bs, int max_det, int nm, int mh, int mw, int ih, int iw,
                            int upsample, uint32_t* bits, int64_t capacity_words, int32_t* status, void* workspace,
                            size_t workspace_bytes, hdy_stream_t stream) {
  int rc = pm_args_ok(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw);
  if (rc) return rc;
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(offsets && bits && status && capacity_words >= 0, "hdy_process_mask_packed: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const float rx = (float)((double)mw / (double)iw), ry = (float)((double)mh / (double)ih);
  // two-phase path: every word of every mask is written exactly once, nothing to clear
  HDY_REQUIRE(!geom || ((uintptr_t)geom & 15) == 0, "hdy_process_mask_packed: geom must be 16-byte aligned");
  rc = launch_process_mask_regions(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw, upsample,
                                   rx, ry, nullptr, geom, offsets, bits, capacity_words, status, workspace,
                                   workspace_bytes, st);
  if (rc != 1) return rc;
  // per-detection path: bits are OR-ed in, clear first (capacity is an upper bound the caller sized)
  cudaError_t e = cudaMemsetAsync(bits, 0, (size_t)capacity_words * 4, st);
  if (e != cudaSuccess) {
    set_error("cudaMemsetAsync: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  return launch_process_mask_kernel<true>(protos, proto_dtype, coef, boxes, counts, bs, max_det, nm, mh, mw, ih, iw,
                                          upsample, rx, ry, nullptr, geom, offsets, bits, capacity_words, status, st,
                                          "hdy_process_mask_packed");
}

}  // extern "C"
