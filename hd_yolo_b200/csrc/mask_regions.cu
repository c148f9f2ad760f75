// Two-phase process_mask: the north-star mask kernel (prototype x coefficient contraction in fp32 FFMA, sigmoid, box
// crop, bilinear upsample, > 0.5, bit-packed), with the prototypes staged through TMA.
//
// Semantics: ultralytics/yolov5 v7 utils/segment/general.py::process_mask + crop_mask (restated in oracle/port.py;
// the reference repo has no such function, see DESIGN.md), identical to process_mask_kernel in mask.cu.
//
// A tile's prototypes are [32, mh, mw] fp32 (8.4 MB at 1024 px); a nucleus touches a ~10x10 window of all 32 planes
// and produces a ~36x36 output window.  The two halves of the work want different decompositions:
//
//   phase 1  proto_patch_kernel, one CTA per (tile, 24x24 proto REGION).  ONE 4-D TMA tile load
//            (cp.async.bulk.tensor.4d, SASS UTMALDG; out-of-bounds zero-filled by the TMA unit) brings the region's
//            24x24x32 box into 72 KB of shared memory, so every proto element leaves HBM/L2 exactly once.  While it is
//            in flight the CTA lists the tile's detections whose box reaches into the region; then one warp per
//            (detection, region) piece computes the cropped sigmoid(coef . proto) of the piece's pixels (32 LDS + 32
//            FFMA each) and writes them into the detection's PATCH (<= 16x16 floats) in the workspace.  Three CTAs
//            per SM, no halo, no atomics.  The tile origin of a TMA load must be 16-byte aligned in the innermost
//            dimension (measured: tools/micro/tma4d_test.cu faults otherwise), hence 24-pixel regions.
//   phase 2  one WARP per detection: the patch (with a ring of zeros: the crop) goes to shared memory and is
//            upsampled with ATen's bilinear (align_corners=False) operation by operation, thresholded and stored.
//            Every word of every mask is stored exactly once, so the bit planes need no clearing.
//              * bit-packed + upsampled (the throughput form): mask_upsample_pack2_kernel (upsample_pack_v2 below).
//              * the other forms (dense output, or packed at proto resolution): mask_upsample_pack_kernel.
//   Detections whose kept range exceeds 16x16 proto pixels (64 px boxes at the usual 4x), or that fall into an overfull
//   region, are listed and handled by the per-detection body of mask.cu.  In the packed + upsampled form they ride in
//   the first CTAs of the phase-1 launch; in the other forms they get a launch of their own behind phase 2.
//   The packed + upsampled form needs the windows of hdy_process_mask_geometry; without them the caller falls back to
//   the per-detection kernel.
#include <algorithm>

#include "tma_common.cuh"
#include "mask_common.cuh"

namespace hdy {

// region == TMA box: a tile origin must be 16-byte aligned in x (24 fp32 = 96 bytes, 24 fp16 = 48 bytes)
constexpr int kRegBoxX = 24, kRegBoxY = 24;
constexpr int kRegNm = 32;
constexpr int kRegThreads = 256;
constexpr int kRegWarps = kRegThreads / 32;
constexpr int kRegList = 512;  // detections examined per pass

template <typename E>
struct RegSmemT {
  E proto[kRegNm][kRegBoxY][kRegBoxX];  // TMA destination (dense, x fastest); fp32, or fp16 widened on use
  float coef[kRegWarps][kRegNm];
  uint16_t list[kRegList];
  int nlist;
  int pad;
  uint64_t bar;
};
__device__ __forceinline__ float proto_f32(float v) { return v; }
__device__ __forceinline__ float proto_f32(__half v) { return __half2float(v); }  // exact

// workspace: [0] large-detection counter, [1] slot ticket of the packed upsample, large list (int32 per slot), the
// patches, then the per-region detection lists (count + kRegCap uint16 entries per (tile, region); sized for the
// largest proto plane, see kMaxRegions)
constexpr int kRegCap = 254;          // detections listed per region; a region with more falls back to scanning
constexpr int kMaxRegionsPerTile = 512;  // ceil(mw/24) * ceil(mh/24) <= 512 covers planes up to 528 x 528 (2112 px tiles)
struct RegionList {
  int32_t count;
  uint16_t det[kRegCap];
};
static_assert(sizeof(RegionList) == 512, "one region list is 512 bytes");
struct PmWorkspace {
  int32_t* large_count;   // detections left to the per-detection kernel
  uint32_t* ticket;       // next slot of the packed + upsampled phase 2 (mask_upsample_pack2_kernel)
  int32_t* large_list;
  float* patches;
  RegionList* regions;
  int4* kr;               // per slot: kept proto range (px0, py0, px1, py1), written by the binning kernel
};
static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
size_t process_mask_workspace_bytes(long long bs, long long max_det) {
  const long long slots = bs * max_det;
  return 256 + align256((size_t)slots * 4) + align256((size_t)slots * 16) +
         (size_t)slots * kPatchPitch * kPatchPitch * 4 + (size_t)bs * kMaxRegionsPerTile * sizeof(RegionList);
}
static PmWorkspace pm_workspace(void* base, long long slots) {
  PmWorkspace w;
  unsigned char* p = static_cast<unsigned char*>(base);
  w.large_count = reinterpret_cast<int32_t*>(p);
  w.ticket = reinterpret_cast<uint32_t*>(p + 4);
  p += 256;
  w.large_list = reinterpret_cast<int32_t*>(p);
  p += align256((size_t)slots * 4);
  w.kr = reinterpret_cast<int4*>(p);
  p += align256((size_t)slots * 16);
  w.patches = reinterpret_cast<float*>(p);
  p += (size_t)slots * kPatchPitch * kPatchPitch * 4;
  w.regions = reinterpret_cast<RegionList*>(p);
  return w;
}

struct KeptRange {
  float x1d, y1d, x2d, y2d;
  int px0, py0, px1, py1;
};
__device__ __forceinline__ KeptRange kept_range(const float4 b, float rx, float ry, int mw, int mh) {
  KeptRange k;
  k.x1d = __fmul_rn(b.x, rx);  // downsampled_bboxes[:, 0] *= mw / iw ...
  k.x2d = __fmul_rn(b.z, rx);
  k.y1d = __fmul_rn(b.y, ry);
  k.y2d = __fmul_rn(b.w, ry);
  k.px0 = ceil_to_int_clamped(k.x1d, 0, mw);
  k.px1 = ceil_to_int_clamped(k.x2d, 0, mw);
  k.py0 = ceil_to_int_clamped(k.y1d, 0, mh);
  k.py1 = ceil_to_int_clamped(k.y2d, 0, mh);
  // a NaN coordinate fails every crop comparison of the reference: nothing is kept.  For finite coordinates the crop
  // test x1d <= col < x2d over integer columns IS col in [px0, px1) (px = ceil, clamped), so the kernels below walk the
  // integer range and never compare against the floats again.
  if (!(k.x1d == k.x1d) || !(k.x2d == k.x2d) || !(k.y1d == k.y1d) || !(k.y2d == k.y2d)) k.px1 = k.px0, k.py1 = k.py0;
  return k;
}

// floor(v / pw) for 0 <= v < 64 and 1 <= pw <= 16 as (v * ceil(2^16 / pw)) >> 16 (exact while v * pw < 2^16): the
// piece loops split the 32 lanes into floor(32 / pw) rows of pw pixels, and an integer division costs ~20 instructions
__constant__ int c_inv16[17] = {0,     65536, 32768, 21846, 16384, 13108, 10923, 9363, 8192,
                                7282,  6554,  5958,  5462,  5042,  4682,  4370,  4096};

// ------------------------------------------------------------------------------------------------ phase 0
// One thread per detection: append it to the list of every region its kept range touches (1-4 for a nucleus), so that
// a phase-1 CTA does not have to scan the whole tile (121 regions x 2 650 boxes per 1024-px tile otherwise).
__global__ void __launch_bounds__(256) proto_bin_kernel(const float4* __restrict__ boxes,
                                                        const int32_t* __restrict__ counts, long long n_slots,
                                                        int max_det, int mh, int mw, int rxn, int ryn, float rx,
                                                        float ry, const int32_t* __restrict__ geom4,
                                                        RegionList* __restrict__ regions, int4* __restrict__ kr) {
  const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  const int tile = (int)(slot / max_det), d = (int)(slot - (long long)tile * max_det);
  // a slot beyond counts, or (packed form) without an output window -- empty, or not KEPT by the slide-level merge --
  // needs no patch: its kept range is recorded as empty
  const bool live = d < counts[tile] && !(geom4 && (geom4[4 * slot + 2] <= 0 || geom4[4 * slot + 3] <= 0));
  KeptRange k;
  k.px0 = k.py0 = k.px1 = k.py1 = 0;
  if (live) k = kept_range(boxes[slot], rx, ry, mw, mh);
  kr[slot] = make_int4(k.px0, k.py0, k.px1, k.py1);
  if (k.px1 <= k.px0 || k.py1 <= k.py0) return;
  if (k.px1 - k.px0 > kPatchPitch || k.py1 - k.py0 > kPatchPitch) return;  // per-detection kernel
  const int rx0 = k.px0 / kRegBoxX, rx1 = (k.px1 - 1) / kRegBoxX;
  const int ry0 = k.py0 / kRegBoxY, ry1 = (k.py1 - 1) / kRegBoxY;
  for (int ryy = ry0; ryy <= ry1; ++ryy)
    for (int rxx = rx0; rxx <= rx1; ++rxx) {
      RegionList& R = regions[(size_t)tile * (rxn * ryn) + ryy * rxn + rxx];
      const int pos = atomicAdd(&R.count, 1);
      if (pos < kRegCap) R.det[pos] = (uint16_t)d;
    }
}

// ------------------------------------------------------------------------------------------------ phase 1
// One piece: the kept pixels of a detection inside one region, contracted against the region's 32 prototype planes in
// shared memory.  Lanes cover floor(32 / pw) rows of pw pixels at a time.  emit(x - px0, y - py0, value).
template <typename E, typename Emit>
__device__ __forceinline__ void contract_piece(const E (*proto)[kRegBoxY][kRegBoxX], const float* __restrict__ coef_smem,
                                               const int4 kr, int X0, int Y0, int lane, Emit emit) {
  float cf[kRegNm];
#pragma unroll
  for (int c = 0; c < kRegNm; c += 4) {
    const float4 v = *reinterpret_cast<const float4*>(coef_smem + c);
    cf[c] = v.x;
    cf[c + 1] = v.y;
    cf[c + 2] = v.z;
    cf[c + 3] = v.w;
  }
  const int qx0 = max(kr.x, X0), qx1 = min(kr.z, X0 + kRegBoxX);
  const int qy0 = max(kr.y, Y0), qy1 = min(kr.w, Y0 + kRegBoxY);
  const int pw = qx1 - qx0;  // 1..16
  const int inv = c_inv16[pw];
  const int rows_per = (32 * inv) >> 16;
  const int ly = (lane * inv) >> 16, lx = lane - ly * pw;
  if (ly >= rows_per) return;
  const int xx = qx0 + lx, sx = xx - X0;
  for (int yy = qy0 + ly; yy < qy1; yy += rows_per) {
    const int sy = yy - Y0;
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < kRegNm; ++c) acc = fmaf(cf[c], proto_f32(proto[c][sy][sx]), acc);
    emit(xx - kr.x, yy - kr.y, sigmoidf_ref(acc));
  }
}

// The detections the patch path leaves out (listed by the binning kernel: windows over 16 x 16 proto pixels, overfull
// regions) ride in the same launch: the first `ctas` CTAs run the per-detection body of mask.cu on them (64 proto tiles
// x ctas / 64 list strides), in a corner of the region buffer, while the others stream the regions.  As a kernel of its
// own behind the upsample that work was a 27-70 us latency chain in a handful of CTAs at the end of every mask call.
struct ListedRide {
  const void* protos;
  const float4* boxes;
  const int64_t* offsets;
  uint32_t* bits;
  int32_t* status;
  const int32_t* list;
  const int32_t* list_count;
  long long capacity_words;
  float rx, ry;
  int nm, mh, mw, ih, iw;
  int ctas;   // 0: nothing rides (dense / not upsampled forms keep the separate launch)
};
constexpr int kListedTiles = 64;

template <typename E>
__global__ void __launch_bounds__(kRegThreads, 3) proto_patch_kernel(
    const __grid_constant__ CUtensorMap tmap, const float* __restrict__ coef, const int4* __restrict__ krs,
    const int32_t* __restrict__ counts, int max_det, int rxn, int ryn, float* __restrict__ patches,
    const RegionList* __restrict__ regions, const ListedRide LR) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  if ((int)blockIdx.x < LR.ctas) {
    float* stage = reinterpret_cast<float*>(smem_raw);
    process_mask_body<true, sizeof(E) == 2>(LR.protos, coef, LR.boxes, counts, max_det, LR.nm, LR.mh, LR.mw, LR.ih, LR.iw,
                                            1, LR.rx, LR.ry, nullptr, nullptr, LR.offsets, LR.bits, LR.capacity_words,
                                            LR.status, LR.list, (long long)*LR.list_count,
                                            (long long)(blockIdx.x / kListedTiles), (long long)(LR.ctas / kListedTiles),
                                            (int)(blockIdx.x % kListedTiles), kListedTiles, stage,
                                            stage + kPmStage * kPmStage);
    return;
  }
  const int bid = (int)blockIdx.x - LR.ctas;
  RegSmemT<E>& S = *reinterpret_cast<RegSmemT<E>*>(smem_raw);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int per_tile = rxn * ryn;
  const int tile = bid / per_tile, reg = bid - tile * per_tile;
  const int RY = reg / rxn, RX = reg - RY * rxn;
  const int X0 = RX * kRegBoxX, Y0 = RY * kRegBoxY;
  const RegionList& RL = regions[bid];
  const int listed = RL.count;
  if (listed <= 0) return;  // nothing reaches into this region: no load at all
  const bool use_list = listed <= kRegCap;
  const int n = use_list ? listed : min(counts[tile], max_det);

  if (t == 0) {
    mbar_init(&S.bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive_expect_tx(&S.bar, (uint32_t)sizeof(S.proto));
    tma_load_4d(&S.proto[0][0][0], &tmap, X0, Y0, 0, tile, &S.bar);
  }
  bool loaded = false;
  for (int base = 0; base < n; base += kRegList) {
    __syncthreads();
    if (t == 0) S.nlist = 0;
    __syncthreads();
    const int lim = min(base + kRegList, n);
    if (use_list) {
      // the binning pass already listed the detections of this region
      for (int i = base + t; i < lim; i += kRegThreads) S.list[i - base] = RL.det[i];
      if (t == 0) S.nlist = lim - base;
    } else {
      // overfull list (more than kRegCap detections in one region): scan the tile (slots the binning pass skipped --
      // beyond counts, empty, not KEPT -- carry no kept range of this launch: they are filtered by counts / geometry
      // in the binning pass only, so the scan re-checks the range itself)
      for (int d = base + t; d < lim; d += kRegThreads) {
        const int4 k = krs[(size_t)tile * max_det + d];
        if (k.z <= k.x || k.w <= k.y) continue;
        if (k.z - k.x > kPatchPitch || k.w - k.y > kPatchPitch) continue;  // per-detection kernel
        if (k.z <= X0 || k.x >= X0 + kRegBoxX || k.w <= Y0 || k.y >= Y0 + kRegBoxY) continue;
        S.list[atomicAdd(&S.nlist, 1)] = (uint16_t)(d - base);
      }
    }
    __syncthreads();
    const int nl = S.nlist;
    // software pipeline over this warp's pieces: the kept range and the coefficients of the NEXT piece are requested
    // before the current one is computed (and those of the first piece before waiting for the TMA load)
    int e = warp;
    size_t nslot = 0;
    int4 nkr = make_int4(0, 0, 0, 0);
    float ncoef = 0.f;
    auto fetch = [&](int ee) {
      nslot = (size_t)tile * max_det + (use_list ? 0 : base) + S.list[ee];
      nkr = krs[nslot];
      ncoef = coef[nslot * kRegNm + lane];
    };
    if (e < nl) fetch(e);
    if (!loaded) {
      while (!mbar_try_wait(&S.bar, 0)) {
      }
      loaded = true;
    }
    for (; e < nl; e += kRegWarps) {
      const size_t slot = nslot;
      const int4 k = nkr;
      __syncwarp();
      S.coef[warp][lane] = ncoef;
      __syncwarp();
      if (e + kRegWarps < nl) fetch(e + kRegWarps);
      float* dst = patches + slot * (kPatchPitch * kPatchPitch);
      contract_piece<E>(S.proto, S.coef[warp], k, X0, Y0, lane,
                        [&](int px, int py, float v) { dst[py * kPatchPitch + px] = v; });
    }
  }
  if (!loaded) {  // never leave with the bulk copy still in flight
    while (!mbar_try_wait(&S.bar, 0)) {
    }
  }
}

// ------------------------------------------------------------------------------------------------ phase 2
constexpr int kUpWarps = 8;
constexpr int kPatchRing = kPatchPitch + 2;  // patch with a ring of zeros (the crop)
constexpr int kRowChunk = 64;

struct RowTab {
  int i0, i1;  // source rows, relative to the ringed patch
  float l0, l1;
};

struct UpSmem {
  float patch[kUpWarps][kPatchRing * kPatchRing];
  float col[kUpWarps][kPatchRing][32];  // x-interpolated values of the lanes' columns, per source row
  RowTab rows[kUpWarps][kRowChunk];
};

template <bool PACKED, bool UPSAMPLE>
__global__ void __launch_bounds__(kUpWarps * 32) mask_upsample_pack_kernel(
    const float* __restrict__ patches, const float4* __restrict__ boxes, const int32_t* __restrict__ counts,
    long long n_slots, int max_det, int mh, int mw, int ih, int iw, float rx, float ry, float* __restrict__ out_dense,
    const int32_t* __restrict__ geom4, const int64_t* __restrict__ offsets, uint32_t* __restrict__ bits,
    long long capacity_words,
    int32_t* __restrict__ status, int32_t* __restrict__ large_count, int32_t* __restrict__ large_list) {
  static_assert(!(PACKED && UPSAMPLE), "the packed + upsampled form runs mask_upsample_pack2_kernel");
  __shared__ UpSmem S;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long slot = (long long)blockIdx.x * kUpWarps + warp;
  if (slot >= n_slots) return;
  const int tile = (int)(slot / max_det), d = (int)(slot - (long long)tile * max_det);
  if (d >= counts[tile]) return;
  PMGeom g;
  if (geom4) {
    // the window was computed (and trimmed) once by the geometry kernel: only the kept proto range is redone here
    const KeptRange k = kept_range(boxes[slot], rx, ry, mw, mh);
    const int4 wdw = reinterpret_cast<const int4*>(geom4)[slot];
    g.x1d = k.x1d, g.y1d = k.y1d, g.x2d = k.x2d, g.y2d = k.y2d;
    g.px0 = k.px0, g.py0 = k.py0, g.px1 = k.px1, g.py1 = k.py1;
    g.x0 = wdw.x, g.y0 = wdw.y, g.w = wdw.z, g.h = wdw.w;
  } else {
    g = pm_geometry(boxes[slot], mh, mw, ih, iw, UPSAMPLE ? 1 : 0, rx, ry);
  }
  if (g.w <= 0 || g.h <= 0) return;
  const int wpr = (g.w + 31) >> 5;
  const int oh = UPSAMPLE ? ih : mh, ow = UPSAMPLE ? iw : mw;
  long long off = 0;
  if (PACKED) {
    off = offsets[slot];
    if (off + (long long)wpr * g.h > capacity_words) {
      if (lane == 0) atomicOr(status, HDY_STATUS_OVERFLOW);
      return;
    }
  }
  const int pw = g.px1 - g.px0, ph = g.py1 - g.py0;
  if (pw > kPatchPitch || ph > kPatchPitch) {
    // too large for the patch path: clear its words (the per-detection kernel ORs into them) and list it
    if (PACKED)
      for (long long i = lane; i < (long long)wpr * g.h; i += 32) bits[off + i] = 0u;
    if (lane == 0) large_list[atomicAdd(large_count, 1)] = (int32_t)slot;
    return;
  }
  // ---- patch with its ring of zeros: element (y, x) of the proto plane sits at [(y - py0 + 1)][(x - px0 + 1)]
  float* P = S.patch[warp];
  {
    // interior: the 16 x 16 patch, coalesced 128-byte rows (entries outside pw x ph are stale: masked to zero)
    const float* src = patches + slot * (kPatchPitch * kPatchPitch);
#pragma unroll
    for (int i = lane; i < kPatchPitch * kPatchPitch; i += 32) {
      const int y = i >> 4, x = i & 15;
      P[(y + 1) * kPatchRing + x + 1] = (y < ph && x < pw) ? src[i] : 0.f;
    }
    // ring: rows 0 and 17, columns 0 and 17
    for (int i = lane; i < 4 * kPatchRing; i += 32) {
      const int k = i / kPatchRing, j = i - k * kPatchRing;
      const int idx = k == 0 ? j : (k == 1 ? (kPatchRing - 1) * kPatchRing + j : (k == 2 ? j * kPatchRing : j * kPatchRing + kPatchRing - 1));
      P[idx] = 0.f;
    }
  }
  __syncwarp();

  if (!UPSAMPLE) {
    // output pixel == proto pixel: the window is the kept range itself
    for (int w = 0; w < wpr; ++w) {
      const int c = (w << 5) + lane;
      const bool valid = c < g.w;
      for (int r = 0; r < g.h; ++r) {
        const bool bit = valid && P[(r + 1) * kPatchRing + (valid ? c + 1 : 0)] > 0.5f;
        if (PACKED) {
          const unsigned word = __ballot_sync(0xffffffffu, bit);
          if (lane == 0) bits[off + (long long)r * wpr + w] = word;
        } else if (valid) {
          out_dense[slot * oh * ow + (size_t)(g.y0 + r) * ow + g.x0 + c] = bit ? 1.f : 0.f;
        }
      }
    }
    return;
  }

  const float sxs = (float)mw / (float)iw, sys = (float)mh / (float)ih;  // ATen: scale = in / out (fp32)
  RowTab* rowtab = S.rows[warp];
  float(*col)[32] = S.col[warp];
  const int src_rows = ph + 2;  // ringed patch rows that can be touched
  for (int r0 = 0; r0 < g.h; r0 += kRowChunk) {
    const int nr = min(kRowChunk, g.h - r0);
    __syncwarp();
    for (int r = lane; r < nr; r += 32) {
      const Lerp Y = lerp_coord(g.y0 + r0 + r, sys, mh);
      RowTab T;
      // taps outside [py0 - 1, py1] contribute nothing (cropped): clamp them onto the ring of zeros
      T.i0 = min(max(Y.i0 - g.py0 + 1, 0), ph + 1);
      T.i1 = min(max(Y.i1 - g.py0 + 1, 0), ph + 1);
      T.l0 = Y.l0;
      T.l1 = Y.l1;
      rowtab[r] = T;
    }
    __syncwarp();
    for (int w = 0; w < wpr; ++w) {
      const int vw = min(32, g.w - (w << 5));  // valid columns of this word
      if (vw <= 16) {
        // narrow word (the tail of a 36-px window is 4 columns): lanes cover floor(32 / vw) output rows at a time
        const int rows_per = 32 / vw;
        const int lr = lane / vw, lc = lane - lr * vw;
        const bool active = lr < rows_per;
        const Lerp X = lerp_coord(g.x0 + (w << 5) + lc, sxs, mw);
        const int xi0 = min(max(X.i0 - g.px0 + 1, 0), pw + 1), xi1 = min(max(X.i1 - g.px0 + 1, 0), pw + 1);
        __syncwarp();
        if (active)
          for (int s = lr; s < src_rows; s += rows_per)
            col[s][lc] = __fadd_rn(__fmul_rn(X.l0, P[s * kPatchRing + xi0]), __fmul_rn(X.l1, P[s * kPatchRing + xi1]));
        __syncwarp();
        for (int rb = 0; rb < nr; rb += rows_per) {
          const int r = rb + lr;
          if (active && r < nr) {
            const float4 rt = *reinterpret_cast<const float4*>(&rowtab[r]);
            const float v = __fadd_rn(__fmul_rn(rt.z, col[__float_as_int(rt.x)][lc]),
                                      __fmul_rn(rt.w, col[__float_as_int(rt.y)][lc]));
            out_dense[slot * oh * ow + (size_t)(g.y0 + r0 + r) * ow + g.x0 + (w << 5) + lc] = v > 0.5f ? 1.f : 0.f;
          }
        }
        continue;
      }
      const int c = (w << 5) + lane;
      const bool valid = c < g.w;
      const Lerp X = lerp_coord(g.x0 + (valid ? c : 0), sxs, mw);
      const int xi0 = min(max(X.i0 - g.px0 + 1, 0), pw + 1), xi1 = min(max(X.i1 - g.px0 + 1, 0), pw + 1);
      // x pass: top/bot of ATen's formula for every source row, once per word
      __syncwarp();
      for (int s = 0; s < src_rows; ++s)
        col[s][lane] = __fadd_rn(__fmul_rn(X.l0, P[s * kPatchRing + xi0]), __fmul_rn(X.l1, P[s * kPatchRing + xi1]));
      __syncwarp();
      float* dd = out_dense + slot * oh * ow + (size_t)(g.y0 + r0) * ow + g.x0 + c;
#pragma unroll 4
      for (int r = 0; r < nr; ++r) {
        const float4 rt = *reinterpret_cast<const float4*>(&rowtab[r]);
        const float v = __fadd_rn(__fmul_rn(rt.z, col[__float_as_int(rt.x)][lane]),
                                  __fmul_rn(rt.w, col[__float_as_int(rt.y)][lane]));
        if (valid) dd[(size_t)r * ow] = v > 0.5f ? 1.f : 0.f;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ packed + upsampled
// The throughput form (bit planes of the upsampled masks) has kernels of its own:
//   * the binning kernel records every slot's kept proto range (so nobody recomputes it from the box) and lists the
//     detections that do not fit the patch path (kept range over 16 x 16 proto pixels, or an overfull region list):
//     those ride in the region launch (ListedRide), their words cleared beforehand by pm_clear_listed_kernel;
//   * upsample_pack_v2: one warp per detection.  The sigmoid patch sits in shared memory with a ring of zeros (the
//     crop).  x pass with lane = output column (two taps per source row), results stored TRANSPOSED; y pass with lane =
//     output ROW: every lane walks the columns of its row, blends two of the stored values per pixel and sets the bit
//     in a register -- 7 instructions per column for 32 rows at once, no ballots, no row tables, one coalesced store
//     of the row words.  (mask_upsample_pack_kernel runs lane = column with a ballot per row: ~13 instructions per row
//     and a special case for narrow tail words; 1 000 warp instructions per detection, 70 % of the issue slots.)
constexpr int kV2Warps = 8;
constexpr int kV2Threads = kV2Warps * 32;
constexpr int kXRows = 20;                // source rows the x pass may compute (src_rows rounded up to a multiple of 4)
// x-pass results of the current 32 output columns, stored for the y pass as PAIRS of adjacent columns:
// [column >> 1][source row][column & 1], kPairPitch floats per column pair.  The y pass (lane = output row) reads
// the two columns of a pair with one 64-bit load and multiplies them with one packed FMUL2 (sm_100 f32x2: two IEEE
// roundings in one instruction); kPairPitch = 42 keeps the x pass's stores (lane = column) conflict-free.
constexpr int kPairPitch = 2 * (kXRows + 1);
// ringed patch in shared memory: ring row s at P[s * kUpPitch ...], element (y, x) of the kept range at
// [(y + 1) * kUpPitch + kUpX0 + x] (rows 16-byte aligned, so a row of the workspace patch is one float4 per 4 pixels),
// ring column xi (0 = left zero column, pw + 1 = right zero column) at [.. + kUpX0 - 1 + xi]
constexpr int kUpPitch = 24;
constexpr int kUpX0 = 4;

struct UpWarpSmem {
  float patch[kXRows * kUpPitch];   // ringed patch (rows beyond ph + 1 are never used, only read by the x pass)
  float colT[16 * kPairPitch];      // x-pass results, see kPairPitch
};

__device__ __forceinline__ unsigned long long f32x2_pack(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
// two IEEE fp32 products in one instruction (FMUL2); the sums stay scalar FADDs: ptxas contracts mul.f32x2 + add.f32x2
// into FFMA2 even under -fmad=false, which would round once where ATen rounds twice
__device__ __forceinline__ void f32x2_mul(unsigned long long a, unsigned long long b, float& lo, float& hi) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(r));
}

// Only what the taps can reach has to be zero: ring rows 0 and ph + 1 (columns 0 .. pw + 1) and the two ring columns
// of the rows in between.  Entries past the kept range that a float4 copy of a workspace row drags in are never read.
__device__ __forceinline__ void up_zero_ring(float* P, int pw, int ph, int lane) {
  if (lane < kPatchRing) {
    P[kUpX0 - 1 + lane] = 0.f;                              // ring row 0
    P[(ph + 1) * kUpPitch + kUpX0 - 1 + lane] = 0.f;        // ring row ph + 1
    if (lane < ph) {
      P[(lane + 1) * kUpPitch + kUpX0 - 1] = 0.f;           // left ring column
      P[(lane + 1) * kUpPitch + kUpX0 + pw] = 0.f;          // right ring column
    }
  }
}

// workspace patch (pitch 16, [ph][pw] valid) -> ringed shared-memory patch: one float4 per lane and 8 rows
__device__ __forceinline__ void up_load_patch(float* P, const float* __restrict__ src, int pw, int ph, int lane) {
  const int row = lane >> 2, quad = lane & 3;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
  const bool ra = row < ph, rb = row + 8 < ph;
  if (ra) a = s4[row * 4 + quad];
  if (rb) b = s4[(row + 8) * 4 + quad];
  if (ra) *reinterpret_cast<float4*>(P + (row + 1) * kUpPitch + kUpX0 + quad * 4) = a;
  if (rb) *reinterpret_cast<float4*>(P + (row + 9) * kUpPitch + kUpX0 + quad * 4) = b;
  __syncwarp();
  up_zero_ring(P, pw, ph, lane);   // after the copy: the right ring column lies inside the copied floats
}

// ATen bilinear (align_corners=False), operation by operation, + threshold + pack of one detection.
// P: ringed patch (layout above).  sxs / sys: ATen's scale = in / out, computed in fp32 on the host.
__device__ __forceinline__ void upsample_pack_v2(const float* __restrict__ P, float* __restrict__ colT, const int4 kr,
                                                 const int4 wdw, long long off, uint32_t* __restrict__ bits, int mh,
                                                 int mw, float sxs, float sys, int lane) {
  const int pw = kr.z - kr.x, ph = kr.w - kr.y;
  const int gx0 = wdw.x, gy0 = wdw.y, gw = wdw.z, gh = wdw.w;
  const int wpr = (gw + 31) >> 5;
  const int src_rows = ph + 2;
  for (int w = 0; w < wpr; ++w) {
    const int vw = min(32, gw - (w << 5));  // valid columns of this word
    // x pass (lane = column): top / bot of ATen's formula for every source row
    const int c = (w << 5) + lane;
    const Lerp X = lerp_coord(gx0 + (c < gw ? c : 0), sxs, mw);
    // taps outside [px0 - 1, px1] contribute nothing (cropped): clamp them onto the ring of zeros
    const float* p0 = P + kUpX0 - 1 + min(max(X.i0 - kr.x + 1, 0), pw + 1);
    const float* p1 = P + kUpX0 - 1 + min(max(X.i1 - kr.x + 1, 0), pw + 1);
    __syncwarp();  // the previous word's y pass is done with colT
    float* ct = colT + (lane >> 1) * kPairPitch + (lane & 1);
    // (source rows in fours: the rows past src_rows hold stale values nobody reads back)
    for (int s = 0; s < src_rows; s += 4) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        ct[(s + j) * 2] = __fadd_rn(__fmul_rn(X.l0, p0[(s + j) * kUpPitch]), __fmul_rn(X.l1, p1[(s + j) * kUpPitch]));
    }
    __syncwarp();
    // y pass (lane = row)
    for (int r0 = 0; r0 < gh; r0 += 32) {
      const int r = r0 + lane;
      const bool act = r < gh;
      const Lerp Y = lerp_coord(gy0 + (act ? r : 0), sys, mh);
      const float* c0 = colT + 2 * min(max(Y.i0 - kr.y + 1, 0), ph + 1);
      const float* c1 = colT + 2 * min(max(Y.i1 - kr.y + 1, 0), ph + 1);
      const unsigned long long W0 = f32x2_pack(Y.l0, Y.l0), W1 = f32x2_pack(Y.l1, Y.l1);
      uint32_t word = 0u;
      // two pixels: one 64-bit load per tap row, two FMUL2, two FADDs, two compares, two predicated ORs of an
      // immediate bit (word |= (v > 0.5f) << x)
#define HDY_SETBIT(v, x)                                                                                          \
  asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, 0f3F000000;\n\t@p or.b32 %0, %0, %2;\n\t}" : "+r"(word) : "f"(v), \
      "n"(1u << (x)));
#define HDY_PX2(x)                                                                                                \
  {                                                                                                               \
    float a0, a1, b0, b1;                                                                                         \
    f32x2_mul(W0, *reinterpret_cast<const unsigned long long*>(c0 + ((x) >> 1) * kPairPitch), a0, a1);            \
    f32x2_mul(W1, *reinterpret_cast<const unsigned long long*>(c1 + ((x) >> 1) * kPairPitch), b0, b1);            \
    const float v0 = __fadd_rn(a0, b0), v1 = __fadd_rn(a1, b1);                                                   \
    HDY_SETBIT(v0, (x))                                                                                           \
    HDY_SETBIT(v1, (x) + 1)                                                                                       \
  }
#define HDY_G4(g) HDY_PX2(g) HDY_PX2((g) + 2)
      // groups of four columns, nested so that the warp-uniform exit costs one branch per group
      HDY_G4(0)
      if (vw > 4) {
        HDY_G4(4)
        if (vw > 8) {
          HDY_G4(8)
          if (vw > 12) {
            HDY_G4(12)
            if (vw > 16) {
              HDY_G4(16)
              if (vw > 20) {
                HDY_G4(20)
                if (vw > 24) {
                  HDY_G4(24)
                  if (vw > 28) {
                    HDY_G4(28)
                  }
                }
              }
            }
          }
        }
      }
#undef HDY_G4
#undef HDY_PX2
#undef HDY_SETBIT
      if (vw < 32) word &= (1u << vw) - 1u;  // columns past the window were computed from clamped taps
      if (act) bits[off + (long long)r * wpr + w] = word;
    }
  }
}

// binning for the packed + upsampled kernels (see above)
__global__ void __launch_bounds__(256) proto_bin_fused_kernel(const float4* __restrict__ boxes,
                                                              const int32_t* __restrict__ counts, long long n_slots,
                                                              int max_det, int mh, int mw, int rxn, int ryn, float rx,
                                                              float ry, const int32_t* __restrict__ geom4,
                                                              RegionList* __restrict__ regions, int4* __restrict__ kr,
                                                              int32_t* __restrict__ large_count,
                                                              int32_t* __restrict__ large_list) {
  const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  const int tile = (int)(slot / max_det), d = (int)(slot - (long long)tile * max_det);
  // empty window, not KEPT (slide form) or beyond counts: no patch, an empty kept range
  const bool live = d < counts[tile] && geom4[4 * slot + 2] > 0 && geom4[4 * slot + 3] > 0;
  KeptRange k;
  k.px0 = k.py0 = k.px1 = k.py1 = 0;
  if (live) k = kept_range(boxes[slot], rx, ry, mw, mh);
  bool leave = false;
  if (k.px1 > k.px0 && k.py1 > k.py0) {
    leave = k.px1 - k.px0 > kPatchPitch || k.py1 - k.py0 > kPatchPitch;
    if (!leave) {
      const int rx0 = k.px0 / kRegBoxX, rx1 = (k.px1 - 1) / kRegBoxX;
      const int ry0 = k.py0 / kRegBoxY, ry1 = (k.py1 - 1) / kRegBoxY;
      for (int ryy = ry0; ryy <= ry1; ++ryy)
        for (int rxx = rx0; rxx <= rx1; ++rxx) {
          RegionList& R = regions[(size_t)tile * (rxn * ryn) + ryy * rxn + rxx];
          const int pos = atomicAdd(&R.count, 1);
          if (pos < kRegCap)
            R.det[pos] = (uint16_t)d;
          else
            leave = true;  // overfull region: hand the detection over (its other pieces are skipped: empty range)
        }
    }
    if (leave) large_list[atomicAdd(large_count, 1)] = (int32_t)slot;
  }
  kr[slot] = leave ? make_int4(0, 0, 0, 0) : make_int4(k.px0, k.py0, k.px1, k.py1);
}

// the words of the listed detections are cleared: the per-detection kernel ORs its bits in
__global__ void pm_clear_listed_kernel(const int32_t* __restrict__ geom4, const int64_t* __restrict__ offsets,
                                       uint32_t* __restrict__ bits, long long capacity_words,
                                       const int32_t* __restrict__ list, const int32_t* __restrict__ list_count) {
  const int n = *list_count;
  for (int item = blockIdx.x; item < n; item += gridDim.x) {
    const long long slot = list[item];
    const int4 g = reinterpret_cast<const int4*>(geom4)[slot];
    const long long words = (long long)((g.z + 31) >> 5) * g.w, off = offsets[slot];
    if (off + words > capacity_words) continue;  // reported by the kernel that would have filled them
    for (long long i = threadIdx.x; i < words; i += blockDim.x) bits[off + i] = 0u;
  }
}

// phase 2 of the packed + upsampled form: one warp per detection, patch from the workspace.  Persistent: as many CTAs
// as fit the GPU at once (6 per SM: 36 KB of shared memory and 256 x 40 registers each), every warp takes `chunk`
// slots at a time from a ticket until none are left (chunk: about four tickets per warp, at most kV2Chunk -- one
// atomic per slot would serialise on the ticket, a chunk larger than the work per warp leaves warps without any).
// With one CTA per 8 slots, a CTA held its shared memory until its slowest warp was done, so the warps of dead slots
// (beyond counts, not KEPT, listed: 16 % in the slide) and of small masks idled beside the large ones; the ticket
// also hands the work of CTAs that start late (the SM still holding region CTAs of another stream) to those already
// running.
constexpr int kV2Chunk = 16;
constexpr int kV2CtasPerSm = 6;
__global__ void __launch_bounds__(kV2Threads, kV2CtasPerSm) mask_upsample_pack2_kernel(
    const float* __restrict__ patches, const int4* __restrict__ krs, const int32_t* __restrict__ geom4,
    const int64_t* __restrict__ offsets, long long n_slots, int mh, int mw, float sxs, float sys,
    uint32_t* __restrict__ bits, long long capacity_words, int32_t* __restrict__ status,
    uint32_t* __restrict__ ticket, int chunk) {
  __shared__ __align__(16) UpWarpSmem S[kV2Warps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* P = S[warp].patch;
  for (;;) {
    uint32_t first = 0;
    if (lane == 0) first = atomicAdd(ticket, (uint32_t)chunk);
    first = __shfl_sync(0xffffffffu, first, 0);
    if ((long long)first >= n_slots) return;
    const long long last = min((long long)first + chunk, n_slots);
    for (long long slot = first; slot < last; ++slot) {
      const int4 kr = krs[slot];
      const int pw = kr.z - kr.x, ph = kr.w - kr.y;
      if (pw <= 0 || ph <= 0) continue;  // dead / empty / handed to the per-detection kernel
      const int4 wdw = reinterpret_cast<const int4*>(geom4)[slot];
      const long long off = offsets[slot];
      if (off + (long long)((wdw.z + 31) >> 5) * wdw.w > capacity_words) {
        if (lane == 0) atomicOr(status, HDY_STATUS_OVERFLOW);
        continue;
      }
      __syncwarp();  // the previous slot's upsample is done with P
      up_load_patch(P, patches + slot * (kPatchPitch * kPatchPitch), pw, ph, lane);
      __syncwarp();
      upsample_pack_v2(P, S[warp].colT, kr, wdw, off, bits, mh, mw, sxs, sys, lane);
    }
  }
}

// CTAs of mask_upsample_pack2_kernel that are resident at once on this device (0 on error)
static int upsample_pack2_grid() {
  int dev = 0, sms = 0, per_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      cudaFuncSetAttribute((const void*)mask_upsample_pack2_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                           cudaSharedmemCarveoutMaxShared) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mask_upsample_pack2_kernel, kV2Threads, 0) != cudaSuccess)
    return 0;
  return sms * per_sm;
}

int launch_process_mask_regions(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                                const int32_t* counts,
                                int bs, int max_det, int nm, int mh, int mw, int ih, int iw, int upsample, float rx,
                                float ry, float* out_dense, const int32_t* geom, const int64_t* offsets, uint32_t* bits,
                                long long capacity_words, int32_t* status, void* workspace, size_t workspace_bytes,
                                cudaStream_t stream) {
  const long long slots = (long long)bs * max_det;
  if (!workspace || workspace_bytes < process_mask_workspace_bytes(bs, max_det)) return 1;
  const bool half = proto_dtype == HDY_F16;
  const int esz = half ? 2 : 4;
  // TMA: the global address and every stride are multiples of 16 bytes; a tile origin too (24 pixels: 96 / 48 bytes)
  if (nm != kRegNm || (mw * esz & 15) != 0 || ((uintptr_t)protos & 15) != 0 || max_det > 65535) return 1;
  // the packed + upsampled kernels read the windows hdy_process_mask_geometry wrote; without them the per-detection
  // kernel recomputes the windows
  const bool packed = out_dense == nullptr;
  if (packed && upsample && !geom) return 1;
  const int rxn = (mw + kRegBoxX - 1) / kRegBoxX, ryn = (mh + kRegBoxY - 1) / kRegBoxY;
  if ((long long)bs * rxn * ryn >= (1ll << 31) || slots >= (1ll << 31) || rxn * ryn > kMaxRegionsPerTile) return 1;
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return 1;
  CUtensorMap map;
  const cuuint64_t dims[4] = {(cuuint64_t)mw, (cuuint64_t)mh, (cuuint64_t)nm, (cuuint64_t)bs};
  const cuuint64_t strides[3] = {(cuuint64_t)mw * esz, (cuuint64_t)mw * mh * esz, (cuuint64_t)mw * mh * nm * esz};
  const cuuint32_t box[4] = {kRegBoxX, kRegBoxY, kRegNm, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = enc(&map, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                         const_cast<void*>(protos), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return 1;
  const PmWorkspace W = pm_workspace(workspace, slots);
  cudaError_t e = cudaMemsetAsync(W.large_count, 0, 8, stream);  // large_count and ticket
  if (e == cudaSuccess) e = cudaMemsetAsync(W.regions, 0, (size_t)bs * rxn * ryn * sizeof(RegionList), stream);
  if (e == cudaSuccess)
    e = half ? cudaFuncSetAttribute(proto_patch_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(RegSmemT<__half>))
             : cudaFuncSetAttribute(proto_patch_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(RegSmemT<float>));
  if (e != cudaSuccess) {
    set_error("process_mask(regions) setup: %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  const float4* b4 = reinterpret_cast<const float4*>(boxes);
  if (packed && upsample) {
    // bit-packed + upsampled (the throughput form): binning, the listed detections' words cleared (their tiles OR into
    // them), regions -> patches with the listed detections riding in the same launch, then upsample_pack_v2
    const float sxs = (float)mw / (float)iw, sys = (float)mh / (float)ih;  // ATen: scale = in / out (fp32)
    proto_bin_fused_kernel<<<(unsigned)((slots + 255) / 256), 256, 0, stream>>>(
        b4, counts, slots, max_det, mh, mw, rxn, ryn, rx, ry, geom, W.regions, W.kr, W.large_count, W.large_list);
    pm_clear_listed_kernel<<<148, 256, 0, stream>>>(geom, offsets, bits, capacity_words, W.large_list, W.large_count);
    ListedRide LR;
    LR.protos = protos, LR.boxes = b4, LR.offsets = offsets, LR.bits = bits, LR.status = status;
    LR.list = W.large_list, LR.list_count = W.large_count, LR.capacity_words = capacity_words;
    LR.rx = rx, LR.ry = ry, LR.nm = nm, LR.mh = mh, LR.mw = mw, LR.ih = ih, LR.iw = iw;
    LR.ctas = kListedTiles * 9;
    const unsigned g1 = (unsigned)((long long)bs * rxn * ryn + LR.ctas);
    if (half)
      proto_patch_kernel<__half><<<g1, kRegThreads, sizeof(RegSmemT<__half>), stream>>>(
          map, coef, W.kr, counts, max_det, rxn, ryn, W.patches, W.regions, LR);
    else
      proto_patch_kernel<float><<<g1, kRegThreads, sizeof(RegSmemT<float>), stream>>>(
          map, coef, W.kr, counts, max_det, rxn, ryn, W.patches, W.regions, LR);
    const int g2 = upsample_pack2_grid();
    if (g2 <= 0) {
      set_error("process_mask(packed): no occupancy for mask_upsample_pack2_kernel");
      return HDY_ERR_CUDA;
    }
    const int chunk = (int)std::min<long long>(kV2Chunk, std::max<long long>(1, slots / (4ll * g2 * kV2Warps)));
    mask_upsample_pack2_kernel<<<(unsigned)min((long long)g2, (slots + kV2Warps - 1) / kV2Warps), kV2Threads, 0,
                                 stream>>>(W.patches, W.kr, geom, offsets, slots, mh, mw, sxs, sys, bits, capacity_words,
                                           status, W.ticket, chunk);
    return check_launch("hdy_process_mask(packed)");
  }
  ListedRide no_ride;
  memset(&no_ride, 0, sizeof(no_ride));
  proto_bin_kernel<<<(unsigned)((slots + 255) / 256), 256, 0, stream>>>(b4, counts, slots, max_det, mh, mw, rxn, ryn, rx,
                                                                        ry, geom, W.regions, W.kr);
  if (half)
    proto_patch_kernel<__half><<<(unsigned)((long long)bs * rxn * ryn), kRegThreads, sizeof(RegSmemT<__half>), stream>>>(
        map, coef, W.kr, counts, max_det, rxn, ryn, W.patches, W.regions, no_ride);
  else
    proto_patch_kernel<float><<<(unsigned)((long long)bs * rxn * ryn), kRegThreads, sizeof(RegSmemT<float>), stream>>>(
        map, coef, W.kr, counts, max_det, rxn, ryn, W.patches, W.regions, no_ride);
  const unsigned g2 = (unsigned)((slots + kUpWarps - 1) / kUpWarps);
#define HDY_UP(P, U)                                                                                              \
  mask_upsample_pack_kernel<P, U><<<g2, kUpWarps * 32, 0, stream>>>(W.patches, b4, counts, slots, max_det, mh, mw, \
                                                                    ih, iw, rx, ry, out_dense, geom, offsets, bits, \
                                                                    capacity_words, status, W.large_count,         \
                                                                    W.large_list)
  if (packed)
    HDY_UP(true, false);
  else if (upsample)
    HDY_UP(false, true);
  else
    HDY_UP(false, false);
#undef HDY_UP
  int rc = check_launch("hdy_process_mask(regions)");
  if (rc) return rc;
  return launch_process_mask_listed(protos, proto_dtype, coef, boxes, counts, max_det, nm, mh, mw, ih, iw, upsample, rx, ry,
                                    out_dense, offsets, bits, capacity_words, status, W.large_list, W.large_count,
                                    stream);
}

}  // namespace hdy
