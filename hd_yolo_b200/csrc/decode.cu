// Grid+anchor decode and the fused decode + confidence filter + stream compaction.
//
// Reference arithmetic (all fp32, evaluated left to right, no FMA contraction):
//   y  = sigmoid(x)                                   yolo_head.py:189
//   xy = (y[0:2]*2 - 0.5 + grid) * stride             yolo_head.py:203,208
//   wh = (y[2:4]*2)**2 * anchor_grid                  yolo_head.py:204,209
//   x1 = cx - w/2 ... y2 = cy + h/2                   utils_general.py:121-128
//   keep (x2-x1)>=min_size & (y2-y1)>=min_size        utils_general.py:332 (torchvision remove_small_boxes)
//   keep obj > conf_thres                             utils_general.py:336-337
//
// HBM layout: a tile's level is a contiguous run of rows*no floats ([bs,na,ny,nx,no]).  One CTA
// stages ROWS_PER_CHUNK rows through shared memory with coalesced 128-bit streaming loads, one
// thread then owns one row.  Only sigmoid(obj) is evaluated for every row; the other channels are
// decoded for survivors alone.  Survivors are appended to the tile's candidate list with one
// atomicAdd per CTA (warp ballot + block prefix); the list is unordered, the 64-bit key carries the
// row index so that the NMS kernel's sort restores the reference's order exactly.
#include <math.h>
#include "hdy_common.cuh"

namespace hdy {

constexpr int kRowsPerChunk = 256;
constexpr int kThreads = 256;

__device__ __forceinline__ const LevelDev& find_level(const LevelTable& T, int chunk, int& l_out) {
  int l = 0;
#pragma unroll 1
  for (int i = 1; i < T.nl; ++i)
    if (chunk >= T.lv[i].chunk_begin) l = i;
  l_out = l;
  return T.lv[l];
}

// Coalesced copy of F floats from global g to shared s_al (whose 16-byte phase equals g's).
__device__ __forceinline__ void stage_rows(const float* __restrict__ g, float* s, int F) {
  const int tid = threadIdx.x;
  int head = (int)((4 - (((uintptr_t)g >> 2) & 3)) & 3);
  if (head > F) head = F;
  if (tid < head) s[tid] = ldg_stream_f(g + tid);
  const int nvec = (F - head) >> 2;
  const float4* g4 = reinterpret_cast<const float4*>(g + head);
  float4* s4 = reinterpret_cast<float4*>(s + head);
  for (int v0 = tid; v0 < nvec; v0 += kThreads * 4) {
    float4 r[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (v0 + k * kThreads < nvec) r[k] = ldg_stream_f4(g4 + v0 + k * kThreads);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (v0 + k * kThreads < nvec) s4[v0 + k * kThreads] = r[k];
  }
  const int done = head + (nvec << 2);
  if (tid < F - done) s[done + tid] = ldg_stream_f(g + done + tid);
}

struct Decoded {
  float cx, cy, w, h;
};

__device__ __forceinline__ Decoded decode_box(float l0, float l1, float l2, float l3, float gx, float gy,
                                              float stride, float aw, float ah) {
  Decoded d;
  float sx = sigmoidf_ref(l0), sy = sigmoidf_ref(l1), sw = sigmoidf_ref(l2), sh = sigmoidf_ref(l3);
  d.cx = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sx, 2.0f), 0.5f), gx), stride);
  d.cy = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sy, 2.0f), 0.5f), gy), stride);
  float tw = __fmul_rn(sw, 2.0f), th = __fmul_rn(sh, 2.0f);
  d.w = __fmul_rn(__fmul_rn(tw, tw), aw);
  d.h = __fmul_rn(__fmul_rn(th, th), ah);
  return d;
}

__device__ __forceinline__ float4 xywh_to_xyxy(float cx, float cy, float w, float h) {
  float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);  // w/2 is exact
  return make_float4(__fsub_rn(cx, hw), __fsub_rn(cy, hh), __fadd_rn(cx, hw), __fadd_rn(cy, hh));
}

// Block-wide append of per-thread candidates (0 or 1 each) to the tile's list.
__device__ __forceinline__ int block_append_pos(bool cand, int32_t* tile_count) {
  __shared__ int warp_cnt[kThreads / 32];
  __shared__ int block_base;
  const unsigned m = __ballot_sync(0xffffffffu, cand);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warp_cnt[warp] = __popc(m);
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
      int c = warp_cnt[w];
      warp_cnt[w] = tot;
      tot += c;
    }
    block_base = tot ? atomicAdd(tile_count, tot) : 0;
  }
  __syncthreads();
  return block_base + warp_cnt[warp] + __popc(m & ((1u << lane) - 1u));
}

// ------------------------------------------------------------------------------------------------
// Fused decode + filter + compact from raw logits.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) filter_compact_logits_kernel(
    const __grid_constant__ LevelTable T, float conf_thres, float min_size, int cap,
    uint64_t* __restrict__ cand_keys, float4* __restrict__ cand_boxes, int32_t* __restrict__ counts,
    int32_t* __restrict__ status) {
  extern __shared__ __align__(16) float smem[];
  const int tile = blockIdx.x / T.chunks_per_tile;
  const int chunk = blockIdx.x - tile * T.chunks_per_tile;
  int l;
  const LevelDev& L = find_level(T, chunk, l);
  const int row0 = (chunk - L.chunk_begin) * kRowsPerChunk;
  const int rows = min(kRowsPerChunk, L.rows - row0);
  const int no = T.no;
  const int t = threadIdx.x;
  const int plane = L.ny * L.nx;

  bool cand = false;
  float p_obj = 0.f;
  float4 box = make_float4(0.f, 0.f, 0.f, 0.f);

  if (T.layout == 0) {
    const float* g = L.ptr + ((size_t)tile * L.rows + row0) * no;
    float* s = smem + (((uintptr_t)g >> 2) & 3);
    stage_rows(g, s, rows * no);
    __syncthreads();
    if (t < rows) {
      const float* r = s + t * no;
      p_obj = sigmoidf_ref(r[4]);
      if (p_obj > conf_thres) {
        const int row = row0 + t;
        const int a = row / plane, p = row - a * plane;
        const int gy = p / L.nx, gx = p - gy * L.nx;
        Decoded d = decode_box(r[0], r[1], r[2], r[3], (float)gx, (float)gy, L.stride, L.aw[a], L.ah[a]);
        box = xywh_to_xyxy(d.cx, d.cy, d.w, d.h);
        cand = (__fsub_rn(box.z, box.x) >= min_size) && (__fsub_rn(box.w, box.y) >= min_size);
      }
    }
  } else {
    // planar [bs, na*no, ny, nx]: only the objectness plane is streamed; survivors gather the rest.
    if (t < rows) {
      const int row = row0 + t;
      const int a = row / plane, p = row - a * plane;
      const float* base = L.ptr + ((size_t)(tile * T.na + a) * no) * plane + p;
      p_obj = sigmoidf_ref(ldg_stream_f(base + (size_t)4 * plane));
      if (p_obj > conf_thres) {
        const int gy = p / L.nx, gx = p - gy * L.nx;
        Decoded d = decode_box(__ldg(base), __ldg(base + plane), __ldg(base + 2 * (size_t)plane),
                               __ldg(base + 3 * (size_t)plane), (float)gx, (float)gy, L.stride, L.aw[a],
                               L.ah[a]);
        box = xywh_to_xyxy(d.cx, d.cy, d.w, d.h);
        cand = (__fsub_rn(box.z, box.x) >= min_size) && (__fsub_rn(box.w, box.y) >= min_size);
      }
    }
  }

  const int pos = block_append_pos(cand, counts + tile);
  if (cand) {
    if (pos < cap) {
      const size_t o = (size_t)tile * cap + pos;
      cand_keys[o] = make_key(p_obj, (uint32_t)(L.row_offset + row0 + t));
      cand_boxes[o] = box;
    } else {
      atomicOr(status, HDY_STATUS_OVERFLOW);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Conv-native layout [bs, na*no, ny, nx] (layout 1, the yolo_head.py:141-145 permute skipped): the objectness logits of
// an (image, anchor) pair are ONE contiguous plane, so the filter streams 4 bytes per row instead of 4*no -- 6.5 MB
// instead of 266 MB per tiles640 batch with mask coefficients.  Every thread takes four consecutive rows with one
// 128-bit load, rejects on the logit, and survivors gather their four box logits from the neighbouring planes.
// ------------------------------------------------------------------------------------------------
constexpr int kPlanarRows = 4;
constexpr int kPlanarChunk = kThreads * kPlanarRows;

__global__ void __launch_bounds__(kThreads) filter_compact_planar_kernel(
    const __grid_constant__ LevelTable T, float t_lo, float conf_thres, float min_size, int cap,
    uint64_t* __restrict__ cand_keys, float4* __restrict__ cand_boxes, int32_t* __restrict__ counts,
    int32_t* __restrict__ status) {
  // phase A (all threads): four objectness logits each, rows that may pass go to a queue in shared memory;
  // phase B (the first q_n threads): sigmoid, box gather, decode, min-size, one global atomic per block.  Handling
  // survivors inline made 3 warps in 4 run the whole decode for one lane each and chained four global atomics per
  // warp behind two dependent loads (ncu: 32 us, 12 M warp instructions for 1.6 M rows).
  __shared__ int q_row[kPlanarChunk];
  __shared__ float q_x[kPlanarChunk];
  __shared__ int q_n;
  const int tile = blockIdx.x / T.chunks_per_tile;
  const int chunk = blockIdx.x - tile * T.chunks_per_tile;
  int l;
  const LevelDev& L = find_level(T, chunk, l);
  const int row0 = (chunk - L.chunk_begin) * kPlanarChunk + threadIdx.x * kPlanarRows;  // first of this thread's rows
  const int no = T.no, lane = threadIdx.x & 31;
  const int plane = L.ny * L.nx;
  if (threadIdx.x == 0) q_n = 0;
  float x[kPlanarRows];
  const bool vec = (plane & 3) == 0 && row0 + kPlanarRows <= L.rows;  // four rows of one plane, 16-byte aligned
  if (vec) {
    const int a = row0 / plane, p = row0 - a * plane;
    const float4 v = ldg_stream_f4(reinterpret_cast<const float4*>(
        L.ptr + ((size_t)(tile * T.na + a) * no + 4) * plane + p));
    x[0] = v.x, x[1] = v.y, x[2] = v.z, x[3] = v.w;
  } else {
#pragma unroll
    for (int k = 0; k < kPlanarRows; ++k) {
      const int r = row0 + k;
      x[k] = -3.0e38f;
      if (r < L.rows) {
        const int a = r / plane, p = r - a * plane;
        x[k] = ldg_stream_f(L.ptr + ((size_t)(tile * T.na + a) * no + 4) * plane + p);
      }
    }
  }
  __syncthreads();  // q_n = 0 is visible
#pragma unroll
  for (int k = 0; k < kPlanarRows; ++k) {
    const bool pass = x[k] >= t_lo;  // (false for the -3e38 padding)
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&q_n, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (pass) {
        const int i = base + __popc(m & ((1u << lane) - 1u));
        q_row[i] = row0 + k;
        q_x[i] = x[k];
      }
    }
  }
  __syncthreads();
  const int n = q_n;
  for (int i0 = 0; i0 < n; i0 += kThreads) {  // block-uniform trip count
    const int i = i0 + threadIdx.x;
    bool cand = false;
    float p_obj = 0.f;
    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = 0;
    if (i < n) {
      r = q_row[i];
      p_obj = sigmoidf_ref(q_x[i]);
      if (p_obj > conf_thres) {
        const int a = r / plane, p = r - a * plane;
        const int gy = p / L.nx, gx = p - gy * L.nx;
        const float* base = L.ptr + ((size_t)(tile * T.na + a) * no) * plane + p;
        Decoded d = decode_box(__ldg(base), __ldg(base + plane), __ldg(base + 2 * (size_t)plane),
                               __ldg(base + 3 * (size_t)plane), (float)gx, (float)gy, L.stride, L.aw[a], L.ah[a]);
        box = xywh_to_xyxy(d.cx, d.cy, d.w, d.h);
        cand = (__fsub_rn(box.z, box.x) >= min_size) && (__fsub_rn(box.w, box.y) >= min_size);
      }
    }
    const int pos = block_append_pos(cand, counts + tile);
    if (cand) {
      if (pos < cap) {
        const size_t o = (size_t)tile * cap + pos;
        cand_keys[o] = make_key(p_obj, (uint32_t)(L.row_offset + r));
        cand_boxes[o] = box;
      } else {
        atomicOr(status, HDY_STATUS_OVERFLOW);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Filter + compact from decoded rows (nms_per_image's input: cx,cy,w,h,obj,cls..,extra..).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) filter_compact_preds_kernel(
    const float* __restrict__ preds, int N, int row_len, int chunks_per_tile, float conf_thres,
    float min_size, int cap, uint64_t* __restrict__ cand_keys, float4* __restrict__ cand_boxes,
    int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) float smem[];
  const int tile = blockIdx.x / chunks_per_tile;
  const int chunk = blockIdx.x - tile * chunks_per_tile;
  const int row0 = chunk * kRowsPerChunk;
  const int rows = min(kRowsPerChunk, N - row0);
  const int t = threadIdx.x;
  const float* g = preds + ((size_t)tile * N + row0) * row_len;
  float* s = smem + (((uintptr_t)g >> 2) & 3);
  stage_rows(g, s, rows * row_len);
  __syncthreads();
  bool cand = false;
  float p_obj = 0.f;
  float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
  if (t < rows) {
    const float* r = s + t * row_len;
    p_obj = r[4];
    box = xywh_to_xyxy(r[0], r[1], r[2], r[3]);
    cand = (__fsub_rn(box.z, box.x) >= min_size) && (__fsub_rn(box.w, box.y) >= min_size) &&
           (p_obj > conf_thres);
  }
  const int pos = block_append_pos(cand, counts + tile);
  if (cand) {
    if (pos < cap) {
      const size_t o = (size_t)tile * cap + pos;
      cand_keys[o] = make_key(p_obj, (uint32_t)(row0 + t));
      cand_boxes[o] = box;
    } else {
      atomicOr(status, HDY_STATUS_OVERFLOW);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Front half of non_max_suppression (utils_general.py:439-491).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) filter_compact_yolo_kernel(
    const float* __restrict__ pred, int N, int nc, int chunks_per_tile, float conf_thres, int multi_label,
    const uint8_t* __restrict__ class_mask, int cap, uint64_t* __restrict__ cand_keys,
    float4* __restrict__ cand_boxes, float* __restrict__ cand_cls, int32_t* __restrict__ counts,
    int32_t* __restrict__ status) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int warp_cnt[kThreads / 32];
  __shared__ int block_base;
  const int row_len = 5 + nc;
  const int tile = blockIdx.x / chunks_per_tile;
  const int chunk = blockIdx.x - tile * chunks_per_tile;
  const int row0 = chunk * kRowsPerChunk;
  const int rows = min(kRowsPerChunk, N - row0);
  const int t = threadIdx.x;
  const float* g = pred + ((size_t)tile * N + row0) * row_len;
  float* s = smem + (((uintptr_t)g >> 2) & 3);
  stage_rows(g, s, rows * row_len);
  __syncthreads();

  // how many candidates this row produces
  int mine = 0;
  float obj = 0.f;
  int best = 0;
  float best_conf = 0.f;
  const float* r = s + t * row_len;
  if (t < rows) {
    obj = r[4];
    if (obj > conf_thres) {  // xc = prediction[..., 4] > conf_thres          :439
      if (multi_label) {
        for (int c = 0; c < nc; ++c) {
          float conf = __fmul_rn(r[5 + c], obj);  // x[:, 5:] *= x[:, 4:5]      :476
          if (conf > conf_thres && (!class_mask || class_mask[c])) ++mine;
        }
      } else {
        best_conf = __fmul_rn(r[5], obj);
        for (int c = 1; c < nc; ++c) {  // max(1): first maximal value wins     :486
          float conf = __fmul_rn(r[5 + c], obj);
          if (conf > best_conf) {
            best_conf = conf;
            best = c;
          }
        }
        if (best_conf > conf_thres && (!class_mask || class_mask[best])) mine = 1;
      }
    }
  }
  // block exclusive scan of `mine`
  const int lane = t & 31, warp = t >> 5;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_cnt[warp] = incl;
  __syncthreads();
  if (t == 0) {
    int tot = 0;
    for (int w = 0; w < kThreads / 32; ++w) {
      int c = warp_cnt[w];
      warp_cnt[w] = tot;
      tot += c;
    }
    block_base = tot ? atomicAdd(counts + tile, tot) : 0;
  }
  __syncthreads();
  if (mine) {
    int pos = block_base + warp_cnt[warp] + incl - mine;
    const float4 box = xywh_to_xyxy(r[0], r[1], r[2], r[3]);
    const uint32_t row = (uint32_t)(row0 + t);
    if (multi_label) {
      for (int c = 0; c < nc; ++c) {
        float conf = __fmul_rn(r[5 + c], obj);
        if (conf > conf_thres && (!class_mask || class_mask[c])) {
          if (pos < cap) {
            const size_t o = (size_t)tile * cap + pos;
            cand_keys[o] = make_key(conf, row * (uint32_t)nc + (uint32_t)c);
            cand_boxes[o] = box;
            cand_cls[o] = (float)c;
          } else {
            atomicOr(status, HDY_STATUS_OVERFLOW);
          }
          ++pos;
        }
      }
    } else {
      if (pos < cap) {
        const size_t o = (size_t)tile * cap + pos;
        cand_keys[o] = make_key(best_conf, row);
        cand_boxes[o] = box;
        cand_cls[o] = (float)best;
      } else {
        atomicOr(status, HDY_STATUS_OVERFLOW);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Full decode (compute_proposals parity) and decode + level column + concat.
// Flat element-wise kernels: element e of a tile's level -> (row, channel).
// ------------------------------------------------------------------------------------------------
template <bool CONCAT>
__global__ void __launch_bounds__(kThreads) decode_kernel(const __grid_constant__ LevelTable T, int level,
                                                           float* __restrict__ out, int bs) {
  // one CTA = kRowsPerChunk rows of one (tile, level); staged through smem so that both the
  // read and the write side are coalesced even when no (or no+1) is odd.
  extern __shared__ __align__(16) float smem[];
  const LevelDev& L = T.lv[level];
  const int chunks = (L.rows + kRowsPerChunk - 1) / kRowsPerChunk;
  const int tile = blockIdx.x / chunks;
  const int chunk = blockIdx.x - tile * chunks;
  const int row0 = chunk * kRowsPerChunk;
  const int rows = min(kRowsPerChunk, L.rows - row0);
  const int no = T.no;
  const int plane = L.ny * L.nx;
  const int t = threadIdx.x;
  float* s = smem + 4;  // data region (phase-adjusted below)
  if (T.layout == 0 && T.dtype == HDY_F16) {
    const size_t e0 = ((size_t)tile * L.rows + row0) * no;
    for (int e = t; e < rows * no; e += kThreads) s[e] = level_elem<true>(L.ptr, e0 + e);
  } else if (T.layout == 0) {
    const float* g = L.ptr + ((size_t)tile * L.rows + row0) * no;
    s = smem + (((uintptr_t)g >> 2) & 3);
    stage_rows(g, s, rows * no);
  } else {
    // planar source: gather channel planes into row-major smem
    for (int e = t; e < rows * no; e += kThreads) {
      const int c = e / rows, rr = e - c * rows;
      const int row = row0 + rr;
      const int a = row / plane, p = row - a * plane;
      s[rr * no + c] = ldg_stream_f(L.ptr + ((size_t)(tile * T.na + a) * no + c) * plane + p);
    }
  }
  __syncthreads();
  // element-wise transform in place
  for (int e = t; e < rows * no; e += kThreads) {
    const int rr = e / no, c = e - rr * no;
    float y = sigmoidf_ref(s[e]);
    if (c < 4) {
      const int row = row0 + rr;
      const int a = row / plane, p = row - a * plane;
      const int gy = p / L.nx, gx = p - gy * L.nx;
      if (c < 2) {
        float gv = (c == 0) ? (float)gx : (float)gy;
        y = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(y, 2.0f), 0.5f), gv), L.stride);
      } else {
        float av = (c == 2) ? L.aw[a] : L.ah[a];
        float tw = __fmul_rn(y, 2.0f);
        y = __fmul_rn(__fmul_rn(tw, tw), av);
      }
    }
    s[e] = y;
  }
  __syncthreads();
  if (CONCAT) {
    const int no1 = no + 1;
    float* o = out + ((size_t)tile * T.N + L.row_offset + row0) * no1;
    const float lvl = (float)level;
    for (int e = t; e < rows * no1; e += kThreads) {
      const int rr = e / no1, c = e - rr * no1;
      o[e] = (c == no) ? lvl : s[rr * no + c];
    }
  } else {
    float* o = out + ((size_t)tile * L.rows + row0) * no;
    for (int e = t; e < rows * no; e += kThreads) o[e] = s[e];
  }
}

static size_t stage_smem_bytes(int row_len) { return ((size_t)kRowsPerChunk * row_len + 8) * sizeof(float); }

template <typename K>
static int ensure_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    if (bytes > 227 * 1024) {
      set_error("row length too large for shared-memory staging (%zu bytes)", bytes);
      return HDY_ERR_INVALID;
    }
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return HDY_ERR_CUDA;
    }
  }
  return HDY_OK;
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_decode_levels(const hdy_level_t* levels_host, int nl, int bs, int na, int no,
                      float* const* out_host, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && out_host != nullptr, "hdy_decode_levels: bad arguments");
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, 0, kRowsPerChunk, &T);
  if (rc) return rc;
  T.nc = no - 5;
  if (bs == 0) return HDY_OK;
  const size_t smem = stage_smem_bytes(no);
  rc = ensure_smem(decode_kernel<false>, smem);
  if (rc) return rc;
  for (int l = 0; l < nl; ++l) {
    HDY_REQUIRE(out_host[l] != nullptr, "out[%d] is NULL", l);
    const int chunks = (T.lv[l].rows + kRowsPerChunk - 1) / kRowsPerChunk;
    decode_kernel<false><<<(unsigned)((size_t)bs * chunks), kThreads, smem, (cudaStream_t)stream>>>(
        T, l, out_host[l], bs);
  }
  return check_launch("hdy_decode_levels");
}

int hdy_decode_concat(const hdy_level_t* levels_host, int nl, int bs, int na, int no, int layout, float* out,
                      hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && out != nullptr, "hdy_decode_concat: bad arguments");
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, layout, kRowsPerChunk, &T);
  if (rc) return rc;
  T.nc = no - 5;
  if (bs == 0) return HDY_OK;
  const size_t smem = stage_smem_bytes(no);
  rc = ensure_smem(decode_kernel<true>, smem);
  if (rc) return rc;
  for (int l = 0; l < nl; ++l) {
    const int chunks = (T.lv[l].rows + kRowsPerChunk - 1) / kRowsPerChunk;
    decode_kernel<true><<<(unsigned)((size_t)bs * chunks), kThreads, smem, (cudaStream_t)stream>>>(T, l, out,
                                                                                                  bs);
  }
  return check_launch("hdy_decode_concat");
}

int hdy_filter_compact_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no,
                              int layout, float conf_thres, float min_size, int cap, uint64_t* cand_keys,
                              float* cand_boxes, int32_t* counts, int32_t* status, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && cap > 0, "hdy_filter_compact_logits: bs=%d cap=%d", bs, cap);
  HDY_REQUIRE(nc >= 0 && no >= 5 + nc, "no=%d must be >= 5+nc (nc=%d)", no, nc);
  HDY_REQUIRE(cand_keys && cand_boxes && counts && status, "hdy_filter_compact_logits: NULL output");
  HDY_REQUIRE(((uintptr_t)cand_boxes & 15) == 0, "cand_boxes must be 16-byte aligned");
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, layout, kRowsPerChunk, &T);
  if (rc) return rc;
  T.nc = nc;
  if (bs == 0) return HDY_OK;
  const bool conf_ok = conf_thres > 1e-6f && conf_thres < 1.0f - 1e-6f;
  if (layout == 1 && conf_ok) {
    bool aligned = true;
    for (int i = 0; i < nl; ++i) aligned = aligned && (((uintptr_t)levels_host[i].logits & 15) == 0);
    if (aligned) {
      LevelTable S;
      rc = build_level_table(levels_host, nl, na, no, 1, kPlanarChunk, &S);
      if (rc) return rc;
      S.nc = nc;
      const double lg = log((double)conf_thres / (1.0 - (double)conf_thres));
      const float t_lo = (float)(lg - 1e-4 * (1.0 + fabs(lg)));  // sigmoid(x) <= conf for certain below this logit
      const size_t nblk = (size_t)bs * S.chunks_per_tile;
      HDY_REQUIRE(nblk < (1ull << 31), "grid too large");
      filter_compact_planar_kernel<<<(unsigned)nblk, kThreads, 0, (cudaStream_t)stream>>>(
          S, t_lo, conf_thres, min_size, cap, cand_keys, reinterpret_cast<float4*>(cand_boxes), counts, status);
      return check_launch("hdy_filter_compact_logits(planar)");
    }
  }
  if (layout == 0) {  // TMA-staged persistent kernel whenever the chunks are 16-byte aligned
    rc = launch_filter_compact_tma(levels_host, nl, bs, na, nc, no, conf_thres, min_size, cap, cand_keys, cand_boxes,
                                   counts, status, (cudaStream_t)stream);
    if (rc != 1) return rc;
  }
  HDY_REQUIRE(T.dtype == HDY_F32, "fp16 logits need 16-byte aligned level tensors and 1e-6 < conf_thres < 1 - 1e-6 "
                                  "(the TMA-staged filter is the only fp16 reader)");
  const size_t smem = layout == 0 ? stage_smem_bytes(no) : 0;
  rc = ensure_smem(filter_compact_logits_kernel, smem);
  if (rc) return rc;
  const size_t blocks = (size_t)bs * T.chunks_per_tile;
  HDY_REQUIRE(blocks < (1ull << 31), "grid too large");
  filter_compact_logits_kernel<<<(unsigned)blocks, kThreads, smem, (cudaStream_t)stream>>>(
      T, conf_thres, min_size, cap, cand_keys, reinterpret_cast<float4*>(cand_boxes), counts, status);
  return check_launch("hdy_filter_compact_logits");
}

int hdy_filter_compact_preds(const float* preds, int bs, int N, int row_len, float conf_thres, float min_size,
                             int cap, uint64_t* cand_keys, float* cand_boxes, int32_t* counts, int32_t* status,
                             hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && N >= 0 && row_len >= 5 && cap > 0, "hdy_filter_compact_preds: bad sizes");
  HDY_REQUIRE(cand_keys && cand_boxes && counts && status, "hdy_filter_compact_preds: NULL output");
  HDY_REQUIRE(((uintptr_t)cand_boxes & 15) == 0, "cand_boxes must be 16-byte aligned");
  if (bs == 0 || N == 0) return HDY_OK;
  HDY_REQUIRE(preds != nullptr && ((uintptr_t)preds & 3) == 0, "preds NULL or misaligned");
  const size_t smem = stage_smem_bytes(row_len);
  int rc = ensure_smem(filter_compact_preds_kernel, smem);
  if (rc) return rc;
  const int chunks = (N + kRowsPerChunk - 1) / kRowsPerChunk;
  const size_t blocks = (size_t)bs * chunks;
  HDY_REQUIRE(blocks < (1ull << 31), "grid too large");
  filter_compact_preds_kernel<<<(unsigned)blocks, kThreads, smem, (cudaStream_t)stream>>>(
      preds, N, row_len, chunks, conf_thres, min_size, cap, cand_keys, reinterpret_cast<float4*>(cand_boxes),
      counts, status);
  return check_launch("hdy_filter_compact_preds");
}

int hdy_filter_compact_yolo(const float* prediction, int bs, int N, int nc, float conf_thres, int multi_label,
                            const uint8_t* class_mask, int cap, uint64_t* cand_keys, float* cand_boxes,
                            float* cand_cls, int32_t* counts, int32_t* status, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && N >= 0 && nc >= 1 && cap > 0, "hdy_filter_compact_yolo: bad sizes");
  HDY_REQUIRE(cand_keys && cand_boxes && cand_cls && counts && status, "hdy_filter_compact_yolo: NULL output");
  HDY_REQUIRE(((uintptr_t)cand_boxes & 15) == 0, "cand_boxes must be 16-byte aligned");
  HDY_REQUIRE((long long)N * nc < (1ll << 32), "N*nc overflows the 32-bit key index");
  if (bs == 0 || N == 0) return HDY_OK;
  HDY_REQUIRE(prediction != nullptr && ((uintptr_t)prediction & 3) == 0, "prediction NULL or misaligned");
  const size_t smem = stage_smem_bytes(5 + nc);
  int rc = ensure_smem(filter_compact_yolo_kernel, smem);
  if (rc) return rc;
  const int chunks = (N + kRowsPerChunk - 1) / kRowsPerChunk;
  const size_t blocks = (size_t)bs * chunks;
  HDY_REQUIRE(blocks < (1ull << 31), "grid too large");
  filter_compact_yolo_kernel<<<(unsigned)blocks, kThreads, smem, (cudaStream_t)stream>>>(
      prediction, N, nc, chunks, conf_thres, multi_label, class_mask, cap, cand_keys,
      reinterpret_cast<float4*>(cand_boxes), cand_cls, counts, status);
  return check_launch("hdy_filter_compact_yolo");
}

}  // extern "C"
