// Per-tile greedy IoU NMS for tiles with more than kNmsSmemCap (4 096) candidates, exact torchvision.ops.nms
// semantics, one CTA per tile; smaller tiles are done by nms_tiles_smem_kernel (nms_smem.cu).
//
// torchvision's kernel builds a dense n x n/64 suppression bitmask in HBM and walks it
// sequentially.  Nuclei are small boxes on a large tile, so almost every pair is disjoint; this
// kernel never forms the matrix.  Per tile, on a global-memory workspace (hdy_nms_workspace_bytes):
//   1. bitonic sort of (key, slot) pairs; ascending key == descending score, ties by lower index
//      (== scores.sort(stable, descending), the order torchvision visits boxes in);
//   2. boxes gathered into rank order; cell size c = 2 x mean box extent (block reduction);
//   3. counting sort of "small" boxes (w,h <= c) into a G x G torus grid by centre, "large"
//      boxes (and anything numerically awkward) into one extra bucket every box scans;
//   4. parallel greedy rounds: box r is KEPT once every higher-ranked box j with IoU(j,r) > thr
//      is SUPPRESSED, and SUPPRESSED as soon as one such j is KEPT.  Two small boxes can only
//      intersect if their centres are less than c apart, i.e. in adjacent cells, so each box looks
//      at 3x3 cells + the large bucket.  The fixed point equals sequential greedy NMS; the number
//      of rounds is the longest suppression chain (a handful for nuclei);
//   5. rank-ordered compaction of KEPT boxes, first max_det.
// The grid/cell choice only affects speed, never the result: the IoU test itself is exact
// (hdy_common.cuh: iou_gt) and is evaluated for every pair that can possibly intersect.
#include "hdy_common.cuh"

namespace hdy {

constexpr int kNmsThreads = 512;
constexpr int kGridGlobal = 64;  // torus grid side
constexpr float kCellMargin = 1.01f;
constexpr float kMaxScaled = 16384.0f;  // |centre|/cell above this -> "large" bucket (fp32 safety)

enum : uint8_t { ST_UNKNOWN = 0, ST_KEPT = 1, ST_SUPPRESSED = 2 };

// Optional phase profile of nms_tiles_smem_kernel (hdy_debug_nms_phases), passed to it as a kernel parameter
static unsigned long long* g_phase_host = nullptr;

__device__ __forceinline__ uint32_t next_pow2(uint32_t v) {
  if (v <= 1) return 1;
  return 1u << (32 - __clz(v - 1));
}

// exclusive scan of a[0..len) in place (ints); returns total.  All threads must call.
__device__ int block_excl_scan(int* a, int len, int* warp_tmp) {
  const int t = threadIdx.x, T = kNmsThreads;
  const int items = (len + T - 1) / T;
  const int b = min(t * items, len), e = min(b + items, len);
  int sum = 0;
  for (int i = b; i < e; ++i) sum += a[i];
  const int lane = t & 31, warp = t >> 5;
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tmp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = (lane < T / 32) ? warp_tmp[lane] : 0;
    int s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += u;
    }
    if (lane < T / 32) warp_tmp[lane] = s - v;  // exclusive warp offsets
    if (lane == T / 32 - 1) warp_tmp[T / 32] = s;  // total
  }
  __syncthreads();
  int run = warp_tmp[warp] + incl - sum;
  for (int i = b; i < e; ++i) {
    int v = a[i];
    a[i] = run;
    run += v;
  }
  const int total = warp_tmp[T / 32];
  __syncthreads();
  return total;
}

struct TileOut {
  int32_t* keep_idx;
  int32_t* keep_slot;
  float4* keep_box;
  float* keep_score;
  float* keep_cls;
  int32_t* keep_count;
  uint8_t* keep_frag;  // optional: 1 for every survivor (this path does not analyse the gray zone; conservative)
};

__device__ void nms_tile_body(const int n_in, const int max_nms, uint64_t* keys, uint32_t* slots, float4* boxes,
                              uint8_t* state, uint32_t* items, int* cell, int* warp_tmp, float* red_tmp,
                              const uint64_t* __restrict__ gkeys, const float4* __restrict__ gboxes,
                              const float* __restrict__ gcls, const float class_offset, const float thr,
                              const int max_det, const TileOut out) {
  const int t = threadIdx.x, T = kNmsThreads;
  const uint32_t P = next_pow2((uint32_t)n_in);
  // `elif n > max_nms: x = x[x[:, 4].argsort(descending=True)[:max_nms]]`  utils_general.py:501-502
  // (ties at the cut are resolved by lower index here; the reference's unstable argsort leaves
  //  them unspecified)
  const int n = (max_nms > 0 && n_in > max_nms) ? max_nms : n_in;
  constexpr int G = kGridGlobal;

  // ---- 1. load + bitonic sort ------------------------------------------------------------------
  for (uint32_t i = t; i < P; i += T) {
    keys[i] = (i < (uint32_t)n_in) ? gkeys[i] : ~0ull;
    slots[i] = i;
  }
  __syncthreads();
  for (uint32_t k = 2; k <= P; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t p = t; p < (P >> 1); p += T) {
        const uint32_t i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
        const uint32_t x = i | j;
        const bool up = ((i & k) == 0);
        const uint64_t a = keys[i], b = keys[x];
        if ((a > b) == up) {
          keys[i] = b;
          keys[x] = a;
          const uint32_t sa = slots[i];
          slots[i] = slots[x];
          slots[x] = sa;
        }
      }
      __syncthreads();
    }
  }

  // ---- 2. boxes into rank order (+ class offset), extent statistics ------------------------------
  float ext_sum = 0.f;
  int ext_cnt = 0;
  for (int r = t; r < n; r += T) {
    const uint32_t s = slots[r];
    float4 b = gboxes[s];
    if (gcls) {
      const float c = __fmul_rn(gcls[s], class_offset);  // c = x[:, 5:6] * max_wh   utils_general.py:505
      b.x = __fadd_rn(b.x, c);
      b.y = __fadd_rn(b.y, c);
      b.z = __fadd_rn(b.z, c);
      b.w = __fadd_rn(b.w, c);
    }
    boxes[r] = b;
    const float w = b.z - b.x, h = b.w - b.y;
    if (w > 0.f && h > 0.f && w < 3.0e38f && h < 3.0e38f) {
      ext_sum += fmaxf(w, h);
      ++ext_cnt;
    }
  }
  // block reduce (sum, count)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ext_sum += __shfl_xor_sync(0xffffffffu, ext_sum, o);
    ext_cnt += __shfl_xor_sync(0xffffffffu, ext_cnt, o);
  }
  __syncthreads();
  if ((t & 31) == 0) {
    red_tmp[t >> 5] = ext_sum;
    warp_tmp[t >> 5] = ext_cnt;
  }
  __syncthreads();
  float tot_sum = 0.f;
  int tot_cnt = 0;
  for (int w = 0; w < T / 32; ++w) {
    tot_sum += red_tmp[w];
    tot_cnt += warp_tmp[w];
  }
  __syncthreads();
  float cell_size = tot_cnt ? 2.0f * (tot_sum / (float)tot_cnt) : 1.0f;
  if (!(cell_size > 1e-20f) || !(cell_size < 1e30f)) cell_size = 1.0f;
  const float inv_cell = 1.0f / (cell_size * kCellMargin);
  const float max_center = cell_size * kMaxScaled;

  // classification: 0 = isolated (degenerate: can never intersect), 1 = small (binned), 2 = large
  auto classify = [&](const float4& b, int& bucket) -> int {
    const float w = b.z - b.x, h = b.w - b.y;
    if (w <= 0.f || h <= 0.f) return 0;
    const float cx = (b.x + b.z) * 0.5f, cy = (b.y + b.w) * 0.5f;
    if (w <= cell_size && h <= cell_size && fabsf(cx) <= max_center && fabsf(cy) <= max_center) {
      const int ix = (int)floorf(cx * inv_cell), iy = (int)floorf(cy * inv_cell);
      bucket = (ix & (G - 1)) + (iy & (G - 1)) * G;
      return 1;
    }
    bucket = G * G;
    return 2;  // also NaN / inf coordinates
  };

  // ---- 3. counting sort into the torus grid ------------------------------------------------------
  constexpr int NB = G * G + 1;
  for (int i = t; i < NB; i += T) cell[i] = 0;
  __syncthreads();
  for (int r = t; r < n; r += T) {
    int bucket = 0;
    const int cls = classify(boxes[r], bucket);
    state[r] = cls ? ST_UNKNOWN : ST_KEPT;
    if (cls) atomicAdd(&cell[bucket], 1);
  }
  __syncthreads();
  block_excl_scan(cell, NB, warp_tmp);
  for (int r = t; r < n; r += T) {
    int bucket = 0;
    if (classify(boxes[r], bucket)) items[atomicAdd(&cell[bucket], 1)] = (uint32_t)r;
  }
  __syncthreads();
  // now: bucket b occupies items[ (b ? cell[b-1] : 0) .. cell[b] )
  const int large_begin = cell[NB - 2], large_end = cell[NB - 1];

  // ---- 4. parallel greedy rounds -------------------------------------------------------------------
  volatile uint8_t* vstate = state;
  while (true) {
    int unknown = 0;
    for (int r = t; r < n; r += T) {
      if (vstate[r] != ST_UNKNOWN) continue;
      const float4 bi = boxes[r];
      int bucket = 0;
      const int cls = classify(bi, bucket);
      int decided = ST_KEPT;
      auto visit = [&](int j) -> bool {  // returns true when r is decided SUPPRESSED
        if (j < r && iou_gt(boxes[j], bi, thr)) {
          const uint8_t sj = vstate[j];
          if (sj == ST_KEPT) {
            decided = ST_SUPPRESSED;
            return true;
          }
          if (sj == ST_UNKNOWN) decided = ST_UNKNOWN;
        }
        return false;
      };
      bool done = false;
      if (cls == 1) {
        const float cx = (bi.x + bi.z) * 0.5f, cy = (bi.y + bi.w) * 0.5f;
        const int ix = (int)floorf(cx * inv_cell), iy = (int)floorf(cy * inv_cell);
#pragma unroll 1
        for (int dy = -1; dy <= 1 && !done; ++dy) {
          const int rowb = ((iy + dy) & (G - 1)) * G;
#pragma unroll 1
          for (int dx = -1; dx <= 1 && !done; ++dx) {
            const int b = ((ix + dx) & (G - 1)) + rowb;
            const int beg = b ? cell[b - 1] : 0, end = cell[b];
            for (int p = beg; p < end; ++p)
              if (visit((int)items[p])) {
                done = true;
                break;
              }
          }
        }
        for (int p = large_begin; p < large_end && !done; ++p) done = visit((int)items[p]);
      } else {
        // large box: every higher-ranked box is a potential dominator
        for (int j = 0; j < r && !done; ++j) done = visit(j);
      }
      if (decided != ST_UNKNOWN)
        vstate[r] = (uint8_t)decided;
      else
        unknown = 1;
    }
    if (!__syncthreads_or(unknown)) break;
  }

  // ---- 5. rank-ordered compaction of survivors ----------------------------------------------------
  {
    const int items_per = (n + T - 1) / T;
    const int b = min(t * items_per, n), e = min(b + items_per, n);
    int cnt = 0;
    for (int r = b; r < e; ++r) cnt += (state[r] == ST_KEPT);
    const int lane = t & 31, warp = t >> 5;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_tmp[warp] = incl;
    __syncthreads();
    int base = 0, total = 0;
    for (int w = 0; w < T / 32; ++w) {
      if (w < warp) base += warp_tmp[w];
      total += warp_tmp[w];
    }
    int pos = base + incl - cnt;
    for (int r = b; r < e && pos < max_det; ++r) {
      if (state[r] == ST_KEPT) {
        const uint32_t s = slots[r];
        const uint64_t k = gkeys[s];
        out.keep_idx[pos] = (int32_t)key_index(k);
        out.keep_slot[pos] = (int32_t)s;
        if (out.keep_box) out.keep_box[pos] = gboxes[s];
        if (out.keep_score) out.keep_score[pos] = key_score(k);
        if (out.keep_cls) out.keep_cls[pos] = gcls ? gcls[s] : 0.f;
        if (out.keep_frag) out.keep_frag[pos] = 1;
        ++pos;
      }
    }
    if (t == 0) *out.keep_count = min(total, max_det);
  }
}

struct WorkspaceLayout {
  size_t keys, slots, boxes, state, items, cell, per_tile;
  uint32_t P;
};

__host__ __device__ inline WorkspaceLayout workspace_layout(int cap) {
  WorkspaceLayout L;
  uint32_t P = 1;
  while (P < (uint32_t)cap) P <<= 1;
  L.P = P;
  size_t o = 0;
  L.keys = o;
  o += (size_t)P * 8;
  L.boxes = o;
  o += (size_t)P * 16;
  L.slots = o;
  o += (size_t)P * 4;
  L.items = o;
  o += (size_t)P * 4;
  L.cell = o;
  o += (size_t)(kGridGlobal * kGridGlobal + 4) * 4;
  L.state = o;
  o += (size_t)P;
  L.per_tile = (o + 255) & ~(size_t)255;
  return L;
}

__global__ void __launch_bounds__(kNmsThreads, 2) nms_tiles_kernel(
    const uint64_t* __restrict__ cand_keys, const float4* __restrict__ cand_boxes,
    const float* __restrict__ cand_cls, const int32_t* __restrict__ counts, int cap, float thr,
    float class_offset, int max_nms, int max_det, int32_t* __restrict__ keep_idx,
    int32_t* __restrict__ keep_slot, float4* __restrict__ keep_box, float* __restrict__ keep_score,
    float* __restrict__ keep_cls, int32_t* __restrict__ keep_counts, unsigned char* __restrict__ workspace,
    uint8_t* __restrict__ keep_fragile) {
  __shared__ int warp_tmp[kNmsThreads / 32 + 1];
  __shared__ float red_tmp[kNmsThreads / 32];
  const int tile = blockIdx.x;
  const int n = min(counts[tile], cap);
  if (n <= kNmsSmemCap) return;  // done by nms_tiles_smem_kernel
  TileOut out;
  out.keep_idx = keep_idx + (size_t)tile * max_det;
  out.keep_slot = keep_slot + (size_t)tile * max_det;
  out.keep_box = keep_box ? keep_box + (size_t)tile * max_det : nullptr;
  out.keep_score = keep_score ? keep_score + (size_t)tile * max_det : nullptr;
  out.keep_cls = keep_cls ? keep_cls + (size_t)tile * max_det : nullptr;
  out.keep_count = keep_counts + tile;
  out.keep_frag = keep_fragile ? keep_fragile + (size_t)tile * max_det : nullptr;
  const uint64_t* gk = cand_keys + (size_t)tile * cap;
  const float4* gb = cand_boxes + (size_t)tile * cap;
  const float* gc = cand_cls ? cand_cls + (size_t)tile * cap : nullptr;
  const WorkspaceLayout L = workspace_layout(cap);
  unsigned char* w = workspace + (size_t)tile * L.per_tile;
  nms_tile_body(n, max_nms, reinterpret_cast<uint64_t*>(w + L.keys), reinterpret_cast<uint32_t*>(w + L.slots),
                reinterpret_cast<float4*>(w + L.boxes), w + L.state, reinterpret_cast<uint32_t*>(w + L.items),
                reinterpret_cast<int*>(w + L.cell), warp_tmp, red_tmp, gk, gb, gc, class_offset, thr, max_det, out);
}

// ------------------------------------------------------------------------------------------------
// Epilogues
// ------------------------------------------------------------------------------------------------
__global__ void gather_preds_kernel(const float* __restrict__ preds, int N, int row_len, int nc,
                                    const int32_t* __restrict__ keep_idx,
                                    const int32_t* __restrict__ keep_counts, int max_det,
                                    float* __restrict__ out_scores, float* __restrict__ out_extra) {
  const int tile = blockIdx.y;
  const int k = keep_counts[tile];
  const int ns = 1 + nc, ne = row_len - 5 - nc;
  for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < k; d += gridDim.x * blockDim.x) {
    const float* r = preds + ((size_t)tile * N + keep_idx[(size_t)tile * max_det + d]) * row_len;
    float* os = out_scores + ((size_t)tile * max_det + d) * ns;
    for (int c = 0; c < ns; ++c) os[c] = r[4 + c];
    if (out_extra) {
      float* oe = out_extra + ((size_t)tile * max_det + d) * ne;
      for (int c = 0; c < ne; ++c) oe[c] = r[5 + nc + c];
    }
  }
}

__global__ void gather_logits_kernel(const __grid_constant__ LevelTable T,
                                     const int32_t* __restrict__ keep_idx,
                                     const int32_t* __restrict__ keep_counts, int max_det,
                                     float* __restrict__ out_scores, float* __restrict__ out_level,
                                     float* __restrict__ out_extra) {
  const int tile = blockIdx.y;
  const int k = keep_counts[tile];
  const int nc = T.nc, no = T.no, ns = 1 + nc, ne = no - 5 - nc;
  for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < k; d += gridDim.x * blockDim.x) {
    const int row = keep_idx[(size_t)tile * max_det + d];
    int l = 0;
    for (int i = 1; i < T.nl; ++i)
      if (row >= T.lv[i].row_offset) l = i;
    const LevelDev& L = T.lv[l];
    const int rr = row - L.row_offset;
    const size_t o = (size_t)tile * max_det + d;
    float* os = out_scores + o * ns;
    if (T.layout == 0 && T.dtype == HDY_F16) {
      const size_t e0 = ((size_t)tile * L.rows + rr) * no;
      for (int c = 0; c < ns; ++c) os[c] = sigmoidf_ref(level_elem<true>(L.ptr, e0 + 4 + c));
      if (out_extra)
        for (int c = 0; c < ne; ++c) out_extra[o * ne + c] = level_elem<true>(L.ptr, e0 + 5 + nc + c);
    } else if (T.layout == 0) {
      const float* r = L.ptr + ((size_t)tile * L.rows + rr) * no;
      for (int c = 0; c < ns; ++c) os[c] = sigmoidf_ref(r[4 + c]);
      if (out_extra)
        for (int c = 0; c < ne; ++c) out_extra[o * ne + c] = r[5 + nc + c];
    } else {
      const int plane = L.ny * L.nx;
      const int a = rr / plane, p = rr - a * plane;
      const float* r = L.ptr + ((size_t)(tile * T.na + a) * no) * plane + p;
      for (int c = 0; c < ns; ++c) os[c] = sigmoidf_ref(r[(size_t)(4 + c) * plane]);
      if (out_extra)
        for (int c = 0; c < ne; ++c) out_extra[o * ne + c] = r[(size_t)(5 + nc + c) * plane];
    }
    if (out_level) out_level[o] = (float)l;
  }
}

__global__ void make_keys_kernel(const float* __restrict__ scores, size_t n, int seg_len,
                                 uint64_t* __restrict__ keys) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = make_key(scores[i], (uint32_t)(i % (size_t)seg_len));
}

struct HierOps {
  int n;
  int8_t dst[2 * HDY_MAX_SCORES], src[2 * HDY_MAX_SCORES];
};

__global__ void select_scores_kernel(float* __restrict__ scores, const int32_t* __restrict__ keep_counts,
                                     int max_det, int nc, const __grid_constant__ HierOps H, float conf_thres,
                                     float* __restrict__ out_score, int64_t* __restrict__ out_label) {
  const int tile = blockIdx.y;
  const int k = keep_counts[tile];
  const int ns = 1 + nc;
  for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < k; d += gridDim.x * blockDim.x) {
    const size_t o = (size_t)tile * max_det + d;
    float* s = scores + o * ns;
    // hierarchical_scores: x[:, v] *= x[:, k]  (yolo_head.py:476-477), applied in dict order
    for (int i = 0; i < H.n; ++i) s[H.dst[i]] = __fmul_rn(s[H.dst[i]], s[H.src[i]]);
    // cls_scores, cls_labels = scores[..., 1:].max(1)   (first maximal value)      :342
    float best = s[1];
    int arg = 0;
    for (int c = 1; c < nc; ++c)
      if (s[1 + c] > best) {
        best = s[1 + c];
        arg = c;
      }
    const bool cls_ok = best > conf_thres;
    if (out_score) out_score[o] = cls_ok ? best : s[0];
    if (out_label) out_label[o] = cls_ok ? (int64_t)(arg + 1) : (int64_t)-100;
  }
}

// Fused gather + S1 for the survivors of the fused head path: ONE WARP per survivor.  Lane c reads channel 4 + c of
// the survivor's row (one coalesced 128-byte request for obj + classes + the first extra channels), lanes < 1 + nc
// apply the sigmoid, hierarchical_scores runs as shuffles (yolo_head.py:473-479), the (score, label) select of
// :336-345 as a shuffle scan, and the raw extra channels (mask coefficients) are written with coalesced stores.
// Replaces gather_logits_kernel + select_scores_kernel (one thread per survivor walking 37 strided floats each).
// G lanes per survivor (G = 8, 16 or 32 >= 1 + nc), 32 / G survivors per warp: one sigmoid evaluation, one round of
// hierarchical-score shuffles and one select scan serve all of the warp's survivors, and their scattered row loads
// are in flight together.
template <bool HALF>
__device__ __forceinline__ float row_elem(const unsigned char* rp, size_t j) {
  if (HALF) return __half2float(*reinterpret_cast<const __half*>(rp + j * 2));
  return __ldg(reinterpret_cast<const float*>(rp + j * 4));
}

template <int G, bool HALF>
__global__ void __launch_bounds__(256) gather_select_logits_kernel(
    const __grid_constant__ LevelTable T, const int32_t* __restrict__ keep_idx,
    const int32_t* __restrict__ keep_counts, int max_det, const __grid_constant__ HierOps H, float conf_thres,
    float* __restrict__ out_scores, float* __restrict__ out_level, float* __restrict__ out_extra,
    float* __restrict__ out_score, int64_t* __restrict__ out_label) {
  constexpr int SPW = 32 / G;
  const int tile = blockIdx.y;
  const int lane = threadIdx.x & 31, grp = lane / G, g = lane - grp * G;
  const int d0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * SPW;
  const int k = min(keep_counts[tile], max_det);
  if (d0 >= k) return;
  const int nc = T.nc, no = T.no, ns = 1 + nc, ne = no - 5 - nc;
  const int d = min(d0 + grp, k - 1);
  const bool live = d0 + grp < k;
  const size_t o = (size_t)tile * max_det + d;
  const int row = keep_idx[o];
  int l = 0;
  for (int i = 1; i < T.nl; ++i)
    if (row >= T.lv[i].row_offset) l = i;
  const LevelDev& L = T.lv[l];
  const int rr = row - L.row_offset;
  constexpr int kEsz = HALF ? 2 : 4;
  const unsigned char* rp;  // first element of the survivor's row (fp16 rows exist in layout 0 only)
  int cs = 1;
  if (T.layout == 0) {
    rp = reinterpret_cast<const unsigned char*>(L.ptr) + ((size_t)tile * L.rows + rr) * no * kEsz;
  } else {
    const int plane = L.ny * L.nx;
    const int a = rr / plane, p = rr - a * plane;
    rp = reinterpret_cast<const unsigned char*>(L.ptr + ((size_t)(tile * T.na + a) * no) * plane + p);
    cs = plane;
  }
  float sc = g < ns ? sigmoidf_ref(row_elem<HALF>(rp, (size_t)(4 + g) * cs)) : 0.f;
  // hierarchical_scores: x[:, dst] *= x[:, src], in order
  for (int i = 0; i < H.n; ++i) {
    const float vs = __shfl_sync(0xffffffffu, sc, H.src[i], G);
    if (g == H.dst[i]) sc = __fmul_rn(sc, vs);
  }
  if (live && g < ns) out_scores[o * ns + g] = sc;
  // cls_scores, cls_labels = scores[..., 1:].max(1)   (first maximal value)
  float best = __shfl_sync(0xffffffffu, sc, 1, G);
  int arg = 0;
  for (int c = 1; c < nc; ++c) {
    const float v = __shfl_sync(0xffffffffu, sc, 1 + c, G);
    if (v > best) {
      best = v;
      arg = c;
    }
  }
  if (live && g == 0) {
    const bool cls_ok = best > conf_thres;
    if (out_score) out_score[o] = cls_ok ? best : sc;
    if (out_label) out_label[o] = cls_ok ? (int64_t)(arg + 1) : (int64_t)-100;
    if (out_level) out_level[o] = (float)l;
  }
  // raw extra channels (mask coefficients): the whole warp copies one survivor's run at a time, coalesced
  if (out_extra && ne > 0 && ne <= 32) {
    // all of the warp's survivors at once: SPW scattered loads per lane are in flight together (one round trip to L2 /
    // HBM instead of SPW; in the conv-native layout every coefficient of a row lives in a different plane)
    const unsigned long long rp_bits = (unsigned long long)(uintptr_t)rp;
    float v[SPW];
#pragma unroll
    for (int j = 0; j < SPW; ++j) {
      const unsigned char* rj = (const unsigned char*)(uintptr_t)__shfl_sync(0xffffffffu, rp_bits, j * G);
      const int csj = __shfl_sync(0xffffffffu, cs, j * G);
      v[j] = (d0 + j < k && lane < ne) ? row_elem<HALF>(rj, (size_t)(5 + nc + lane) * csj) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < SPW; ++j)
      if (d0 + j < k && lane < ne) out_extra[((size_t)tile * max_det + d0 + j) * ne + lane] = v[j];
  } else if (out_extra && ne > 0) {
    const unsigned long long rp_bits = (unsigned long long)(uintptr_t)rp;
#pragma unroll
    for (int j = 0; j < SPW; ++j) {
      const unsigned char* rj = (const unsigned char*)(uintptr_t)__shfl_sync(0xffffffffu, rp_bits, j * G);
      const int csj = __shfl_sync(0xffffffffu, cs, j * G);
      if (d0 + j >= k) break;  // warp-uniform
      float* oe = out_extra + ((size_t)tile * max_det + d0 + j) * ne;
      for (int c = lane; c < ne; c += 32) oe[c] = row_elem<HALF>(rj, (size_t)(5 + nc + c) * csj);
    }
  }
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_debug_nms_phases(uint64_t* device_buf8) {
  g_phase_host = reinterpret_cast<unsigned long long*>(device_buf8);
  return HDY_OK;
}

size_t hdy_nms_workspace_bytes(int bs, int cap) {
  if (bs <= 0 || cap <= kNmsSmemCap) return 0;
  return (size_t)bs * workspace_layout(cap).per_tile;
}

int hdy_nms_tiles(const uint64_t* cand_keys, const float* cand_boxes, const float* cand_cls,
                  const int32_t* counts, int bs, int cap, float iou_thres, float class_offset, int max_nms,
                  int max_det, int32_t* keep_idx, int32_t* keep_slot, float* keep_box, float* keep_score,
                  float* keep_cls, int32_t* keep_counts, float gray_eps, uint8_t* keep_fragile, void* workspace,
                  size_t workspace_bytes, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && cap > 0 && max_det > 0, "hdy_nms_tiles: bs=%d cap=%d max_det=%d", bs, cap, max_det);
  HDY_REQUIRE(iou_thres >= 0.f, "hdy_nms_tiles: iou_thres must be >= 0");
  HDY_REQUIRE(cand_keys && cand_boxes && counts && keep_idx && keep_slot && keep_counts,
              "hdy_nms_tiles: NULL pointer");
  HDY_REQUIRE(((uintptr_t)cand_boxes & 15) == 0 && ((uintptr_t)keep_box & 15) == 0,
              "box arrays must be 16-byte aligned");
  if (bs == 0) return HDY_OK;
  const size_t need = hdy_nms_workspace_bytes(bs, cap);
  if (need > 0 && (workspace == nullptr || workspace_bytes < need)) {
    set_error("hdy_nms_tiles: workspace too small (%zu < %zu)", workspace_bytes, need);
    return HDY_ERR_CAPACITY;
  }
  // tiles with at most 4096 candidates: shared-memory kernel (nms_smem.cu); the rest: workspace kernel below
  int rc = launch_nms_tiles_smem(cand_keys, reinterpret_cast<const float4*>(cand_boxes), cand_cls, counts, bs, cap,
                                 iou_thres, class_offset, max_nms, max_det, keep_idx, keep_slot,
                                 reinterpret_cast<float4*>(keep_box), keep_score, keep_cls, keep_counts, gray_eps,
                                 keep_fragile, g_phase_host, (cudaStream_t)stream);
  if (rc || cap <= kNmsSmemCap) return rc;
  nms_tiles_kernel<<<(unsigned)bs, kNmsThreads, 0, (cudaStream_t)stream>>>(
      cand_keys, reinterpret_cast<const float4*>(cand_boxes), cand_cls, counts, cap, iou_thres, class_offset,
      max_nms, max_det, keep_idx, keep_slot, reinterpret_cast<float4*>(keep_box), keep_score, keep_cls,
      keep_counts, static_cast<unsigned char*>(workspace), keep_fragile);
  return check_launch("hdy_nms_tiles");
}

int hdy_make_keys(const float* scores, int bs, int seg_len, uint64_t* keys, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && seg_len >= 0, "hdy_make_keys: bad sizes");
  const size_t n = (size_t)bs * seg_len;
  if (n == 0) return HDY_OK;
  HDY_REQUIRE(scores && keys, "hdy_make_keys: NULL pointer");
  make_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scores, n, seg_len, keys);
  return check_launch("hdy_make_keys");
}

int hdy_gather_preds(const float* preds, int bs, int N, int row_len, int nc, const int32_t* keep_idx,
                     const int32_t* keep_counts, int max_det, float* out_scores, float* out_extra,
                     hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && row_len >= 5 + nc && nc >= 0 && max_det > 0, "hdy_gather_preds: bad sizes");
  HDY_REQUIRE(keep_idx && keep_counts && out_scores, "hdy_gather_preds: NULL pointer");
  if (bs == 0 || N == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "hdy_gather_preds: bs > 65535");
  dim3 grid((unsigned)((max_det + 127) / 128), (unsigned)bs);
  gather_preds_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(preds, N, row_len, nc, keep_idx, keep_counts,
                                                              max_det, out_scores, out_extra);
  return check_launch("hdy_gather_preds");
}

int hdy_gather_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no, int layout,
                      const int32_t* keep_idx, const int32_t* keep_counts, int max_det, float* out_scores,
                      float* out_level, float* out_extra, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det > 0 && nc >= 0 && no >= 5 + nc, "hdy_gather_logits: bad sizes");
  HDY_REQUIRE(keep_idx && keep_counts && out_scores, "hdy_gather_logits: NULL pointer");
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, layout, 256, &T);
  if (rc) return rc;
  T.nc = nc;
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "hdy_gather_logits: bs > 65535");
  dim3 grid((unsigned)((max_det + 127) / 128), (unsigned)bs);
  gather_logits_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(T, keep_idx, keep_counts, max_det, out_scores,
                                                               out_level, out_extra);
  return check_launch("hdy_gather_logits");
}

static int fill_hier_ops(const int32_t* hier_ops_host, int n_ops, int nc, HierOps* H) {
  HDY_REQUIRE(n_ops >= 0 && n_ops <= 2 * HDY_MAX_SCORES && (n_ops == 0 || hier_ops_host), "bad hier ops");
  H->n = n_ops;
  for (int i = 0; i < n_ops; ++i) {
    const int d = hier_ops_host[2 * i], s = hier_ops_host[2 * i + 1];
    HDY_REQUIRE(d >= 0 && d <= nc && s >= 0 && s <= nc && d != s, "hier op %d: (%d,%d) out of range", i, d, s);
    H->dst[i] = (int8_t)d;
    H->src[i] = (int8_t)s;
  }
  return HDY_OK;
}

int hdy_gather_select_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no, int layout,
                             const int32_t* keep_idx, const int32_t* keep_counts, int max_det,
                             const int32_t* hier_ops_host, int n_ops, float conf_thres, float* out_scores,
                             float* out_level, float* out_extra, float* out_score, int64_t* out_label,
                             hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det > 0 && nc >= 1 && 1 + nc <= 32 && no >= 5 + nc,
              "hdy_gather_select_logits: bad sizes (1 + nc must be <= 32; use hdy_gather_logits + hdy_select_scores)");
  HDY_REQUIRE(keep_idx && keep_counts && out_scores, "hdy_gather_select_logits: NULL pointer");
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, layout, 256, &T);
  if (rc) return rc;
  T.nc = nc;
  HierOps H;
  rc = fill_hier_ops(hier_ops_host, n_ops, nc, &H);
  if (rc) return rc;
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "hdy_gather_select_logits: bs > 65535");
  const int G = 1 + nc <= 8 ? 8 : (1 + nc <= 16 ? 16 : 32);
  const int per_cta = 8 * (32 / G);
  dim3 grid((unsigned)((max_det + per_cta - 1) / per_cta), (unsigned)bs);
  cudaStream_t st = (cudaStream_t)stream;
#define HDY_GS(GG, HH)                                                                                          \
  gather_select_logits_kernel<GG, HH><<<grid, 256, 0, st>>>(T, keep_idx, keep_counts, max_det, H, conf_thres,     \
                                                            out_scores, out_level, out_extra, out_score, out_label)
  const bool half = T.dtype == HDY_F16;
  if (G == 8) {
    if (half) HDY_GS(8, true); else HDY_GS(8, false);
  } else if (G == 16) {
    if (half) HDY_GS(16, true); else HDY_GS(16, false);
  } else {
    if (half) HDY_GS(32, true); else HDY_GS(32, false);
  }
#undef HDY_GS
  return check_launch("hdy_gather_select_logits");
}

int hdy_select_scores(float* scores, const int32_t* keep_counts, int bs, int max_det, int nc,
                      const int32_t* hier_ops_host, int n_ops, float conf_thres, float* out_score,
                      int64_t* out_label, hdy_stream_t stream) {
  HDY_REQUIRE(bs >= 0 && max_det > 0 && nc >= 1 && 1 + nc <= HDY_MAX_SCORES, "hdy_select_scores: bad sizes");
  HDY_REQUIRE(scores && keep_counts, "hdy_select_scores: NULL pointer");
  HDY_REQUIRE(n_ops >= 0 && n_ops <= 2 * HDY_MAX_SCORES && (n_ops == 0 || hier_ops_host),
              "hdy_select_scores: bad hier ops");
  HierOps H;
  H.n = n_ops;
  for (int i = 0; i < n_ops; ++i) {
    const int d = hier_ops_host[2 * i], s = hier_ops_host[2 * i + 1];
    HDY_REQUIRE(d >= 0 && d <= nc && s >= 0 && s <= nc && d != s, "hier op %d: (%d,%d) out of range", i, d, s);
    H.dst[i] = (int8_t)d;
    H.src[i] = (int8_t)s;
  }
  if (bs == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "hdy_select_scores: bs > 65535");
  dim3 grid((unsigned)((max_det + 127) / 128), (unsigned)bs);
  select_scores_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(scores, keep_counts, max_det, nc, H, conf_thres,
                                                               out_score, out_label);
  return check_launch("hdy_select_scores");
}

}  // extern "C"
