// Per-tile greedy IoU NMS for tiles with at most 4096 candidates: one CTA per tile, everything in shared memory.
// Exact torchvision.ops.nms semantics (called at metayolo/models/utils_general.py:342 and :507).
//
//   1. sort      the 64-bit order keys (score desc, row asc).  Up to THREADS keys: a bitonic sort, one key per
//                thread in a register; strides inside a warp are shuffles, only the strides that cross warps go
//                through shared memory.  Only keys move; the slot of every rank is recovered afterwards by a binary
//                search of each candidate's (unique) key in the sorted array.  More keys: an LSD radix sort in shared
//                memory that moves keys and slots together.
//   2. bin       boxes are fetched once (by slot, from L2), classified against a torus grid whose cell is the
//                largest box side (2 x mean side if the sizes are very uneven; larger boxes go to one "large"
//                bucket everybody scans), counted per cell, and copied into CELL ORDER (box + rank), each cell
//                sorted by rank.  A box can only intersect boxes of its own and the 8 neighbouring cells.
//   3. pairs     one thread per box in cell order (neighbouring lanes walk the same candidate runs): every
//                higher-ranked box of the 3x3 neighbourhood with IoU > thr is recorded as a DOMINATOR (up to 4 are
//                stored; a box with more is re-scanned in step 4).  Rank-sorted cells let the walk stop at the
//                first lower-ranked candidate.  A box without dominators is KEPT.
//   4. resolve   fixed point over the dominator lists: KEPT once every dominator is SUPPRESSED, SUPPRESSED as soon
//                as one is KEPT.  This equals sequential greedy NMS; the number of sweeps is the longest
//                suppression chain (a handful for nuclei).
//   5. emit      rank-ordered compaction of KEPT boxes, first max_det.
// Binning only prunes pairs that cannot intersect; every pair that can is tested with hdy_common.cuh's iou_gt
// (fp32, torchvision's operation order), so cell size and bucket choice never change a verdict.
#include <stddef.h>
#include "hdy_common.cuh"
#include "scan_common.cuh"

namespace hdy {

constexpr int kFastCap = 4096;       // candidates per tile of the full-size instance (168 KB: one CTA per SM)
constexpr int kFastCapSmall = 3072;  // ... and of the instance that shares an SM: 126 KB leave room for a 93 KB
                                     // filter CTA, so the HBM-bound filter of the next tile batch (another stream) runs
                                     // WHILE this latency-bound kernel works -- with the 168 KB instance the two
                                     // alternate, and the slide's per-tile part was filter + NMS instead of the filter
constexpr int kFastG = 32;  // torus grid side
constexpr int kFastNB = kFastG * kFastG + 1;
constexpr int kMaxDom = 4;
constexpr int kSortCellMax = 48;  // cells longer than this are left unsorted (then no early stop anywhere)
constexpr float kFastCellMargin = 1.01f;
constexpr float kFastMaxScaled = 16384.0f;

enum : uint8_t { FS_UNKNOWN = 0, FS_KEPT = 1, FS_SUPPRESSED = 2 };

template <int CAP>
struct FastSmemT {
  uint64_t skey[CAP];       // sorted keys (rank order)
  float4 cbox[CAP];         // boxes in cell order (class offset applied)
  uint16_t crank[CAP];      // rank of the box at a cell-order position
  uint16_t pos[CAP];        // rank -> cell-order position (0xffff: degenerate box, KEPT)
  uint16_t slot[CAP];       // rank -> candidate slot (index into the tile's cand_* arrays)
  uint16_t dom[CAP * kMaxDom];
  uint8_t ndom[CAP];
  uint8_t state[CAP];
  uint8_t frag[CAP];        // cell-order position -> has a neighbour whose IoU could cross thr after the shift
  int cell[kFastNB + 3];
  int warp_i[33];
  float warp_f[2][32];
  int flags[4];             // 0: all small cells rank-sorted
};
// the radix sort keeps two [32][256] uint16 count buffers in dom (+ the three byte arrays behind it, all unused until
// the sort is over): 32 KB
static_assert(sizeof(FastSmemT<kFastCapSmall>::dom) + 3 * kFastCapSmall >= 2 * 32 * 256 * 2 &&
                  offsetof(FastSmemT<kFastCapSmall>, ndom) ==
                      offsetof(FastSmemT<kFastCapSmall>, dom) + sizeof(FastSmemT<kFastCapSmall>::dom) &&
                  offsetof(FastSmemT<kFastCapSmall>, cell) >= offsetof(FastSmemT<kFastCapSmall>, dom) + 2 * 32 * 256 * 2,
              "radix count buffers must fit behind dom");

// Bitonic sort of THREADS keys, one per thread (thread t owns element t).
template <int THREADS>
__device__ __forceinline__ void bitonic_sort_regs(uint64_t& k, uint64_t* smem) {
  const int t = threadIdx.x;
#pragma unroll 1
  for (int kk = 2; kk <= THREADS; kk <<= 1) {
#pragma unroll 1
    for (int j = kk >> 1; j >= 32; j >>= 1) {  // partner lives in another warp: through shared memory
      __syncthreads();
      smem[t] = k;
      __syncthreads();
      const uint64_t o = smem[t ^ j];
      const bool keep_min = ((t & j) == 0) == ((t & kk) == 0);
      k = keep_min ? (k < o ? k : o) : (k > o ? k : o);
    }
    const int jmax = min(kk >> 1, 16);
#pragma unroll 1
    for (int j = jmax; j >= 1; j >>= 1) {  // partner lives in another lane: shuffles
      const bool keep_min = ((t & j) == 0) == ((t & kk) == 0);
      const uint64_t o = __shfl_xor_sync(0xffffffffu, k, j);
      k = keep_min ? (k < o ? k : o) : (k > o ? k : o);
    }
  }
}

template <int THREADS>
__device__ __forceinline__ void load_sort_store(const uint64_t* __restrict__ gkeys, int n_in, uint64_t* skey,
                                                uint16_t* slot) {
  const int t = threadIdx.x;
  const uint64_t mine = (t < n_in) ? gkeys[t] : ~0ull;  // (~orderable(score) << 32) | row, unique inside a tile
  uint64_t k = mine;
  bitonic_sort_regs<THREADS>(k, skey);
  __syncthreads();
  skey[t] = k;
  __syncthreads();
  // rank of candidate t = position of its key in the sorted array (keys are unique)
  if (t < n_in) {
    int lo = 0;
#pragma unroll
    for (int step = THREADS >> 1; step > 0; step >>= 1)
      if (skey[lo + step] <= mine) lo += step;
    slot[lo] = (uint16_t)t;
  }
  __syncthreads();
}

// ---- LSD radix sort of the tile's keys in shared memory (tiles with more than THREADS keys; the bitonic network above
// sorts the smaller ones).  Eight 8-bit digits, least significant first, bytes that are equal in every key skipped (row indices
// below 65 536 leave two of them constant).  Per pass: every warp ranks its own contiguous run of keys with
// ballots (stable: item e of lane l is element w*EPW + e*32 + l), leaving per-warp digit counts in `whist`; a column
// scan over the 32 warps and a 256-entry scan give every (warp, digit) its base; keys and slots are scattered to the
// other buffer.  ~2.6 k cycles per pass at 4096 keys against ~72 k cycles for the 78-step bitonic network.
template <int THREADS, int CAP>
__device__ __forceinline__ void radix_sort_store(const uint64_t* __restrict__ gkeys, int n_in, FastSmemT<CAP>& S) {
  static_assert(THREADS == 1024, "32 warps, 4 threads per digit in the column scan");
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int items = (n_in + THREADS - 1) / THREADS;  // 1..4 keys per thread
  const int epw = items * 32;                       // keys per warp
  // buffers: A = (skey, slot), B = first half of cbox / crank; per-warp digit counts in dom; digit bases behind B
  uint64_t* keyA = S.skey;
  uint64_t* keyB = reinterpret_cast<uint64_t*>(S.cbox);
  uint16_t* slotA = S.slot;
  uint16_t* slotB = S.crank;
  uint16_t* whist = S.dom;  // [32][256]
  int* dbase = reinterpret_cast<int*>(S.cbox + CAP / 2);  // [256] exclusive digit offsets
  int* dflag = dbase + 256;   // [128], start-up only
  int* gpart = dbase + 256;   // [4][256] group sums of the column scan

  // load, and find the bytes that differ at all (OR ^ AND over the keys)
  uint32_t or_lo = 0u, or_hi = 0u, and_lo = ~0u, and_hi = ~0u;
  for (int e = 0; e < items; ++e) {
    const int i = w * epw + e * 32 + lane;
    if (i < n_in) {
      const uint64_t k = gkeys[i];
      keyA[i] = k;
      slotA[i] = (uint16_t)i;
      or_lo |= (uint32_t)k;
      or_hi |= (uint32_t)(k >> 32);
      and_lo &= (uint32_t)k;
      and_hi &= (uint32_t)(k >> 32);
    }
  }
  or_lo = __reduce_or_sync(0xffffffffu, or_lo);
  or_hi = __reduce_or_sync(0xffffffffu, or_hi);
  and_lo = __reduce_and_sync(0xffffffffu, and_lo);
  and_hi = __reduce_and_sync(0xffffffffu, and_hi);
  if (lane == 0) {
    dflag[w] = (int)or_lo;   // differing bits ACROSS warps: or / and of the warp results
    dflag[32 + w] = (int)and_lo;
    dflag[64 + w] = (int)or_hi;
    dflag[96 + w] = (int)and_hi;
  }
  __syncthreads();
  uint32_t diff_lo, diff_hi;
  {
    const uint32_t a = (uint32_t)dflag[lane], b = (uint32_t)dflag[32 + lane];
    const uint32_t c = (uint32_t)dflag[64 + lane], d = (uint32_t)dflag[96 + lane];
    diff_lo = __reduce_or_sync(0xffffffffu, a) ^ __reduce_and_sync(0xffffffffu, b);
    diff_hi = __reduce_or_sync(0xffffffffu, c) ^ __reduce_and_sync(0xffffffffu, d);
  }
  __syncthreads();  // dflag is reused below

  {  // clear the first per-warp count buffer (32 x 256 uint16 = 4096 words)
    uint32_t* z = reinterpret_cast<uint32_t*>(whist);
#pragma unroll
    for (int j = 0; j < 4; ++j) z[t + j * THREADS] = 0u;
  }
  __syncthreads();
  uint64_t* ksrc = keyA;
  uint64_t* kdst = keyB;
  uint16_t* ssrc = slotA;
  uint16_t* sdst = slotB;
#pragma unroll 1
  for (int byte = 0; byte < 8; ++byte) {
    const uint32_t diff = byte < 4 ? (diff_lo >> (8 * byte)) & 255u : (diff_hi >> (8 * (byte - 4))) & 255u;
    if (diff == 0u) continue;  // every key has the same digit here (block-uniform)
    const int shift = 8 * byte;
    // (the per-warp counts of this pass were cleared during the previous pass's scatter, or before the loop)
    // 1. rank inside the warp's run
    uint64_t k[4];
    uint16_t sl[4];
    int loc[4], dig[4];
    uint16_t* wh = whist + w * 256;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (e < items) {
        const int i = w * epw + e * 32 + lane;
        const bool valid = i < n_in;
        k[e] = valid ? ksrc[i] : 0ull;
        sl[e] = valid ? ssrc[i] : (uint16_t)0;
        const int d = valid ? (int)((k[e] >> shift) & 255ull) : 0;
        // lanes holding the same digit: eight ballots (match_any is microcoded and far slower for 32 distinct values)
        unsigned peers = __ballot_sync(0xffffffffu, valid);
#pragma unroll
        for (int bit = 0; bit < 8; ++bit) {
          const unsigned m = __ballot_sync(0xffffffffu, (d >> bit) & 1);
          peers &= ((d >> bit) & 1) ? m : ~m;
        }
        const int r = __popc(peers & ((1u << lane) - 1u));
        const int pre = valid ? (int)wh[d] : 0;
        __syncwarp();
        if (valid && r == 0) wh[d] = (uint16_t)(pre + __popc(peers));
        __syncwarp();
        loc[e] = pre + r;
        dig[e] = valid ? d : -1;
      }
    }
    __syncthreads();
    // 2. column scan: thread (g, d) covers warps 8g .. 8g+7 of digit d; a warp reads 32 consecutive digits of one
    //    row at a time (conflict-free), the four groups meet through gpart
    {
      const int g = t >> 8, d = t & 255;
      int c[8], part = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        c[j] = whist[(g * 8 + j) * 256 + d];
        part += c[j];
      }
      gpart[g * 256 + d] = part;
      __syncthreads();
      int run = 0;
      for (int gg = 0; gg < g; ++gg) run += gpart[gg * 256 + d];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        whist[(g * 8 + j) * 256 + d] = (uint16_t)run;
        run += c[j];
      }
      if (g == 3) dbase[d] = run;  // digit total
    }
    __syncthreads();
    if (w == 0) {  // exclusive scan of the 256 digit totals
      int v[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = dbase[lane * 8 + j];
        sum += v[j];
      }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
      }
      int run = incl - sum;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        dbase[lane * 8 + j] = run;
        run += v[j];
      }
    }
    __syncthreads();
    // 3. scatter; the other count buffer is cleared for the next pass meanwhile
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (e < items && dig[e] >= 0) {
        const int dst = dbase[dig[e]] + (int)wh[dig[e]] + loc[e];
        kdst[dst] = k[e];
        sdst[dst] = sl[e];
      }
    }
    {
      uint16_t* other = whist == S.dom ? S.dom + 32 * 256 : S.dom;
      uint32_t* z = reinterpret_cast<uint32_t*>(other);
#pragma unroll
      for (int j = 0; j < 4; ++j) z[t + j * THREADS] = 0u;
      whist = other;
    }
    __syncthreads();
    uint64_t* tk = ksrc;
    ksrc = kdst;
    kdst = tk;
    uint16_t* ts = ssrc;
    ssrc = sdst;
    sdst = ts;
  }
  if (ksrc != keyA) {  // an odd number of passes ran: bring the result home
    for (int i = t; i < n_in; i += THREADS) {
      keyA[i] = ksrc[i];
      slotA[i] = ssrc[i];
    }
    __syncthreads();
  }
}

struct FastGeom {
  float cell_size, inv_cell, max_center;
};

// 0 = degenerate (can never intersect), 1 = small (binned by centre), 2 = large
__device__ __forceinline__ int fast_classify(const float4& b, const FastGeom& g, int& bucket, int& ix, int& iy) {
  const float w = b.z - b.x, h = b.w - b.y;
  if (w <= 0.f || h <= 0.f) return 0;
  const float cx = (b.x + b.z) * 0.5f, cy = (b.y + b.w) * 0.5f;
  if (w <= g.cell_size && h <= g.cell_size && fabsf(cx) <= g.max_center && fabsf(cy) <= g.max_center) {
    ix = (int)floorf(cx * g.inv_cell);
    iy = (int)floorf(cy * g.inv_cell);
    bucket = (ix & (kFastG - 1)) + (iy & (kFastG - 1)) * kFastG;
    return 1;
  }
  bucket = kFastG * kFastG;
  return 2;  // also NaN / inf coordinates
}

template <int THREADS, int CAP>
__global__ void __maxnreg__(CAP <= 3072 ? 56 : 64) nms_tiles_smem_kernel(
    const uint64_t* __restrict__ cand_keys, const float4* __restrict__ cand_boxes,
    const float* __restrict__ cand_cls, const int32_t* __restrict__ counts, int cap, float thr, float class_offset,
    int max_nms, int max_det, int32_t* __restrict__ keep_idx, int32_t* __restrict__ keep_slot,
    float4* __restrict__ keep_box, float* __restrict__ keep_score, float* __restrict__ keep_cls,
    int32_t* __restrict__ keep_counts, float gray_eps, uint8_t* __restrict__ keep_fragile,
    unsigned long long* __restrict__ phase_cycles) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FastSmemT<CAP>& S = *reinterpret_cast<FastSmemT<CAP>*>(smem_raw);
  // gray zone: pairs that this NMS leaves alone (IoU <= thr in tile coordinates) but whose IoU may exceed thr once both
  // boxes are shifted to slide coordinates and rounded.  Both boxes of such a pair are reported FRAGILE: the slide-level
  // merge must look at them even if they sit in the interior of their tile (see DESIGN.md, interior shortcut).
  const bool gray = keep_fragile != nullptr && gray_eps > 0.f;
  uint8_t* o_frag = keep_fragile ? keep_fragile + (size_t)blockIdx.x * max_det : nullptr;
  constexpr int MAXR = CAP / THREADS;  // ranks owned by one thread
  const int tile = blockIdx.x;
  const int t = threadIdx.x;
  const int n_in = min(counts[tile], cap);
  if (n_in > CAP) return;  // handled by the workspace kernel (the launcher picks CAP >= cap when cap fits an instance)
  int32_t* o_idx = keep_idx + (size_t)tile * max_det;
  int32_t* o_slot = keep_slot + (size_t)tile * max_det;
  float4* o_box = keep_box ? keep_box + (size_t)tile * max_det : nullptr;
  float* o_score = keep_score ? keep_score + (size_t)tile * max_det : nullptr;
  float* o_cls = keep_cls ? keep_cls + (size_t)tile * max_det : nullptr;
  if (n_in <= 0) {
    if (t == 0) keep_counts[tile] = 0;
    return;
  }
  const uint64_t* gkeys = cand_keys + (size_t)tile * cap;
  const float4* gboxes = cand_boxes + (size_t)tile * cap;
  const float* gcls = cand_cls ? cand_cls + (size_t)tile * cap : nullptr;
  // `elif n > max_nms: x = x[x[:, 4].argsort(descending=True)[:max_nms]]`            utils_general.py:501-502
  const int n = (max_nms > 0 && n_in > max_nms) ? max_nms : n_in;
  long long t0 = 0;
  auto mark = [&](int phase) {
    if (phase_cycles && t == 0) {
      const long long t1 = clock64();
      if (phase >= 0) atomicAdd(phase_cycles + phase, (unsigned long long)(t1 - t0));
      t0 = t1;
    }
  };
  mark(-1);

  // ---- 1. sort ----------------------------------------------------------------------------------------------
  // the sorting network wins up to THREADS = 1024 keys (20.7 k vs 22.7 k cycles), the radix sort above
  if (n_in > THREADS)
    radix_sort_store<THREADS, CAP>(gkeys, n_in, S);
  else
    load_sort_store<THREADS>(gkeys, n_in, S.skey, S.slot);
  mark(1);

  // ---- 2. boxes (one L2 gather, kept in registers), statistics, binning -------------------------------------
  float4 bx[MAXR];
  float ext_sum = 0.f, ext_max = 0.f;
  int ext_cnt = 0;
#pragma unroll
  for (int e = 0; e < MAXR; ++e) {
    const int r = t + e * THREADS;
    bx[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < n) {
      const uint32_t s = S.slot[r];
      float4 b = gboxes[s];
      if (gcls) {
        const float c = __fmul_rn(gcls[s], class_offset);  // c = x[:, 5:6] * max_wh     utils_general.py:505
        b.x = __fadd_rn(b.x, c);
        b.y = __fadd_rn(b.y, c);
        b.z = __fadd_rn(b.z, c);
        b.w = __fadd_rn(b.w, c);
      }
      bx[e] = b;
      const float w = b.z - b.x, h = b.w - b.y;
      if (w > 0.f && h > 0.f && w < 3.0e38f && h < 3.0e38f) {
        const float m = fmaxf(w, h);
        ext_sum += m;
        ext_max = fmaxf(ext_max, m);
        ++ext_cnt;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ext_sum += __shfl_xor_sync(0xffffffffu, ext_sum, o);
    ext_max = fmaxf(ext_max, __shfl_xor_sync(0xffffffffu, ext_max, o));
    ext_cnt += __shfl_xor_sync(0xffffffffu, ext_cnt, o);
  }
  if ((t & 31) == 0) {
    S.warp_f[0][t >> 5] = ext_sum;
    S.warp_f[1][t >> 5] = ext_max;
    S.warp_i[t >> 5] = ext_cnt;
  }
  for (int i = t; i < kFastNB + 3; i += THREADS) S.cell[i] = 0;
  if (gray)
    for (int i = t; i < CAP; i += THREADS) S.frag[i] = 0;
  if (t == 0) S.flags[0] = 1;
  __syncthreads();
  FastGeom g;
  {
    float tot_sum = 0.f, tot_max = 0.f;
    int tot_cnt = 0;
    for (int w = 0; w < THREADS / 32; ++w) {
      tot_sum += S.warp_f[0][w];
      tot_max = fmaxf(tot_max, S.warp_f[1][w]);
      tot_cnt += S.warp_i[w];
    }
    const float mean = tot_cnt ? tot_sum / (float)tot_cnt : 1.0f;
    float cs = (tot_max <= 2.5f * mean) ? tot_max : 2.0f * mean;
    if (!(cs > 1e-20f) || !(cs < 1e30f)) cs = 1.0f;
    g.cell_size = cs;
    g.inv_cell = 1.0f / (cs * kFastCellMargin);
    g.max_center = cs * kFastMaxScaled;
  }
  __syncthreads();  // warp_i is reused by the scan

  int bucket_of[MAXR], ofs[MAXR];
#pragma unroll
  for (int e = 0; e < MAXR; ++e) {
    const int r = t + e * THREADS;
    bucket_of[e] = -1;
    ofs[e] = 0;
    if (r < n) {
      int bucket = 0, ix, iy;
      if (fast_classify(bx[e], g, bucket, ix, iy)) {
        bucket_of[e] = bucket;
        ofs[e] = atomicAdd(&S.cell[bucket], 1);
      } else {
        S.pos[r] = 0xffffu;  // degenerate: never intersects anything -> KEPT
      }
    }
  }
  __syncthreads();
  // cell[b] = first position of bucket b, cell[NB] = number of binned boxes
  const int n_active = block_exclusive_scan_inplace<THREADS>(S.cell, kFastNB + 1, S.warp_i);
  const int large_begin = S.cell[kFastNB - 1];
#pragma unroll
  for (int e = 0; e < MAXR; ++e)
    if (bucket_of[e] >= 0) S.crank[S.cell[bucket_of[e]] + ofs[e]] = (uint16_t)(t + e * THREADS);
  __syncthreads();
  // every small cell sorted by rank (tiny insertion sorts, one thread per cell)
  for (int b = t; b < kFastNB - 1; b += THREADS) {
    const int beg = S.cell[b], end = S.cell[b + 1];
    if (end - beg > kSortCellMax) {
      S.flags[0] = 0;
    } else {
      for (int i = beg + 1; i < end; ++i) {
        const uint16_t v = S.crank[i];
        int j = i - 1;
        while (j >= beg && S.crank[j] > v) {
          S.crank[j + 1] = S.crank[j];
          --j;
        }
        S.crank[j + 1] = v;
      }
    }
  }
  __syncthreads();
  for (int p = t; p < n_active; p += THREADS) S.pos[S.crank[p]] = (uint16_t)p;
  __syncthreads();
#pragma unroll
  for (int e = 0; e < MAXR; ++e)
    if (bucket_of[e] >= 0) S.cbox[S.pos[t + e * THREADS]] = bx[e];
  const bool sorted = S.flags[0] != 0;
  __syncthreads();
  mark(3);

  // ---- 3. dominators ----------------------------------------------------------------------------------------
  // begin offsets -> the walker wants [cell[b-1], cell[b]) with cell[-1] = 0: shift view by one
  const int* cell_end = S.cell + 1;  // cell_end[b] = end of bucket b; begin = b ? cell_end[b-1] : 0 (== S.cell[b])
  for (int p = t; p < large_begin; p += THREADS) {
    const float4 bi = S.cbox[p];
    const int ri = S.crank[p];
    int nd = 0;
    auto record = [&](int q) {
      const float4 bq = S.cbox[q];
      if (iou_gt(bq, bi, thr)) {
        if (nd < kMaxDom) S.dom[p * kMaxDom + nd] = (uint16_t)q;
        ++nd;
      } else if (gray && iou_may_exceed(bq, bi, thr, gray_eps)) {
        S.frag[p] = 1;
        S.frag[q] = 1;
      }
    };
    const float cx = (bi.x + bi.z) * 0.5f, cy = (bi.y + bi.w) * 0.5f;
    const int ix = (int)floorf(cx * g.inv_cell), iy = (int)floorf(cy * g.inv_cell);
#pragma unroll 1
    for (int dy = -1; dy <= 1; ++dy) {
      const int rowb = ((iy + dy) & (kFastG - 1)) * kFastG;
#pragma unroll 1
      for (int dx = -1; dx <= 1; ++dx) {
        const int b = ((ix + dx) & (kFastG - 1)) + rowb;
        const int beg = S.cell[b], end = cell_end[b];
        for (int q = beg; q < end; ++q) {
          if ((int)S.crank[q] >= ri) {
            if (sorted) break;
            continue;
          }
          record(q);
        }
      }
    }
    for (int q = large_begin; q < n_active; ++q)
      if ((int)S.crank[q] < ri) record(q);
    S.ndom[p] = (uint8_t)min(nd, 255);
    S.state[p] = nd ? FS_UNKNOWN : FS_KEPT;
  }
  // entries of the "large" bucket can intersect anything: the whole CTA scans the tile for each of them (there are
  // none for nuclei-sized boxes; a serial scan by one thread would take longer than the rest of the kernel)
  for (int p = large_begin; p < n_active; ++p) {
    __syncthreads();
    if (t == 0) S.flags[1] = 0;
    __syncthreads();
    const float4 bi = S.cbox[p];
    const int ri = S.crank[p];
    for (int q = t; q < n_active; q += THREADS) {
      if ((int)S.crank[q] < ri) {
        const float4 bq = S.cbox[q];
        if (iou_gt(bq, bi, thr)) {
          const int k = atomicAdd(&S.flags[1], 1);
          if (k < kMaxDom) S.dom[p * kMaxDom + k] = (uint16_t)q;
        } else if (gray && iou_may_exceed(bq, bi, thr, gray_eps)) {
          S.frag[p] = 1;
          S.frag[q] = 1;
        }
      }
    }
    __syncthreads();
    if (t == 0) {
      const int nd = S.flags[1];
      S.ndom[p] = (uint8_t)min(nd, 255);
      S.state[p] = nd ? FS_UNKNOWN : FS_KEPT;
    }
  }
  __syncthreads();
  mark(4);

  // ---- 4. fixed point over the dominator lists --------------------------------------------------------------
  volatile uint8_t* vstate = S.state;
  int rounds = 0;
  while (true) {
    int unknown = 0;
    for (int p = t; p < n_active; p += THREADS) {
      if (vstate[p] != FS_UNKNOWN) continue;
      const int nd = S.ndom[p];
      int decided = FS_KEPT;
      if (nd <= kMaxDom) {
        for (int k = 0; k < nd; ++k) {
          const uint8_t sq = vstate[S.dom[p * kMaxDom + k]];
          if (sq == FS_KEPT) {
            decided = FS_SUPPRESSED;
            break;
          }
          if (sq == FS_UNKNOWN) decided = FS_UNKNOWN;
        }
      } else if (p >= large_begin) {
        continue;  // overflowed large entry: resolved by the whole CTA below
      } else {
        // more dominators than slots: walk the neighbourhood again
        const float4 bi = S.cbox[p];
        const int ri = S.crank[p];
        auto visit = [&](int q) -> bool {
          if (iou_gt(S.cbox[q], bi, thr)) {
            const uint8_t sq = vstate[q];
            if (sq == FS_KEPT) {
              decided = FS_SUPPRESSED;
              return true;
            }
            if (sq == FS_UNKNOWN) decided = FS_UNKNOWN;
          }
          return false;
        };
        const float cx = (bi.x + bi.z) * 0.5f, cy = (bi.y + bi.w) * 0.5f;
        const int ix = (int)floorf(cx * g.inv_cell), iy = (int)floorf(cy * g.inv_cell);
        bool done = false;
#pragma unroll 1
        for (int dy = -1; dy <= 1 && !done; ++dy) {
          const int rowb = ((iy + dy) & (kFastG - 1)) * kFastG;
#pragma unroll 1
          for (int dx = -1; dx <= 1 && !done; ++dx) {
            const int b = ((ix + dx) & (kFastG - 1)) + rowb;
            const int beg = S.cell[b], end = cell_end[b];
            for (int q = beg; q < end && !done; ++q) {
              if ((int)S.crank[q] >= ri) {
                if (sorted) break;
                continue;
              }
              done = visit(q);
            }
          }
        }
        for (int q = large_begin; q < n_active && !done; ++q)
          if ((int)S.crank[q] < ri) done = visit(q);
      }
      if (decided != FS_UNKNOWN)
        vstate[p] = (uint8_t)decided;
      else
        unknown = 1;
    }
    for (int p = large_begin; p < n_active; ++p) {  // overflowed large entries, one at a time, all threads
      __syncthreads();
      if (S.ndom[p] <= kMaxDom || vstate[p] != FS_UNKNOWN) continue;  // uniform: only thread 0 writes these, below
      const float4 bi = S.cbox[p];
      const int ri = S.crank[p];
      int kept_dom = 0, unk_dom = 0;
      for (int q = t; q < n_active; q += THREADS) {
        if ((int)S.crank[q] < ri && iou_gt(S.cbox[q], bi, thr)) {
          const uint8_t sq = vstate[q];
          kept_dom |= sq == FS_KEPT;
          unk_dom |= sq == FS_UNKNOWN;
        }
      }
      kept_dom = __syncthreads_or(kept_dom);
      unk_dom = __syncthreads_or(unk_dom);
      if (kept_dom) {
        if (t == 0) vstate[p] = FS_SUPPRESSED;
      } else if (!unk_dom) {
        if (t == 0) vstate[p] = FS_KEPT;
      } else {
        unknown = 1;
      }
    }
    ++rounds;
    if (!__syncthreads_or(unknown)) break;
  }
  mark(5);

  // ---- 5. rank-ordered compaction of survivors --------------------------------------------------------------
  {
    const int items_per = (n + THREADS - 1) / THREADS;
    const int b = min(t * items_per, n), e = min(b + items_per, n);
    auto kept = [&](int r) -> bool {
      const uint16_t p = S.pos[r];
      return p == 0xffffu || S.state[p] == FS_KEPT;
    };
    int cnt = 0;
    for (int r = b; r < e; ++r) cnt += kept(r);
    const int lane = t & 31, warp = t >> 5;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) S.warp_i[warp] = incl;
    __syncthreads();
    int base = 0, total = 0;
    for (int w = 0; w < THREADS / 32; ++w) {
      if (w < warp) base += S.warp_i[w];
      total += S.warp_i[w];
    }
    int opos = base + incl - cnt;
    for (int r = b; r < e && opos < max_det; ++r) {
      if (kept(r)) {
        const uint64_t k = S.skey[r];
        const uint32_t s = S.slot[r];
        o_idx[opos] = (int32_t)key_index(k);
        o_slot[opos] = (int32_t)s;
        if (o_box) o_box[opos] = gboxes[s];
        if (o_score) o_score[opos] = key_score(k);
        if (o_cls) o_cls[opos] = gcls ? gcls[s] : 0.f;
        if (o_frag) {
          const uint16_t pp = S.pos[r];
          o_frag[opos] = (gray && pp != 0xffffu) ? S.frag[pp] : (uint8_t)0;
        }
        ++opos;
      }
    }
    if (t == 0) keep_counts[tile] = min(total, max_det);
  }
  mark(6);
  if (phase_cycles && t == 0) {
    atomicAdd(phase_cycles + 7, 1ull);
    atomicAdd(phase_cycles + 0, (unsigned long long)rounds);
  }
}

constexpr int kFastThreads = 1024;

template <int CAP>
static int launch_nms_instance(const uint64_t* cand_keys, const float4* cand_boxes, const float* cand_cls,
                               const int32_t* counts, int bs, int cap, float thr, float class_offset, int max_nms,
                               int max_det, int32_t* keep_idx, int32_t* keep_slot, float4* keep_box, float* keep_score,
                               float* keep_cls, int32_t* keep_counts, float gray_eps, uint8_t* keep_fragile,
                               unsigned long long* phase_cycles, cudaStream_t stream) {
  // the attribute is per DEVICE: a process-wide flag would leave every GPU but the first without the opt-in
  static bool attr_set[64] = {};
  int dev_i = 0;
  cudaGetDevice(&dev_i);
  if (dev_i < 0 || dev_i >= 64 || !attr_set[dev_i]) {
    cudaError_t e = cudaFuncSetAttribute(nms_tiles_smem_kernel<kFastThreads, CAP>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmemT<CAP>));
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute(nms_tiles_smem_kernel): %s", cudaGetErrorString(e));
      return HDY_ERR_CUDA;
    }
    if (dev_i >= 0 && dev_i < 64) attr_set[dev_i] = true;
  }
  nms_tiles_smem_kernel<kFastThreads, CAP><<<(unsigned)bs, kFastThreads, sizeof(FastSmemT<CAP>), stream>>>(
      cand_keys, cand_boxes, cand_cls, counts, cap, thr, class_offset, max_nms, max_det, keep_idx, keep_slot,
      keep_box, keep_score, keep_cls, keep_counts, gray_eps, keep_fragile, phase_cycles);
  return check_launch("hdy_nms_tiles(smem)");
}

int launch_nms_tiles_smem(const uint64_t* cand_keys, const float4* cand_boxes, const float* cand_cls,
                          const int32_t* counts, int bs, int cap, float thr, float class_offset, int max_nms,
                          int max_det, int32_t* keep_idx, int32_t* keep_slot, float4* keep_box, float* keep_score,
                          float* keep_cls, int32_t* keep_counts, float gray_eps, uint8_t* keep_fragile,
                          unsigned long long* phase_cycles, cudaStream_t stream) {
  // candidate lists of at most 3072 entries take the instance that leaves room for a filter CTA on the same SM
  if (cap <= kFastCapSmall)
    return launch_nms_instance<kFastCapSmall>(cand_keys, cand_boxes, cand_cls, counts, bs, cap, thr, class_offset,
                                              max_nms, max_det, keep_idx, keep_slot, keep_box, keep_score, keep_cls,
                                              keep_counts, gray_eps, keep_fragile, phase_cycles, stream);
  return launch_nms_instance<kFastCap>(cand_keys, cand_boxes, cand_cls, counts, bs, cap, thr, class_offset, max_nms,
                                       max_det, keep_idx, keep_slot, keep_box, keep_score, keep_cls, keep_counts,
                                       gray_eps, keep_fragile, phase_cycles, stream);
}

}  // namespace hdy
