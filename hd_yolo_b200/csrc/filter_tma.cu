// Fused decode + confidence filter + stream compaction, TMA-staged (layout 0: [bs, na, ny, nx, no] rows).
//
// Same arithmetic and outputs as filter_compact_logits_kernel in decode.cu (reference: yolo_head.py:185-213,
// utils_general.py:121-128, :332, :336-337); this is the path taken whenever the level tensors are 16-byte aligned.
//
// HBM -> SM:  every WARP is an independent streamer.  It owns NBUF shared-memory buffers, each filled by ONE bulk-async
//             copy (cp.async.bulk.shared::cluster.global, the 1-D TMA path: SASS UBLKCP) of 32*rpl whole rows
//             (~4.5 KB) that completes an mbarrier through complete_tx; lane 0 re-arms the barrier and issues the copy
//             for chunk k+NBUF as soon as the warp has read chunk k.  There is no producer warp, no `empty` barrier
//             and no CTA-wide synchronisation: measured on B200 (tools/micro/ring_trace.cu), a CTA-wide ring in which
//             every consumer warp visits every chunk is a serial chain of ~270 ns per chunk (try_wait + handshake),
//             which capped the first version of this kernel at 2.3 TB/s whatever the number of stages.
//             No thread spends instructions on moving the 95 % of rows that are rejected.
// phase A:    (every row) one LDS of the objectness logit + one compare.  Rows are rejected on the LOGIT:
//             x < t_lo = logit(conf) - margin implies sigmoid(x) <= conf for certain (margin = 1e-4 (1 + |logit|),
//             ~1000x the error of expf + division).  Rows that may pass copy their five logits and their identity
//             into the warp's private QUEUE in shared memory (64 entries).  ~5 % of the rows get here, but ~80 % of
//             the 32-row groups contain at least one, so decoding them in place (one divergent pass per group) made
//             the kernel issue-bound (profiles/r01_a, r01_b).
// phase B:    (32 survivors at a time) every lane takes one queue entry: sigmoid, the reference's own `> conf` test
//             (so the verdict is identical to comparing the fp32 sigmoid), box decode, min-size test; one atomicAdd
//             per (warp, tile) reserves the run in the tile's candidate list and the lanes write key + box.
#include "hdy_common.cuh"

namespace hdy {

// A level's tensor [bs, na, ny, nx, no] is ONE contiguous run of bs * rows rows, so chunks are cut from that run
// without regard to tile boundaries (tile = global row / rows); only the last chunk of a level is short.
struct ItemTable {
  int begin[HDY_MAX_LEVELS + 1];  // first item of every level, total in [nl]
};

struct QueueA {
  float l0, l1, l2, l3;
};
struct QueueB {
  float obj;
  int row;    // row inside the tile's level
  int tile;
  int level;
};
static_assert(sizeof(QueueA) == 16 && sizeof(QueueB) == 16, "queue entries are 128-bit");
constexpr int kQueueLen = 64;
// per-warp shared memory: [NBUF x buf_bytes][queue A 1 KB][queue B 1 KB][pick list 256 B][NBUF barriers, 64 B]
__host__ __device__ constexpr size_t per_warp_bytes(int nbuf, int buf_bytes) {
  return (size_t)nbuf * buf_bytes + 2 * kQueueLen * 16 + 256 + 64;
}

template <bool HALF>
struct LogitElem {
  using type = float;
};
template <>
struct LogitElem<true> {
  using type = __half;
};
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }  // exact

// WARPS independent streamers per CTA.  Per-warp shared memory: NBUF chunk buffers, NBUF mbarriers, one queue.
// HALF: the level tensors hold fp16 logits (a half() model's head, val_nuclei.py:115-116); they are widened to fp32 as
// they are read from shared memory -- half the HBM bytes, the same arithmetic.
template <int WARPS, int NBUF, int RPL, bool HALF>
__global__ void __launch_bounds__(WARPS * 32) filter_compact_tma_kernel(
    const __grid_constant__ LevelTable T, const __grid_constant__ ItemTable I, int bs, int buf_bytes,
    float t_lo, float conf_thres, float min_size, int cap, uint64_t* __restrict__ cand_keys,
    float4* __restrict__ cand_boxes, int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using E = typename LogitElem<HALF>::type;
  constexpr int kEsz = (int)sizeof(E);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int no = T.no;
  constexpr int chunk_rows = 32 * RPL;
  const size_t per_warp = per_warp_bytes(NBUF, buf_bytes);
  unsigned char* base = smem_raw + (size_t)warp * per_warp;
  E* bufs = reinterpret_cast<E*>(base);
  QueueA* qa = reinterpret_cast<QueueA*>(base + (size_t)NBUF * buf_bytes);
  QueueB* qb = reinterpret_cast<QueueB*>(base + (size_t)NBUF * buf_bytes + kQueueLen * 16);
  uint8_t* pick = base + (size_t)NBUF * buf_bytes + 2 * kQueueLen * 16;  // [256] chunk rows that passed phase A
  uint64_t* full = reinterpret_cast<uint64_t*>(pick + 256);

  const int total = I.begin[T.nl];
  const int gw = (int)blockIdx.x * WARPS + warp, GW = (int)gridDim.x * WARPS;
  const int n_my = gw < total ? (total - gw + GW - 1) / GW : 0;
  if (n_my == 0) return;

  if (lane == 0) {
    for (int b = 0; b < NBUF; ++b) mbar_init(&full[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  struct Item {
    const E* src;
    int rows, level, grow0;
  };
  auto item_at = [&](int j) -> Item {
    int l = 0;
#pragma unroll 1
    for (int i = 1; i < T.nl; ++i)
      if (j >= I.begin[i]) l = i;
    Item it;
    it.level = l;
    it.grow0 = (j - I.begin[l]) * chunk_rows;
    it.rows = min(chunk_rows, bs * T.lv[l].rows - it.grow0);
    it.src = reinterpret_cast<const E*>(T.lv[l].ptr) + (size_t)it.grow0 * no;
    return it;
  };
  auto issue = [&](int k, int b) {  // lane 0 only: chunk k of this warp -> buffer b
    const Item it = item_at(gw + k * GW);
    const uint32_t bytes = ((uint32_t)(it.rows * no) * (uint32_t)kEsz) & ~15u;
    mbar_arrive_expect_tx(&full[b], bytes);
    if (bytes) bulk_copy_g2s(reinterpret_cast<unsigned char*>(bufs) + (size_t)b * buf_bytes, it.src, bytes, &full[b]);
  };
  if (lane == 0)
    for (int b = 0; b < NBUF && b < n_my; ++b) issue(b, b);

  int qn = 0;  // entries in the queue (warp-uniform)
  const unsigned lt_mask = (1u << lane) - 1u;

  // The run reserved by the previous phase B is written one phase B later, so that the atomicAdd's round trip to
  // L2 (~0.4 us, the largest single stall in profiles/r01_c) overlaps the next chunks.
  bool p_any = false, p_cand = false;
  int p_base = 0, p_leader = 0, p_tile = 0;
  unsigned p_grp = 0;
  uint64_t p_key = 0;
  float4 p_box = make_float4(0.f, 0.f, 0.f, 0.f);
  auto put = [&](int t0, int pos, unsigned grp, uint64_t key, const float4& box) {
    const int q = pos + __popc(grp & lt_mask);
    if (q < cap) {
      const size_t o = (size_t)t0 * cap + q;
      cand_keys[o] = key;
      cand_boxes[o] = box;
    } else {
      atomicOr(status, HDY_STATUS_OVERFLOW);
    }
  };
  auto flush_pending = [&]() {
    if (!p_any) return;
    const int pos = __shfl_sync(0xffffffffu, p_base, p_leader);
    if (p_cand) put(p_tile, pos, p_grp, p_key, p_box);
    p_any = false;
  };

  // phase B: lanes [0, cnt) take the cnt newest entries
  auto drain = [&](int cnt) {
    __syncwarp();
    flush_pending();
    const int e = qn - cnt + lane;
    qn -= cnt;
    bool cand = false;
    uint64_t key = 0;
    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
    int tile = -1;
    if (lane < cnt) {
      const QueueA A = qa[e];
      const QueueB B = qb[e];
      const float p_obj = sigmoidf_ref(B.obj);
      if (p_obj > conf_thres) {  // the reference's own comparison                      utils_general.py:336-337
        tile = B.tile;
        const LevelDev& L = T.lv[B.level];
        const int plane = L.ny * L.nx;
        const int a = B.row / plane, p = B.row - a * plane;
        const int gy = p / L.nx, gx = p - gy * L.nx;
        // xy = (sigmoid*2 - 0.5 + grid) * stride ; wh = (sigmoid*2)^2 * anchor_grid     yolo_head.py:203-204
        const float sx = sigmoidf_ref(A.l0), sy = sigmoidf_ref(A.l1);
        const float sw = sigmoidf_ref(A.l2), sh = sigmoidf_ref(A.l3);
        const float cx = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sx, 2.0f), 0.5f), (float)gx), L.stride);
        const float cy = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sy, 2.0f), 0.5f), (float)gy), L.stride);
        const float tw = __fmul_rn(sw, 2.0f), th = __fmul_rn(sh, 2.0f);
        const float bw = __fmul_rn(__fmul_rn(tw, tw), L.aw[a]), bh = __fmul_rn(__fmul_rn(th, th), L.ah[a]);
        const float hw = __fmul_rn(bw, 0.5f), hh = __fmul_rn(bh, 0.5f);  // xywh2xyxy utils_general.py:121-128
        box = make_float4(__fsub_rn(cx, hw), __fsub_rn(cy, hh), __fadd_rn(cx, hw), __fadd_rn(cy, hh));
        // remove_small_boxes(min_size)                                             utils_general.py:332
        cand = (__fsub_rn(box.z, box.x) >= min_size) && (__fsub_rn(box.w, box.y) >= min_size);
        key = make_key(p_obj, (uint32_t)(L.row_offset + B.row));
      }
    }
    unsigned todo = __ballot_sync(0xffffffffu, cand);
    while (todo) {  // one pass per tile present among the lanes (almost always one)
      const int leader = __ffs(todo) - 1;
      const int t0 = __shfl_sync(0xffffffffu, tile, leader);
      const unsigned grp = __ballot_sync(0xffffffffu, cand && tile == t0);
      if (!p_any) {  // first tile of the batch: reserve now, write at the next phase B
        if (lane == leader) p_base = atomicAdd(counts + t0, __popc(grp));
        p_any = true;
        p_leader = leader;
        p_tile = t0;
        p_grp = grp;
        p_cand = cand && tile == t0;
        p_key = key;
        p_box = box;
      } else {
        int pos = 0;
        if (lane == leader) pos = atomicAdd(counts + t0, __popc(grp));
        pos = __shfl_sync(0xffffffffu, pos, leader);
        if (cand && tile == t0) put(t0, pos, grp, key, box);
      }
      todo &= ~grp;
    }
    __syncwarp();
  };

  int b = 0;
  uint32_t parity = 0;
  for (int k = 0; k < n_my; ++k) {
    const Item w = item_at(gw + k * GW);
    E* sm = reinterpret_cast<E*>(reinterpret_cast<unsigned char*>(bufs) + (size_t)b * buf_bytes);
    const int nfl = w.rows * no;
    const int avail = (nfl * kEsz & ~15) / kEsz;  // elements that arrive through the bulk copy
    while (!mbar_try_wait(&full[b], parity)) {
    }
    if (avail < nfl) {  // last chunk of a level whose size is not a multiple of 16 bytes: patch the <= 3 (7) elements
      if (lane < nfl - avail) sm[avail + lane] = w.src[avail + lane];
      __syncwarp();
    }

    // phase A on all RPL row groups at once (independent LDS + compare + ballot):
    // x < t_lo (or NaN) means sigmoid(x) <= conf for certain.  Passing rows are listed in `pick`.
    int total = 0;
#pragma unroll
    for (int g = 0; g < RPL; ++g) {
      const int rr = g * 32 + lane;
      const bool pass = rr < w.rows && to_f32(sm[rr * no + 4]) >= t_lo;
      const unsigned m = __ballot_sync(0xffffffffu, pass);
      if (pass) pick[total + __popc(m & lt_mask)] = (uint8_t)rr;
      total += __popc(m);
    }
    if (total) {
      __syncwarp();
      const int lrows = T.lv[w.level].rows;
      // survivors of the chunk, 32 at a time: lane j copies the j-th one into the queue
      for (int j0 = 0; j0 < total; j0 += 32) {
        const int j = j0 + lane;
        if (j < total) {
          const int rr = pick[j];
          const E* r = sm + rr * no;
          QueueA A;
          A.l0 = to_f32(r[0]);
          A.l1 = to_f32(r[1]);
          A.l2 = to_f32(r[2]);
          A.l3 = to_f32(r[3]);
          QueueB B;
          B.obj = to_f32(r[4]);
          const int grow = w.grow0 + rr;
          B.tile = grow / lrows;
          B.row = grow - B.tile * lrows;
          B.level = w.level;
          qa[qn + lane] = A;
          qb[qn + lane] = B;
        }
        qn += min(32, total - j0);
        if (qn >= 32) drain(32);
      }
    }
    __syncwarp();  // every lane has read its rows: the buffer may be overwritten
    if (lane == 0 && k + NBUF < n_my) issue(k + NBUF, b);
    if (++b == NBUF) {
      b = 0;
      parity ^= 1u;
    }
  }
  if (qn) drain(qn);
  flush_pending();
}

// The launched shape, measured best on B200 (DESIGN.md 3.5): four streamer warps per CTA with two buffers each, and
// chunks of at most kTmaChunkBytes
constexpr int kTmaWarps = 4, kTmaNbuf = 2;
constexpr int kTmaChunkBytes = 14336;

template <int RPL, bool HALF>
static int launch_tma(const LevelTable& T, const ItemTable& I, int bs, int buf_bytes, int ctas_per_sm, int sm_count,
                      float t_lo, float conf_thres, float min_size, int cap, uint64_t* cand_keys, float* cand_boxes,
                      int32_t* counts, int32_t* status, cudaStream_t stream) {
  const size_t smem = per_warp_bytes(kTmaNbuf, buf_bytes) * kTmaWarps;
  cudaError_t e = cudaFuncSetAttribute(filter_compact_tma_kernel<kTmaWarps, kTmaNbuf, RPL, HALF>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(filter_compact_tma_kernel): %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  const int total = I.begin[T.nl];
  long long grid = (long long)sm_count * ctas_per_sm;
  const long long need = ((long long)total + kTmaWarps - 1) / kTmaWarps;
  if (grid > need) grid = need;
  filter_compact_tma_kernel<kTmaWarps, kTmaNbuf, RPL, HALF><<<(unsigned)grid, kTmaWarps * 32, smem, stream>>>(
      T, I, bs, buf_bytes, t_lo, conf_thres, min_size, cap, cand_keys, reinterpret_cast<float4*>(cand_boxes),
      counts, status);
  return check_launch("hdy_filter_compact_logits(tma)");
}

template <int RPL>
static int launch_tma_rpl(const LevelTable& T, const ItemTable& I, int bs, int buf_bytes, int ctas_per_sm,
                          int sm_count, float t_lo, float conf_thres, float min_size, int cap, uint64_t* cand_keys,
                          float* cand_boxes, int32_t* counts, int32_t* status, cudaStream_t stream) {
  if (T.dtype == HDY_F16)
    return launch_tma<RPL, true>(T, I, bs, buf_bytes, ctas_per_sm, sm_count, t_lo, conf_thres, min_size, cap,
                                 cand_keys, cand_boxes, counts, status, stream);
  return launch_tma<RPL, false>(T, I, bs, buf_bytes, ctas_per_sm, sm_count, t_lo, conf_thres, min_size, cap,
                                cand_keys, cand_boxes, counts, status, stream);
}

// Host side: returns HDY_OK, an error, or 1 when the layout does not meet the bulk-copy alignment rules
// (the caller then uses the generic kernel).
int launch_filter_compact_tma(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no, float conf_thres,
                              float min_size, int cap, uint64_t* cand_keys, float* cand_boxes, int32_t* counts,
                              int32_t* status, cudaStream_t stream) {
  // rows per lane and chunk: 1, 2, 4 or 8, the largest whose chunk stays within kTmaChunkBytes (9 KB chunks at no = 9,
  // 10.5 KB at no = 41: measured best on B200, smaller chunks pay the per-chunk handshake, larger ones leave too few
  // warps per SM)
  const int esz = levels_host[0].dtype == HDY_F16 ? 2 : 4;
  int rpl = kTmaChunkBytes / (32 * no * esz);
  rpl = rpl >= 8 ? 8 : (rpl >= 4 ? 4 : (rpl >= 2 ? 2 : 1));
  const int chunk_rows = 32 * rpl;
  const int buf_bytes = (chunk_rows * no * esz + 127) & ~127;
  const size_t smem = per_warp_bytes(kTmaNbuf, buf_bytes) * kTmaWarps;
  if (smem > 227 * 1024) return 1;
  if (!(conf_thres > 1e-6f && conf_thres < 1.0f - 1e-6f)) return 1;  // logit(conf) is not finite enough
  for (int l = 0; l < nl; ++l)
    if (((uintptr_t)levels_host[l].logits & 15) != 0) return 1;
  LevelTable T;
  int rc = build_level_table(levels_host, nl, na, no, 0, chunk_rows, &T);
  if (rc) return rc;
  T.nc = nc;
  ItemTable I;
  long long run = 0;
  for (int l = 0; l < nl; ++l) {
    I.begin[l] = (int)run;
    run += ((long long)bs * T.lv[l].rows + chunk_rows - 1) / chunk_rows;
    if ((long long)bs * T.lv[l].rows >= (1ll << 31)) return 1;
  }
  if (run >= (1ll << 30)) return 1;
  for (int l = nl; l <= HDY_MAX_LEVELS; ++l) I.begin[l] = (int)run;
  // sigmoid(x) > conf  <=>  x > logit(conf) up to rounding: decide far from the boundary on the logit
  const double lg = log((double)conf_thres / (1.0 - (double)conf_thres));
  const double margin = 1e-4 * (1.0 + fabs(lg));
  const float t_lo = (float)(lg - margin);
  static int sm_count = 0;
  if (!sm_count) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (sm_count <= 0) sm_count = 148;
  }
  int per_sm = (int)((228 * 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);
  if (rpl == 8)
    return launch_tma_rpl<8>(T, I, bs, buf_bytes, per_sm, sm_count, t_lo, conf_thres, min_size, cap, cand_keys,
                             cand_boxes, counts, status, stream);
  if (rpl == 4)
    return launch_tma_rpl<4>(T, I, bs, buf_bytes, per_sm, sm_count, t_lo, conf_thres, min_size, cap, cand_keys,
                             cand_boxes, counts, status, stream);
  if (rpl == 2)
    return launch_tma_rpl<2>(T, I, bs, buf_bytes, per_sm, sm_count, t_lo, conf_thres, min_size, cap, cand_keys,
                             cand_boxes, counts, status, stream);
  return launch_tma_rpl<1>(T, I, bs, buf_bytes, per_sm, sm_count, t_lo, conf_thres, min_size, cap, cand_keys,
                           cand_boxes, counts, status, stream);
}

}  // namespace hdy
