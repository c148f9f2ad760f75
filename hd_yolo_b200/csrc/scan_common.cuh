// Prefix sums and stable stream compaction, shared by the merge, mask and NMS kernels.
//
//   block_exclusive_scan          one value per thread of a CTA (int or long long)
//   block_exclusive_scan_inplace  an int array in shared memory, a run of items per thread
//   scan_carry_kernel             one CTA over any number of values, THREADS x 4 per round, with a carry-in
//   device_exclusive_scan         v(0..n) -> out[0..n) over the device, in place or not, without scratch memory
//   launch_compaction             stable compaction: per-block counts -> their scan -> ballot-and-write
// The producers, accessors and predicates the callers pass are structs; their pointer members are not __restrict__,
// so they read what no kernel of the call writes through __ldg.
#pragma once
#include "hdy_common.cuh"

namespace hdy {

template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// Exclusive scan of one value per thread over a CTA of THREADS threads; all threads call.  Returns the thread's
// exclusive prefix; `total` receives the CTA's sum.  smem: 33 T.
template <typename T, int THREADS>
__device__ __forceinline__ T block_exclusive_scan(T v, T* smem, T& total) {
  static_assert(THREADS % 32 == 0 && THREADS <= 1024, "whole warps, at most 1024 threads");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const T incl = warp_inclusive_scan(v);
  if (lane == 31) smem[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const T s = lane < THREADS / 32 ? smem[lane] : T(0);
    const T t = warp_inclusive_scan(s);
    smem[lane] = t - s;
    if (lane == 31) smem[32] = t;
  }
  __syncthreads();
  const T excl = smem[warp] + incl - v;
  total = smem[32];
  __syncthreads();
  return excl;
}

// Exclusive scan of a[0..len) in place (shared memory), ceil(len / THREADS) consecutive items per thread; returns
// the total.  All threads call; warp_tmp: 33 ints.
template <int THREADS>
__device__ __forceinline__ int block_exclusive_scan_inplace(int* a, int len, int* warp_tmp) {
  const int t = threadIdx.x;
  const int items = (len + THREADS - 1) / THREADS;
  const int b = min(t * items, len), e = min(b + items, len);
  int sum = 0;
  for (int i = b; i < e; ++i) sum += a[i];
  const int lane = t & 31, warp = t >> 5;
  const int incl = warp_inclusive_scan(sum);
  if (lane == 31) warp_tmp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int v = (lane < THREADS / 32) ? warp_tmp[lane] : 0;
    const int s = warp_inclusive_scan(v);
    warp_tmp[lane] = s - v;
    if (lane == 31) warp_tmp[32] = s;
  }
  __syncthreads();
  int run = warp_tmp[warp] + incl - sum;
  for (int i = b; i < e; ++i) {
    const int v = a[i];
    a[i] = run;
    run += v;
  }
  const int total = warp_tmp[32];
  __syncthreads();
  return total;
}

// ------------------------------------------------------------------------------------------------
// device-wide exclusive scan
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024;
constexpr int kCarryItems = 4;  // values per thread and round of scan_carry_kernel

// One CTA scans the n >= 1 values acc.load(0..n) in rounds of kScanThreads * kCarryItems, carrying the running sum
// (from *carry_in, or 0) from round to round: acc.store(i, exclusive prefix) for every i < n, then
// acc.store(n, total).  A thread stores only where it loaded, and every thread reads *carry_in before thread 0 stores
// the total, so acc may store to the values it loads and to *carry_in.
template <typename T, class Acc>
__global__ void __launch_bounds__(kScanThreads) scan_carry_kernel(Acc acc, long long n, const T* carry_in) {
  __shared__ T smem[33];
  T carry = carry_in ? *carry_in : T(0);
  for (long long r = 0; r < n; r += (long long)kScanThreads * kCarryItems) {
    const long long base = r + (long long)threadIdx.x * kCarryItems;
    T v[kCarryItems], s = 0;
#pragma unroll
    for (int k = 0; k < kCarryItems; ++k) {
      v[k] = base + k < n ? acc.load(base + k) : T(0);
      s += v[k];
    }
    T total;
    T run = carry + block_exclusive_scan<T, kScanThreads>(s, smem, total);
#pragma unroll
    for (int k = 0; k < kCarryItems; ++k) {
      if (base + k < n) acc.store(base + k, run);
      run += v[k];
    }
    carry += total;
  }
  if (threadIdx.x == 0) acc.store(n, carry);
}

// scan_carry_kernel over a[i * STRIDE], i < n, in place; the total goes to *total_out (may be NULL)
template <typename T, int STRIDE>
struct StridedSlots {
  T* a;
  long long n;
  T* total_out;
  __device__ T load(long long i) const { return a[i * STRIDE]; }
  __device__ void store(long long i, T x) const {
    if (i < n)
      a[i * STRIDE] = x;
    else if (total_out)
      *total_out = x;
  }
};

// v(i) = a[i]
template <typename T>
struct ArrayValues {
  const T* a;
  __device__ T operator()(long long i) const { return a[i]; }
};

// Pass 1: CTA b scans tile b, the values [b * TILE, (b + 1) * TILE), ITEMS consecutive ones per thread, and stores
// their exclusive prefixes within the tile.  While there are other tiles, the tile's first slot (prefix 0) takes the
// tile's total instead; a single tile is the whole scan, and its total goes to *total_out.
template <typename T, int ITEMS, class V>
__global__ void __launch_bounds__(kScanThreads) scan_tiles_kernel(V v, long long n, T* out, T* total_out) {
  __shared__ T smem[33];
  const long long first = (long long)blockIdx.x * kScanThreads * ITEMS;
  const long long base = first + (long long)threadIdx.x * ITEMS;
  T x[ITEMS], s = 0;
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    x[k] = base + k < n ? v(base + k) : T(0);
    s += x[k];
  }
  T total;
  T run = block_exclusive_scan<T, kScanThreads>(s, smem, total);
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    if (base + k < n) out[base + k] = run;
    run += x[k];
  }
  if (threadIdx.x == 0) {
    if (gridDim.x > 1)
      out[first] = total;
    else if (total_out)
      *total_out = total;
  }
}

// Pass 3: tile b + 1 adds its base, which pass 2 left in its first slot, to its other slots.
template <typename T, int ITEMS>
__global__ void __launch_bounds__(kScanThreads) scan_add_kernel(T* a, long long n) {
  const long long first = (long long)(blockIdx.x + 1) * kScanThreads * ITEMS;
  const T base = a[first];
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    const long long i = first + (long long)k * kScanThreads + threadIdx.x;
    if (i > first && i < n) a[i] += base;
  }
}

// Exclusive scan of v(0..n), n >= 1, into out[0..n); the total goes to *total_out (device, may be NULL).  out may be
// the array v reads: a CTA of a pass reads only what it writes.  Tiles hold kScanThreads * ITEMS values; one tile
// takes one launch, more take three (pass 2 turns the tile totals into tile bases in place).
template <typename T, int ITEMS, class V>
static void device_exclusive_scan(V v, long long n, T* out, T* total_out, cudaStream_t st) {
  constexpr int kTile = kScanThreads * ITEMS;
  const long long nt = (n + kTile - 1) / kTile;
  scan_tiles_kernel<T, ITEMS><<<(unsigned)nt, kScanThreads, 0, st>>>(v, n, out, total_out);
  if (nt == 1) return;
  scan_carry_kernel<T><<<1, kScanThreads, 0, st>>>(StridedSlots<T, kTile>{out, nt, total_out}, nt, (const T*)nullptr);
  scan_add_kernel<T, ITEMS><<<(unsigned)(nt - 1), kScanThreads, 0, st>>>(out, n);
}

// ------------------------------------------------------------------------------------------------
// stable stream compaction
// ------------------------------------------------------------------------------------------------
// The rows [0, f.rows()) for which f.keep holds go to slots 0, 1, ... in row order.  F provides
//   struct Shared;                                      per-CTA state in shared memory
//   void init(Shared&) const;                           all threads call it first; if it writes Shared, it ends
//                                                       in __syncthreads()
//   long long rows() const;
//   bool keep(const Shared&, long long i) const;
//   void emit(const Shared&, long long i, long long slot) const;
// CTAs own contiguous row ranges: count per CTA -> scan of the counts -> every CTA writes its rows in order.
constexpr int kSelThreads = 256;
constexpr int kSelMaxBlocks = 4096;

template <class F>
__global__ void __launch_bounds__(kSelThreads) compact_count_kernel(F f, long long chunk,
                                                                    int* __restrict__ block_counts) {
  __shared__ typename F::Shared sh;
  __shared__ int part[kSelThreads / 32];
  f.init(sh);
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, f.rows());
  int c = 0;
  for (long long i = lo + threadIdx.x; i < hi; i += kSelThreads) c += f.keep(sh, i);
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

template <class F>
__global__ void __launch_bounds__(kSelThreads) compact_write_kernel(F f, long long chunk,
                                                                    const int* __restrict__ block_offsets) {
  __shared__ typename F::Shared sh;
  __shared__ int wcount[kSelThreads / 32];
  f.init(sh);
  const long long lo = (long long)blockIdx.x * chunk, hi = min(lo + chunk, f.rows());
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long running = block_offsets[blockIdx.x];
  for (long long i0 = lo; i0 < hi; i0 += kSelThreads) {
    const long long i = i0 + threadIdx.x;
    const bool k = i < hi && f.keep(sh, i);
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
    if (k) f.emit(sh, i, running + before + __popc(m & ((1u << lane) - 1u)));
    running += total;
    __syncthreads();
  }
}

// Compaction of at most n_max >= 1 rows in three launches.  The rows are cut into at most kSelMaxBlocks ranges, each
// a whole number of CTA widths and at least four; block_scratch holds kSelMaxBlocks ints, *count_out (device)
// receives the number of rows kept.
template <class F>
static void launch_compaction(const F& f, long long n_max, int* block_scratch, int* count_out, cudaStream_t st) {
  long long chunk = (n_max + kSelMaxBlocks - 1) / kSelMaxBlocks;
  chunk = ((chunk + kSelThreads - 1) / kSelThreads) * kSelThreads;
  if (chunk < 4 * kSelThreads) chunk = 4 * kSelThreads;
  const int nblocks = (int)((n_max + chunk - 1) / chunk);
  compact_count_kernel<<<nblocks, kSelThreads, 0, st>>>(f, chunk, block_scratch);
  scan_carry_kernel<int><<<1, kScanThreads, 0, st>>>(StridedSlots<int, 1>{block_scratch, nblocks, count_out},
                                                      (long long)nblocks, (const int*)nullptr);
  compact_write_kernel<<<nblocks, kSelThreads, 0, st>>>(f, chunk, block_scratch);
}

}  // namespace hdy
