// Morphometry of the cropped bit-packed masks (PackedMasks.measure): area, tight box, first and second moments, the
// 2 x 2 corner-pattern counts (perimeters, Euler number), and the convex hull of the set pixels' unit squares with its
// area, vertex count, perimeter and calipers.  The contract is in include/hd_yolo_b200.h and DESIGN §3.10b.
//
// Everything but the hull is a sum over plane words:
//   * moments: per word, popc and two bit-weight popcount sums (sum of b and of b^2 over the set bits b) -- no loop over
//     set bits;
//   * corner patterns: the 32 corners of a word against the row above, NW/SW neighbours by __funnelshift_l, classified
//     with a half adder of the top pair and one of the bottom pair;
//   * row extremes by ffs / clz.
// The hull of a union of pixel squares has its vertices among the corners (xl, y), (xl, y+1), (xr+1, y), (xr+1, y+1) of
// each row's extreme set pixels.  Per corner row c, the left point is the lesser xl of rows c-1 and c and the right point
// the greater xr+1; Andrew's monotone chain over those (already sorted by y) gives the left and right chains, built by
// two threads of different warps in parallel.  The hull is then: left chain's first point (the least vertex in (y, x)
// order), the right chain top to bottom, the left chain bottom to top -- the exterior rings' rotational sense.  The
// calipers are brute force over (edge, vertex) pairs, lane- or thread-parallel; the perimeter is summed in hull order
// (by one thread, or by a warp whose lanes take the square roots and add them up in order by shuffle), so it is
// reproducible bit for bit.
//
// Two paths:
//   * windows up to 64 x 64 (nuclei, process_mask boxes): one warp per mask, lanes over rows; a row is at most two
//     words, kept in registers, and the row above comes from the neighbouring lane by shuffle, so each plane word is
//     read once;
//   * larger windows, sides up to kMaxSide: one CTA per mask (persistent CTAs pick them out of geom), one warp per row,
//     lanes over words; the row extremes of up to 32 768 rows live in 128 KB of shared memory as two 16-bit values.
// Windows with a side beyond kMaxSide get area -1 and zeros: kMaxSide keeps every sum exact in int64.
#include <climits>

#include "hdy_common.cuh"

namespace hdy {

constexpr int kMaxSide = 32768;
constexpr int kMeasSmallSide = 64;
constexpr int kMeasThreads = 256;
constexpr int kMeasWarps = kMeasThreads / 32;
constexpr int kSmallChain = kMeasSmallSide + 2;      // a chain has at most one point per corner row
// A chain is strictly convex and y-monotone, so its edges are pairwise distinct vectors (a, b), b >= 1.  Their b add up
// to at most h; their x first moves one way and then the other (a left chain bulges left), so their |a| add up to at
// most 2 (w - 1).  With both sides up to kMaxSide, sum(|a| + b) <= 98 302.  There are 2t - 1 vectors with |a| + b = t,
// and the 2 765 shortest already need more than that: a chain has at most 2 765 points.
constexpr int kLargeChain = 2768;
constexpr int kLargeMaxBlocks = 148;
constexpr unsigned kFull = 0xffffffffu;
constexpr unsigned short kEmptyRow = 0xffff;
// How much of the small path runs, for the time breakdown of tools/measure_bench.py (built with
// -DHDY_MEASURE_STAGES=n): 1 the sums and corner patterns, 2 also the two chains, 3 (the library) also the hull, the
// calipers and the perimeter.  Below 3 the hull fields are not written.
#ifndef HDY_MEASURE_STAGES
#define HDY_MEASURE_STAGES 3
#endif

struct MeasureOut {
  int32_t* area;        // [K]
  int32_t* bbox;        // [K, 4]
  int64_t* moments;     // [K, 5]
  int32_t* quads;       // [K, 4]
  int64_t* hull;        // [K, 3]
  double* hull_len;     // [K, 2]
};

// Sum of b and of b^2 over the set bits b of v.
__device__ __forceinline__ int bit_sum1(uint32_t v) {
  return __popc(v & 0xaaaaaaaau) + 2 * __popc(v & 0xccccccccu) + 4 * __popc(v & 0xf0f0f0f0u) +
         8 * __popc(v & 0xff00ff00u) + 16 * __popc(v & 0xffff0000u);
}
__device__ __forceinline__ int bit_sum2(uint32_t v) {
  const uint32_t m[5] = {0xaaaaaaaau, 0xccccccccu, 0xf0f0f0f0u, 0xff00ff00u, 0xffff0000u};
  int s = 0;
#pragma unroll
  for (int a = 0; a < 5; ++a) {
    s += (1 << (2 * a)) * __popc(v & m[a]);                       // b_a^2 = b_a
#pragma unroll
    for (int b = a + 1; b < 5; ++b) s += (1 << (a + b + 1)) * __popc(v & m[a] & m[b]);
  }
  return s;
}

// The corners 32k .. 32k+31 of a corner row: a = the pixel row above (word k, and word k-1 as a_prev), b = the row
// below.  q += n1 (one set), n2 (two sharing an edge), n3 (three), nD (two on a diagonal).
__device__ __forceinline__ void corner_patterns(uint32_t a_prev, uint32_t a, uint32_t b_prev, uint32_t b, int q[4]) {
  const uint32_t ne = a, nw = __funnelshift_l(a_prev, a, 1), se = b, sw = __funnelshift_l(b_prev, b, 1);
  const uint32_t x1 = nw ^ ne, c1 = nw & ne, x2 = sw ^ se, c2 = sw & se;
  const uint32_t odd = x1 ^ x2, pair = c1 | c2, cross = x1 & x2;
  q[0] += __popc(odd & ~pair);
  q[1] += __popc((cross & ~(nw ^ sw)) | (~(x1 | x2) & (c1 ^ c2)));
  q[2] += __popc(odd & pair);
  q[3] += __popc(cross & (nw ^ sw));
}

__device__ __forceinline__ uint32_t pack_pt(int x, int y) { return (uint32_t)x | ((uint32_t)y << 16); }
__device__ __forceinline__ int pt_x(uint32_t p) { return (int)(p & 0xffffu); }
__device__ __forceinline__ int pt_y(uint32_t p) { return (int)(p >> 16); }

// I: int for windows up to 64 x 64 (every product below fits), long long beyond.
template <class I>
__device__ __forceinline__ I cross3(uint32_t o, uint32_t a, uint32_t b) {
  return (I)(pt_x(a) - pt_x(o)) * (pt_y(b) - pt_y(o)) - (I)(pt_y(a) - pt_y(o)) * (pt_x(b) - pt_x(o));
}

// One monotone chain over corner rows ya .. yb (ya = first set row, yb = last set row + 1) of rows[] (xl, xr per pixel
// row, kEmptyRow for none): the left chain keeps strict turns with cross < 0 (y down), the right chain cross > 0.
template <class I>
__device__ __forceinline__ int build_chain(const ushort2* rows, int ya, int yb, bool right, uint32_t* st) {
  int n = 0;
  for (int c = ya; c <= yb; ++c) {
    const ushort2 u = c > ya ? rows[c - 1] : make_ushort2(kEmptyRow, 0);
    const ushort2 d = c < yb ? rows[c] : make_ushort2(kEmptyRow, 0);
    const bool ue = u.x == kEmptyRow, de = d.x == kEmptyRow;
    if (ue && de) continue;
    const int x = right ? max(ue ? 0 : u.y + 1, de ? 0 : d.y + 1) : min(ue ? kMaxSide : u.x, de ? kMaxSide : d.x);
    const uint32_t p = pack_pt(x, c);
    while (n >= 2) {
      const I cr = cross3<I>(st[n - 2], st[n - 1], p);
      if (right ? cr > 0 : cr < 0) break;
      --n;
    }
    st[n++] = p;
  }
  return n;
}

// Hull vertex j in the exterior sense, from the two chains (both top to bottom).
__device__ __forceinline__ uint32_t hull_vertex(const uint32_t* L, const uint32_t* R, int nL, int nR, int j) {
  return j == 0 ? L[0] : j <= nR ? R[j - 1] : L[nL + nR - j];
}

// Edge j of the hull (vertex j to j+1): its term of the doubled shoelace area, the greatest squared distance from its
// first vertex to any vertex, and its caliper width max_v |cross(e, v - a)| / |e|.
template <class I>
__device__ __forceinline__ void edge_calipers(const uint32_t* hull, int n, int j, I& area2, I& d2max, double& width) {
  const uint32_t a = hull[j], b = hull[j + 1 == n ? 0 : j + 1];
  const I ax = pt_x(a), ay = pt_y(a), ex = pt_x(b) - ax, ey = pt_y(b) - ay;
  area2 += ax * pt_y(b) - (I)pt_x(b) * ay;
  I m = 0, d2 = 0;
  for (int v = 0; v < n; ++v) {
    const uint32_t p = hull[v];
    const I dx = pt_x(p) - ax, dy = pt_y(p) - ay;
    const I cr = ex * dy - ey * dx;
    m = max(m, cr < 0 ? -cr : cr);
    d2 = max(d2, dx * dx + dy * dy);
  }
  d2max = max(d2max, d2);
  width = fmin(width, (double)m / sqrt((double)(ex * ex + ey * ey)));
}

__device__ __forceinline__ double edge_length(const uint32_t* hull, int n, int j) {
  const uint32_t a = hull[j], b = hull[j + 1 == n ? 0 : j + 1];
  const long long dx = pt_x(b) - pt_x(a), dy = pt_y(b) - pt_y(a);
  return sqrt((double)(dx * dx + dy * dy));
}

__device__ __forceinline__ double hull_perimeter(const uint32_t* hull, int n) {
  double s = 0.0;
  for (int j = 0; j < n; ++j) s += edge_length(hull, n, j);
  return s;
}

// The same sum, in the same order, by a whole warp: lanes take the square roots, every lane adds them up in order.
__device__ __forceinline__ double hull_perimeter_warp(const uint32_t* hull, int n, int lane) {
  double s = 0.0;
  for (int j0 = 0; j0 < n; j0 += 32) {
    const double len = j0 + lane < n ? edge_length(hull, n, j0 + lane) : 0.0;
    const int m = min(32, n - j0);
    for (int t = 0; t < m; ++t) s += __shfl_sync(kFull, len, t);
  }
  return s;
}

struct Row {
  int area;
  int bbox[4];
  long long mom[5];
  int q[4];
  long long area2, fmax2;
  int verts;
  double perim, fmin;
};

__device__ __forceinline__ void write_row(const MeasureOut& o, long long i, const Row& r) {
  o.area[i] = r.area;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    o.bbox[i * 4 + t] = r.bbox[t];
    o.quads[i * 4 + t] = r.q[t];
  }
#pragma unroll
  for (int t = 0; t < 5; ++t) o.moments[i * 5 + t] = r.mom[t];
  o.hull[i * 3 + 0] = r.area2;
  o.hull[i * 3 + 1] = r.fmax2;
  o.hull[i * 3 + 2] = r.verts;
  o.hull_len[i * 2 + 0] = r.perim;
  o.hull_len[i * 2 + 1] = r.fmin;
}

__device__ __forceinline__ void write_empty(const MeasureOut& o, long long i, int area) {
  Row r{};
  r.area = area;
  write_row(o, i, r);
}

__device__ __forceinline__ long long warp_sum64(long long v) {
#pragma unroll
  for (int s = 16; s; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
  return v;
}
__device__ __forceinline__ long long warp_max64(long long v) {
#pragma unroll
  for (int s = 16; s; s >>= 1) v = max(v, __shfl_xor_sync(kFull, v, s));
  return v;
}
__device__ __forceinline__ double warp_min_f64(double v) {
#pragma unroll
  for (int s = 16; s; s >>= 1) v = fmin(v, __shfl_xor_sync(kFull, v, s));
  return v;
}

__device__ __forceinline__ bool too_large(const int4& g) { return g.z > kMaxSide || g.w > kMaxSide; }
__device__ __forceinline__ bool is_small(const int4& g) { return g.z <= kMeasSmallSide && g.w <= kMeasSmallSide; }

// ---------------------------------------------------------------------------------------------- one warp per mask
// Also writes the rows of empty and too-large windows.  Sums fit int32 here: a 64 x 64 window has sum dx^2 < 2^23.
__global__ void __launch_bounds__(kMeasThreads) measure_small_kernel(const int32_t* __restrict__ geom,
                                                                     const int64_t* __restrict__ offsets,
                                                                     const uint32_t* __restrict__ bits, long long K,
                                                                     MeasureOut o) {
  __shared__ ushort2 s_rows[kMeasWarps][kMeasSmallSide];
  __shared__ uint32_t s_chain[kMeasWarps][2][kSmallChain];
  __shared__ uint32_t s_hull[kMeasWarps][2 * kSmallChain];
  __shared__ int s_n[kMeasWarps][2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * kMeasWarps + warp;
  if (i >= K) return;                                               // uniform per warp
  const int4 g = reinterpret_cast<const int4*>(geom)[i];
  if (g.z <= 0 || g.w <= 0 || too_large(g)) {
    if (lane == 0) write_empty(o, i, g.z > 0 && g.w > 0 ? -1 : 0);
    return;
  }
  if (!is_small(g)) return;                                         // measure_large_kernel
  const int h = g.w, wpr = (g.z + 31) >> 5;
  const uint32_t last = (g.z & 31) ? (1u << (g.z & 31)) - 1u : kFull;
  const uint32_t* p = bits + offsets[i];
  int area = 0, sx = 0, sy = 0, sxx = 0, syy = 0, sxy = 0, q[4] = {0, 0, 0, 0};
  int xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;
  uint32_t up0 = 0, up1 = 0;                                         // row y0 - 1, from lane 31 of the last round
  for (int y0 = 0; y0 <= h; y0 += 32) {                              // corner rows 0 .. h
    const int y = y0 + lane;
    uint32_t w0 = 0, w1 = 0;
    if (y < h) {
      w0 = __ldg(p + y * wpr);
      if (wpr == 2) w1 = __ldg(p + y * wpr + 1) & last;
      else w0 &= last;
    }
    uint32_t a0 = __shfl_up_sync(kFull, w0, 1), a1 = __shfl_up_sync(kFull, w1, 1);
    if (lane == 0) {
      a0 = up0;
      a1 = up1;
    }
    up0 = __shfl_sync(kFull, w0, 31);
    up1 = __shfl_sync(kFull, w1, 31);
    const int c = __popc(w0) + __popc(w1);
    if (c) {
      const int s1 = bit_sum1(w0) + 32 * __popc(w1) + bit_sum1(w1);
      area += c;
      sx += s1;
      sxx += bit_sum2(w0) + 1024 * __popc(w1) + 64 * bit_sum1(w1) + bit_sum2(w1);
      sy += y * c;
      syy += y * y * c;
      sxy += y * s1;
      const int xl = w0 ? __ffs(w0) - 1 : 31 + __ffs(w1), xr = w1 ? 63 - __clz(w1) : 31 - __clz(w0);
      xmin = min(xmin, xl);
      xmax = max(xmax, xr);
      ymin = min(ymin, y);
      ymax = y;
      s_rows[warp][y] = make_ushort2((unsigned short)xl, (unsigned short)xr);
    } else if (y < h) {
      s_rows[warp][y] = make_ushort2(kEmptyRow, 0);
    }
    if (y <= h) {
      corner_patterns(0u, a0, 0u, w0, q);
      corner_patterns(a0, a1, w0, w1, q);
      corner_patterns(a1, 0u, w1, 0u, q);
    }
  }
  Row r{};
  r.area = __reduce_add_sync(kFull, area);
  if (r.area == 0) {                                                // uniform
    if (lane == 0) write_empty(o, i, 0);
    return;
  }
  r.mom[0] = __reduce_add_sync(kFull, sx);
  r.mom[1] = __reduce_add_sync(kFull, sy);
  r.mom[2] = __reduce_add_sync(kFull, sxx);
  r.mom[3] = __reduce_add_sync(kFull, syy);
  r.mom[4] = __reduce_add_sync(kFull, sxy);
#pragma unroll
  for (int t = 0; t < 4; ++t) r.q[t] = __reduce_add_sync(kFull, q[t]);
  const int x0 = (int)__reduce_min_sync(kFull, (unsigned)xmin), y_lo = (int)__reduce_min_sync(kFull, (unsigned)ymin);
  const int x1 = __reduce_max_sync(kFull, xmax) + 1, y_hi = __reduce_max_sync(kFull, ymax) + 1;
  r.bbox[0] = g.x + x0;
  r.bbox[1] = g.y + y_lo;
  r.bbox[2] = g.x + x1;
  r.bbox[3] = g.y + y_hi;
  if (HDY_MEASURE_STAGES == 1) {
    if (lane == 0) write_row(o, i, r);
    return;
  }
  __syncwarp();
  if (lane < 2) s_n[warp][lane] = build_chain<int>(s_rows[warp], y_lo, y_hi, lane == 1, s_chain[warp][lane]);
  __syncwarp();
  const int nL = s_n[warp][0], nR = s_n[warp][1], n = nL + nR;
  if (HDY_MEASURE_STAGES == 2) {
    r.verts = n;
    if (lane == 0) write_row(o, i, r);
    return;
  }
  uint32_t* hull = s_hull[warp];
  for (int j = lane; j < n; j += 32) hull[j] = hull_vertex(s_chain[warp][0], s_chain[warp][1], nL, nR, j);
  __syncwarp();
  int area2 = 0, d2 = 0;
  double width = INFINITY;
  for (int j = lane; j < n; j += 32) edge_calipers<int>(hull, n, j, area2, d2, width);
  r.area2 = __reduce_add_sync(kFull, area2);
  r.fmax2 = __reduce_max_sync(kFull, d2);
  r.fmin = warp_min_f64(width);
  r.verts = n;
  r.perim = hull_perimeter_warp(hull, n, lane);
  if (lane == 0) write_row(o, i, r);
}

// ---------------------------------------------------------------------------------------------- one CTA per mask
struct LargePlane {
  const uint32_t* p;
  int w, h, wpr;
  // pixels 32k .. 32k + 31 of row y (0 outside the window, padding bits cleared)
  __device__ uint32_t word(int y, int k) const {
    if ((unsigned)y >= (unsigned)h || (unsigned)k >= (unsigned)wpr) return 0u;
    const uint32_t v = __ldg(p + (long long)y * wpr + k);
    const int rem = w - (k << 5);
    return rem >= 32 ? v : v & ((1u << rem) - 1u);
  }
};

struct LargeAcc {
  unsigned long long sum[10];        // area, 5 moments, 4 corner patterns
  unsigned long long area2, fmax2, fmin_bits;
  int x0, y0, x1, y1;
};

constexpr size_t kLargeSmem = sizeof(ushort2) * kMaxSide + sizeof(uint32_t) * 4 * kLargeChain;

__device__ __forceinline__ void large_mask(const int4& g, const uint32_t* plane, long long i, const MeasureOut& o, ushort2* rows,
                           uint32_t* chain, uint32_t* hull, LargeAcc& acc, int* s_n) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const LargePlane pl{plane, g.z, g.w, (g.z + 31) >> 5};
  const int cw = (g.z >> 5) + 1;                                    // words of corners 0 .. w
  if (threadIdx.x < 10) acc.sum[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    acc.area2 = acc.fmax2 = 0;
    acc.fmin_bits = __double_as_longlong(INFINITY);
    acc.x0 = acc.y0 = INT_MAX;
    acc.x1 = acc.y1 = -1;
  }
  __syncthreads();
  long long s[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  int xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;
  for (int y = warp; y < pl.h; y += kMeasWarps) {
    int q[4] = {0, 0, 0, 0};
    int xl = INT_MAX, xr = -1;
    long long c = 0, sx = 0;
    for (int k = lane; k < cw; k += 32) {
      const uint32_t cur = pl.word(y, k), prev = pl.word(y, k - 1);
      const uint32_t up = pl.word(y - 1, k), up_prev = pl.word(y - 1, k - 1);
      corner_patterns(up_prev, up, prev, cur, q);
      if (y == pl.h - 1) corner_patterns(prev, cur, 0u, 0u, q);
      if (cur) {
        const long long base = (long long)k << 5, n = __popc(cur), b1 = bit_sum1(cur);
        c += n;
        sx += base * n + b1;
        s[3] += base * base * n + 2 * base * b1 + bit_sum2(cur);
        xl = min(xl, (k << 5) + __ffs(cur) - 1);
        xr = max(xr, (k << 5) + 31 - __clz(cur));
      }
    }
    s[0] += c;
    s[1] += sx;
    s[2] += y * c;
    s[4] += (long long)y * y * c;
    s[5] += y * sx;
#pragma unroll
    for (int t = 0; t < 4; ++t) s[6 + t] += q[t];
    xl = (int)__reduce_min_sync(kFull, (unsigned)xl);
    xr = __reduce_max_sync(kFull, xr);
    if (lane == 0) rows[y] = xr >= 0 ? make_ushort2((unsigned short)xl, (unsigned short)xr) : make_ushort2(kEmptyRow, 0);
    if (xr >= 0) {
      xmin = min(xmin, xl);
      xmax = max(xmax, xr);
      ymin = min(ymin, y);
      ymax = y;
    }
  }
  // s: area, sum dx, sum dy, sum dx^2, sum dy^2, sum dx dy, n1, n2, n3, nD
#pragma unroll
  for (int t = 0; t < 10; ++t) {
    const long long v = warp_sum64(s[t]);
    if (lane == 0) atomicAdd(&acc.sum[t], (unsigned long long)v);
  }
  if (lane == 0 && xmax >= 0) {
    atomicMin(&acc.x0, xmin);
    atomicMax(&acc.x1, xmax + 1);
    atomicMin(&acc.y0, ymin);
    atomicMax(&acc.y1, ymax + 1);
  }
  __syncthreads();
  const long long area = (long long)acc.sum[0];
  if (area == 0) {
    if (threadIdx.x == 0) write_empty(o, i, 0);
    __syncthreads();
    return;
  }
  if (threadIdx.x == 0 || threadIdx.x == 32) {                       // two warps: the chains run side by side
    const int side = threadIdx.x >> 5;
    s_n[side] = build_chain<long long>(rows, acc.y0, acc.y1, side == 1, chain + side * kLargeChain);
  }
  __syncthreads();
  const int nL = s_n[0], nR = s_n[1], n = nL + nR;
  for (int j = threadIdx.x; j < n; j += kMeasThreads) hull[j] = hull_vertex(chain, chain + kLargeChain, nL, nR, j);
  __syncthreads();
  long long area2 = 0, d2 = 0;
  double width = INFINITY;
  for (int j = threadIdx.x; j < n; j += kMeasThreads) edge_calipers<long long>(hull, n, j, area2, d2, width);
  area2 = warp_sum64(area2);
  d2 = warp_max64(d2);
  width = warp_min_f64(width);
  if (lane == 0) {
    atomicAdd(&acc.area2, (unsigned long long)area2);
    atomicMax(&acc.fmax2, (unsigned long long)d2);
    atomicMin(&acc.fmin_bits, (unsigned long long)__double_as_longlong(width));   // widths are >= 0: bits order
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Row r;
    r.area = (int)area;
    r.bbox[0] = g.x + acc.x0;
    r.bbox[1] = g.y + acc.y0;
    r.bbox[2] = g.x + acc.x1;
    r.bbox[3] = g.y + acc.y1;
    r.mom[0] = (long long)acc.sum[1];
    r.mom[1] = (long long)acc.sum[2];
    r.mom[2] = (long long)acc.sum[3];
    r.mom[3] = (long long)acc.sum[4];
    r.mom[4] = (long long)acc.sum[5];
#pragma unroll
    for (int t = 0; t < 4; ++t) r.q[t] = (int)acc.sum[6 + t];
    r.area2 = (long long)acc.area2;
    r.fmax2 = (long long)acc.fmax2;
    r.verts = n;
    r.fmin = __longlong_as_double((long long)acc.fmin_bits);
    r.perim = hull_perimeter(hull, n);
    write_row(o, i, r);
  }
  __syncthreads();
}

// Persistent CTAs: each round of 256 masks, the large windows among them are listed and taken one after another.  The
// shared memory allows one CTA per SM, so the kernel may take the registers of one.
__global__ void __launch_bounds__(kMeasThreads, 1) measure_large_kernel(const int32_t* __restrict__ geom,
                                                                     const int64_t* __restrict__ offsets,
                                                                     const uint32_t* __restrict__ bits, long long K,
                                                                     MeasureOut o) {
  extern __shared__ __align__(16) unsigned char smem[];
  ushort2* rows = reinterpret_cast<ushort2*>(smem);
  uint32_t* chain = reinterpret_cast<uint32_t*>(rows + kMaxSide);
  uint32_t* hull = chain + 2 * kLargeChain;
  __shared__ LargeAcc acc;
  __shared__ int s_n[2];
  __shared__ int list[kMeasThreads];
  __shared__ int n_list;
  for (long long i0 = (long long)blockIdx.x * kMeasThreads; i0 < K; i0 += (long long)gridDim.x * kMeasThreads) {
    if (threadIdx.x == 0) n_list = 0;
    __syncthreads();
    const long long i = i0 + threadIdx.x;
    if (i < K) {
      const int4 g = reinterpret_cast<const int4*>(geom)[i];
      if (g.z > 0 && g.w > 0 && !too_large(g) && !is_small(g)) list[atomicAdd(&n_list, 1)] = (int)i;
    }
    __syncthreads();
    const int n = n_list;
    for (int j = 0; j < n; ++j) {
      const int m = list[j];
      const int4 g = reinterpret_cast<const int4*>(geom)[m];
      large_mask(g, bits + offsets[m], m, o, rows, chain, hull, acc, s_n);
    }
    __syncthreads();
  }
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_mask_measure(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int32_t* area,
                     int32_t* bbox, int64_t* moments, int32_t* quads, int64_t* hull, double* hull_len,
                     hdy_stream_t stream) {
  HDY_REQUIRE(K >= 0, "hdy_mask_measure: negative K");
  if (K == 0) return HDY_OK;
  HDY_REQUIRE(geom && offsets && bits && area && bbox && moments && quads && hull && hull_len,
              "hdy_mask_measure: NULL pointer");
  HDY_REQUIRE(((uintptr_t)geom & 15) == 0, "hdy_mask_measure: geom must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const MeasureOut o{area, bbox, moments, quads, hull, hull_len};
  measure_small_kernel<<<(unsigned)(((long long)K + kMeasWarps - 1) / kMeasWarps), kMeasThreads, 0, st>>>(
      geom, offsets, bits, K, o);
  const cudaError_t e =
      cudaFuncSetAttribute(measure_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLargeSmem);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(measure_large_kernel): %s", cudaGetErrorString(e));
    return HDY_ERR_CUDA;
  }
  const int blocks = (int)min((long long)kLargeMaxBlocks, ((long long)K + kMeasThreads - 1) / kMeasThreads);
  measure_large_kernel<<<blocks, kMeasThreads, kLargeSmem, st>>>(geom, offsets, bits, K, o);
  return check_launch("hdy_mask_measure");
}

}  // extern "C"
