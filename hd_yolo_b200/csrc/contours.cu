// Boundary polygons of the cropped bit-packed masks (PackedMasks.contours): every ring of every mask, as the exact
// pixel boundary, with its parent exterior ring for holes.  The contract is in include/hd_yolo_b200.h and DESIGN §3.10;
// in short: rings run along pixel corners with the set pixels on their right (y down), turn right at saddle corners,
// list only the corners where they turn, start at their least corner in (y, x) order and are ordered by that start.
//
// The least corner of a ring is one of two corner patterns, both read off the 2 x 2 pixels around the corner
// (x, y) = the top-left corner of pixel (x, y):
//   A  (x, y) set, (x, y-1) and (x-1, y) unset              -> an exterior ring leaves it heading +x;
//   B  (x, y) unset, (x, y-1), (x-1, y) and (x-1, y-1) set  -> a hole ring leaves it heading +y.
// Every ring has at least one such corner, and may have several (a ring with two "tops").  A candidate corner starts a
// ring iff walking the ring from it meets no smaller corner, so each candidate is walked with an early exit at the
// first smaller corner; no visited-edge state is kept, and nothing is allocated.
//
// Two paths, the same walk:
//   * windows up to kSmallSide on both sides (nuclei, process_mask boxes): one thread per mask, which walks its
//     candidates in raster order and writes each ring as it goes;
//   * larger windows: one CTA per mask (persistent CTAs pick them out of geom).  Threads take (row, word) items in
//     raster order, 256 at a time; a block scan of the rings and vertices each item starts places them.
// A hole's parent: the pixel above the hole's start belongs to the hole's component; from it, go up the column to the
// component's boundary and walk that ring.  If it is a hole of the same component, its start is higher up: repeat.
// Otherwise its start is the exterior ring's, which a binary search over the mask's ring starts (already written, and
// sorted) turns into the ring's index.
#include <climits>

#include "scan_common.cuh"

namespace hdy {

constexpr int kSmallSide = 64;       // windows up to 64 x 64 pixels take the one-thread path
constexpr int kSmallThreads = 128;
constexpr int kLargeThreads = 256;
constexpr int kLargeMaxBlocks = 148 * 4;

// headings, clockwise on screen (y down): 0 = +x, 1 = +y, 2 = -x, 3 = -y.  A right turn is d + 1.
__device__ __forceinline__ int head_dx(int d) { return (d == 0) - (d == 2); }
__device__ __forceinline__ int head_dy(int d) { return (d == 1) - (d == 3); }
// the pixels around a corner, clockwise from the one below right: q = 0 (x, y), 1 (x-1, y), 2 (x-1, y-1), 3 (x, y-1).
// Heading d, the pixel ahead on the right is quadrant d and the one ahead on the left is quadrant d + 3.
__device__ __forceinline__ int quad_dx(int q) { return -(q == 1 || q == 2); }
__device__ __forceinline__ int quad_dy(int q) { return -(q >= 2); }

// One mask's bit plane; pixels outside the window, and padding bits, read as unset.
struct Plane {
  const uint32_t* p;
  int w, h, wpr;
  __device__ bool at(int x, int y) const {
    if ((unsigned)x >= (unsigned)w || (unsigned)y >= (unsigned)h) return false;
    return (__ldg(p + (long long)y * wpr + (x >> 5)) >> (x & 31)) & 1u;
  }
  // pixels 32k .. 32k + 31 of row y (0 outside the window, padding bits cleared); k < wpr
  __device__ uint32_t word(int y, int k) const {
    if ((unsigned)y >= (unsigned)h) return 0u;
    const uint32_t v = __ldg(p + (long long)y * wpr + k);
    const int rem = w - (k << 5);
    return rem >= 32 ? v : v & ((1u << rem) - 1u);
  }
  // candidate start corners among pixels 32k .. 32k + 31 of row y: bit b of .x (pattern A) or .y (pattern B)
  __device__ uint2 candidates(int y, int k) const {
    const uint32_t cur = word(y, k), up = word(y - 1, k);
    const uint32_t cl = k ? word(y, k - 1) : 0u, ul = k ? word(y - 1, k - 1) : 0u;
    const uint32_t left = __funnelshift_l(cl, cur, 1), upleft = __funnelshift_l(ul, up, 1);
    return make_uint2(cur & ~up & ~left, ~cur & up & left & upleft);
  }
};

// Walks the ring through the boundary edge that leaves corner (x0, y0) heading d0, until it is back on that edge.
// visit(x, y, closing) is called at every corner where the ring turns, the corner it closes at last (closing: that
// corner is (x0, y0)); a false return stops the walk, and walk returns false.
template <class Visit>
__device__ bool walk(const Plane& pl, int x0, int y0, int d0, Visit& visit) {
  int x = x0, y = y0, d = d0;
  while (true) {
    x += head_dx(d);
    y += head_dy(d);
    int nd;
    if (!pl.at(x + quad_dx(d), y + quad_dy(d)))
      nd = (d + 1) & 3;                                              // convex corner, or a saddle: turn right
    else if (pl.at(x + quad_dx((d + 3) & 3), y + quad_dy((d + 3) & 3)))
      nd = (d + 3) & 3;                                              // concave corner: turn left
    else
      nd = d;
    const bool closing = x == x0 && y == y0 && nd == d0;
    if (nd != d && !visit(x, y, closing)) return false;
    if (closing) return true;
    d = nd;
  }
}

// Counts the corners of the ring that starts at candidate (x0, y0); stops at the first smaller corner.
struct CountFromStart {
  int x0, y0;
  long long n;
  __device__ bool operator()(int x, int y, bool closing) {
    if (!closing && (y < y0 || (y == y0 && x < x0))) return false;
    ++n;
    return true;
  }
};

// CountFromStart that also writes the corners, in canvas pixels: the start at xy[base], the others after it.  Writes
// stop at `end`, so a walk that turns out not to start a ring stays inside its mask's range.
struct WriteFromStart {
  int x0, y0, gx, gy;
  long long base, end, n;
  int2* xy;
  __device__ bool operator()(int x, int y, bool closing) {
    if (!closing && (y < y0 || (y == y0 && x < x0))) return false;
    const long long at = base + (closing ? 0 : n + 1);
    if (at < end) xy[at] = make_int2(gx + x, gy + y);
    ++n;
    return true;
  }
};

// The least corner of a ring in (y, x) order.
struct LeastCorner {
  int x, y;
  __device__ bool operator()(int cx, int cy, bool) {
    if (cy < y || (cy == y && cx < x)) {
      x = cx;
      y = cy;
    }
    return true;
  }
};

// Parent of the hole ring that starts at (hx, hy) (window pixels): the index of its component's exterior ring among
// rings [r_lo, r_hi) of the mask, whose starts xy[ring_verts[r]] (written by this thread or its CTA) are sorted.
__device__ int hole_parent(const Plane& pl, int hx, int hy, int gx, int gy, const int2* xy, const int64_t* ring_verts,
                           long long r_lo, long long r_hi) {
  int x = hx, y = hy - 1;
  while (true) {
    while (pl.at(x, y - 1)) --y;
    LeastCorner lc{INT_MAX, INT_MAX};
    walk(pl, x, y, 0, lc);                  // the top edge of pixel (x, y), a boundary of the component
    if (pl.at(lc.x, lc.y)) {                // pattern A: the exterior ring
      x = lc.x;
      y = lc.y;
      break;
    }
    x = lc.x;                               // a hole of the component, starting higher up
    y = lc.y - 1;
  }
  const int tx = gx + x, ty = gy + y;
  long long lo = r_lo, hi = r_hi - 1;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    const int2 s = xy[ring_verts[mid]];
    if (s.y < ty || (s.y == ty && s.x < tx))
      lo = mid + 1;
    else
      hi = mid;
  }
  return (int)lo;
}

__device__ __forceinline__ bool is_small(const int4& g) { return g.z <= kSmallSide && g.w <= kSmallSide; }

// ---------------------------------------------------------------------------------------------- one thread per mask
// Sizes pass (FILL false): ring_off[i], vert_off[i] = the mask's rings and corners (scanned afterwards).
// Fill pass: every candidate is walked once, writing as it goes; the next ring overwrites what a candidate that is not
// a start wrote.  Holes get parent -2 until the mask's rings are all written.
template <bool FILL>
__global__ void __launch_bounds__(kSmallThreads) contours_small_kernel(
    const int32_t* __restrict__ geom, const int64_t* __restrict__ offsets, const uint32_t* __restrict__ bits, int K,
    int64_t* ring_off, int64_t* vert_off, int64_t* ring_verts, int32_t* parent, int2* xy) {
  const int i = blockIdx.x * kSmallThreads + threadIdx.x;
  if (FILL && i == 0) ring_verts[ring_off[K]] = vert_off[K];
  if (i >= K) return;
  const int4 g = reinterpret_cast<const int4*>(geom)[i];
  const bool empty = g.z <= 0 || g.w <= 0;
  if (!empty && !is_small(g)) return;                       // contours_large_kernel
  if (empty) {
    if (!FILL) ring_off[i] = vert_off[i] = 0;
    return;
  }
  const Plane pl{bits + offsets[i], g.z, g.w, (g.z + 31) >> 5};
  long long rings = FILL ? ring_off[i] : 0, verts = FILL ? vert_off[i] : 0;
  const long long r_lo = rings, v_end = FILL ? vert_off[i + 1] : 0;
  for (int y = 0; y < pl.h; ++y) {
    for (int k = 0; k < pl.wpr; ++k) {
      const uint2 c = pl.candidates(y, k);
      for (uint32_t m = c.x | c.y; m; m &= m - 1) {
        const int b = __ffs(m) - 1, x = (k << 5) + b;
        const bool ext = (c.x >> b) & 1u;
        if (FILL) {
          WriteFromStart v{x, y, g.x, g.y, verts, v_end, 0, xy};
          if (!walk(pl, x, y, ext ? 0 : 1, v)) continue;
          ring_verts[rings] = verts;
          parent[rings] = ext ? -1 : -2;
          verts += v.n;
        } else {
          CountFromStart v{x, y, 0};
          if (!walk(pl, x, y, ext ? 0 : 1, v)) continue;
          verts += v.n;
        }
        ++rings;
      }
    }
  }
  if (FILL) {
    for (long long r = r_lo; r < rings; ++r) {
      if (parent[r] != -2) continue;
      const int2 s = xy[ring_verts[r]];
      parent[r] = hole_parent(pl, s.x - g.x, s.y - g.y, g.x, g.y, xy, ring_verts, r_lo, rings);
    }
  } else {
    ring_off[i] = rings;
    vert_off[i] = verts;
  }
}

// ---------------------------------------------------------------------------------------------- one CTA per mask
// The rings of one large window.  Thread t of a round takes item (row, word) = round * 256 + t; `starts` marks which of
// its candidates start a ring, found by walking every candidate with the early exit; the fill pass places the item's
// rings with a block scan and walks those again to write them.
template <bool FILL>
__device__ void large_mask(const int4& g, const uint32_t* plane, long long i, int64_t* ring_off, int64_t* vert_off,
                           int64_t* ring_verts, int32_t* parent, int2* xy) {
  __shared__ long long scan_smem[33];
  const Plane pl{plane, g.z, g.w, (g.z + 31) >> 5};
  const long long items = (long long)pl.h * pl.wpr;
  const long long r_lo = FILL ? ring_off[i] : 0, v_lo = FILL ? vert_off[i] : 0;
  long long r_carry = r_lo, v_carry = v_lo;
  for (long long t0 = 0; t0 < items; t0 += kLargeThreads) {
    const long long t = t0 + threadIdx.x;
    long long rings = 0, verts = 0;
    uint32_t starts = 0;
    uint2 c = make_uint2(0u, 0u);
    int y = 0, k = 0;
    if (t < items) {
      y = (int)(t / pl.wpr);
      k = (int)(t - (long long)y * pl.wpr);
      c = pl.candidates(y, k);
      for (uint32_t m = c.x | c.y; m; m &= m - 1) {
        const int b = __ffs(m) - 1, x = (k << 5) + b;
        CountFromStart v{x, y, 0};
        if (walk(pl, x, y, ((c.x >> b) & 1u) ? 0 : 1, v)) {
          starts |= 1u << b;
          ++rings;
          verts += v.n;
        }
      }
    }
    long long r_total, v_total;
    const long long r_base = r_carry + block_exclusive_scan<long long, kLargeThreads>(rings, scan_smem, r_total);
    const long long v_base = v_carry + block_exclusive_scan<long long, kLargeThreads>(verts, scan_smem, v_total);
    if (FILL) {
      long long r = r_base, v0 = v_base;
      for (uint32_t m = starts; m; m &= m - 1) {
        const int b = __ffs(m) - 1, x = (k << 5) + b;
        const bool ext = (c.x >> b) & 1u;
        WriteFromStart v{x, y, g.x, g.y, v0, v0 + (1ll << 62), 0, xy};
        walk(pl, x, y, ext ? 0 : 1, v);
        ring_verts[r] = v0;
        parent[r] = ext ? -1 : -2;
        v0 += v.n;
        ++r;
      }
    }
    r_carry += r_total;
    v_carry += v_total;
  }
  if (!FILL) {
    if (threadIdx.x == 0) {
      ring_off[i] = r_carry;
      vert_off[i] = v_carry;
    }
    return;
  }
  __syncthreads();                                         // every ring start of the mask is written
  for (long long r = r_lo + threadIdx.x; r < r_carry; r += kLargeThreads) {
    if (parent[r] != -2) continue;
    const int2 s = xy[ring_verts[r]];
    parent[r] = hole_parent(pl, s.x - g.x, s.y - g.y, g.x, g.y, xy, ring_verts, r_lo, r_carry);
  }
  __syncthreads();
}

// Persistent CTAs: each round of 256 masks, the large windows among them are listed and taken one after another.
template <bool FILL>
__global__ void __launch_bounds__(kLargeThreads) contours_large_kernel(
    const int32_t* __restrict__ geom, const int64_t* __restrict__ offsets, const uint32_t* __restrict__ bits, int K,
    int64_t* ring_off, int64_t* vert_off, int64_t* ring_verts, int32_t* parent, int2* xy) {
  __shared__ int list[kLargeThreads];
  __shared__ int n_list;
  for (long long i0 = (long long)blockIdx.x * kLargeThreads; i0 < K; i0 += (long long)gridDim.x * kLargeThreads) {
    if (threadIdx.x == 0) n_list = 0;
    __syncthreads();
    const long long i = i0 + threadIdx.x;
    if (i < K) {
      const int4 g = reinterpret_cast<const int4*>(geom)[i];
      if (g.z > 0 && g.w > 0 && !is_small(g)) list[atomicAdd(&n_list, 1)] = (int)i;
    }
    __syncthreads();
    const int n = n_list;
    for (int j = 0; j < n; ++j) {
      const int m = list[j];
      const int4 g = reinterpret_cast<const int4*>(geom)[m];
      large_mask<FILL>(g, bits + offsets[m], m, ring_off, vert_off, ring_verts, parent, xy);
    }
    __syncthreads();
  }
}

static int contour_args_ok(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K,
                           const int64_t* ring_off, const int64_t* vert_off, const char* what) {
  HDY_REQUIRE(K >= 0, "%s: negative K", what);
  HDY_REQUIRE(ring_off && vert_off, "%s: NULL pointer", what);
  if (K > 0) {
    HDY_REQUIRE(geom && offsets && bits, "%s: NULL pointer", what);
    HDY_REQUIRE(((uintptr_t)geom & 15) == 0, "%s: geom must be 16-byte aligned", what);
  }
  return HDY_OK;
}

template <bool FILL>
static void launch_contours(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int64_t* ring_off,
                            int64_t* vert_off, int64_t* ring_verts, int32_t* parent, int2* xy, cudaStream_t st) {
  contours_small_kernel<FILL><<<(unsigned)((K + kSmallThreads - 1) / kSmallThreads), kSmallThreads, 0, st>>>(
      geom, offsets, bits, K, ring_off, vert_off, ring_verts, parent, xy);
  const int blocks = (int)min((long long)kLargeMaxBlocks, ((long long)K + kLargeThreads - 1) / kLargeThreads);
  contours_large_kernel<FILL><<<blocks, kLargeThreads, 0, st>>>(geom, offsets, bits, K, ring_off, vert_off, ring_verts,
                                                                  parent, xy);
}

}  // namespace hdy

using namespace hdy;

extern "C" {

int hdy_mask_contour_sizes(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int64_t* ring_off,
                           int64_t* vert_off, hdy_stream_t stream) {
  int rc = contour_args_ok(geom, offsets, bits, K, ring_off, vert_off, "hdy_mask_contour_sizes");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (K == 0) {
    cudaMemsetAsync(ring_off, 0, sizeof(int64_t), st);
    cudaMemsetAsync(vert_off, 0, sizeof(int64_t), st);
    return check_launch("hdy_mask_contour_sizes");
  }
  launch_contours<false>(geom, offsets, bits, K, ring_off, vert_off, nullptr, nullptr, nullptr, st);
  device_exclusive_scan<int64_t, 4>(ArrayValues<int64_t>{ring_off}, K, ring_off, ring_off + K, st);
  device_exclusive_scan<int64_t, 4>(ArrayValues<int64_t>{vert_off}, K, vert_off, vert_off + K, st);
  return check_launch("hdy_mask_contour_sizes");
}

int hdy_mask_contours(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K,
                      const int64_t* ring_off, const int64_t* vert_off, int64_t* ring_verts, int32_t* parent,
                      int32_t* xy, hdy_stream_t stream) {
  int rc = contour_args_ok(geom, offsets, bits, K, ring_off, vert_off, "hdy_mask_contours");
  if (rc) return rc;
  HDY_REQUIRE(ring_verts, "hdy_mask_contours: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (K == 0) {
    cudaMemsetAsync(ring_verts, 0, sizeof(int64_t), st);
    return check_launch("hdy_mask_contours");
  }
  HDY_REQUIRE(parent && xy, "hdy_mask_contours: NULL pointer");
  HDY_REQUIRE(((uintptr_t)xy & 7) == 0, "hdy_mask_contours: xy must be 8-byte aligned");
  launch_contours<true>(geom, offsets, bits, K, const_cast<int64_t*>(ring_off), const_cast<int64_t*>(vert_off),
                        ring_verts, parent, reinterpret_cast<int2*>(xy), st);
  return check_launch("hdy_mask_contours");
}

}  // extern "C"
