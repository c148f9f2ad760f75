// Prediction <-> ground-truth matching on the device: the step right after the hot path in val_nuclei.run
// (SURVEY 8f rank 2).
//
// Reference: APMeter.add, metayolo/models/metrics.py:270-303 -- predictions sorted by score, a dense
// box_iou(pred[order], gt) matrix (metayolo/models/utils_general.py:247-265), `torch.where(ious >= iouv.min())`,
// the matching pairs sorted by IoU descending.  The reference builds the k x g matrix per image on the host side of a
// D2H copy; here only the matching pairs ever exist:
//   * match_pairs_kernel: one thread per prediction (in score order), ground-truth boxes staged through shared memory
//     in chunks; a pair with iou >= iou_min is appended to the image's pair list as a 64-bit order key
//     (~orderable(iou) << 32 | row-major index r*g + j), so that ONE ascending sort (hdy_nms_tiles with iou_thres = 2:
//     sorts, suppresses nothing) returns the pairs IoU-descending with ties in `torch.where`'s row-major order;
//   * box_iou_kernel: the dense matrix itself, for callers that want it (box_iou is also used on its own).
// IoU arithmetic is the reference's: inter = clamp(min(a2,b2) - max(a1,b1), 0).prod(); iou = inter / (area1 + area2 -
// inter), fp32, one rounding per operation; 0/0 = NaN fails `>=` exactly as in the reference.
#include "match_common.cuh"

namespace hdy {

constexpr int kMatchThreads = 256;

__global__ void __launch_bounds__(kMatchThreads) match_pairs_kernel(
    const float4* __restrict__ pred_boxes, const int32_t* __restrict__ pred_order,
    const int32_t* __restrict__ pred_counts, int P, const float4* __restrict__ gt_boxes,
    const int32_t* __restrict__ gt_counts, int G, float iou_min, int cap, uint64_t* __restrict__ pair_keys,
    float4* __restrict__ pair_boxes, int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  __shared__ float4 gb[kMatchThreads];
  __shared__ float ga[kMatchThreads];
  const int img = blockIdx.y;
  const int k = min(pred_counts[img], P), g = min(gt_counts[img], G);
  const int r = blockIdx.x * kMatchThreads + threadIdx.x;  // rank of the prediction in score order
  if (blockIdx.x * kMatchThreads >= k) return;
  const bool have = r < k;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (have) {
    const int row = pred_order ? pred_order[(size_t)img * P + r] : r;
    a = pred_boxes[(size_t)img * P + row];
  }
  const float area_a = box_area(a);
  for (int j0 = 0; j0 < g; j0 += kMatchThreads) {
    __syncthreads();
    if (j0 + threadIdx.x < g) {
      const float4 b = gt_boxes[(size_t)img * G + j0 + threadIdx.x];
      gb[threadIdx.x] = b;
      ga[threadIdx.x] = box_area(b);
    }
    __syncthreads();
    if (!have) continue;
    const int lim = min(kMatchThreads, g - j0);
    for (int j = 0; j < lim; ++j) {
      const float iou = ref_box_iou(a, area_a, gb[j], ga[j]);
      if (iou >= iou_min) {
        const int pos = atomicAdd(&counts[img], 1);
        if (pos < cap) {
          pair_keys[(size_t)img * cap + pos] = make_key(iou, (uint32_t)r * (uint32_t)g + (uint32_t)(j0 + j));
          pair_boxes[(size_t)img * cap + pos] = a;
        } else {
          atomicOr(status, HDY_STATUS_OVERFLOW);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) box_iou_kernel(const float4* __restrict__ b1, long long n,
                                                      const float4* __restrict__ b2, long long m,
                                                      float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * m) return;
  const long long r = i / m, c = i - r * m;
  const float4 a = b1[r], b = b2[c];
  out[i] = ref_box_iou(a, box_area(a), b, box_area(b));
}

}  // namespace hdy

extern "C" {

int hdy_match_pairs(const float* pred_boxes, const int32_t* pred_order, const int32_t* pred_counts, int bs, int P,
                    const float* gt_boxes, const int32_t* gt_counts, int G, float iou_min, int cap,
                    uint64_t* pair_keys, float* pair_boxes, int32_t* counts, int32_t* status, hdy_stream_t stream) {
  using namespace hdy;
  HDY_REQUIRE(bs >= 0 && P >= 0 && G >= 0 && cap >= 1, "match_pairs: bs=%d P=%d G=%d cap=%d", bs, P, G, cap);
  if (bs == 0 || P == 0 || G == 0) return HDY_OK;
  HDY_REQUIRE(bs <= 65535, "match_pairs: more than 65535 images per call");
  HDY_REQUIRE((long long)P * G < (1ll << 32), "match_pairs: P*G must fit 32 bits (the row-major pair index)");
  HDY_REQUIRE(pred_boxes && pred_counts && gt_boxes && gt_counts && pair_keys && pair_boxes && counts && status,
              "match_pairs: NULL pointer");
  HDY_REQUIRE((((uintptr_t)pred_boxes | (uintptr_t)gt_boxes | (uintptr_t)pair_boxes) & 15) == 0,
              "match_pairs: box arrays must be 16-byte aligned");
  const dim3 grid((unsigned)((P + kMatchThreads - 1) / kMatchThreads), (unsigned)bs);
  match_pairs_kernel<<<grid, kMatchThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(pred_boxes), pred_order, pred_counts, P,
      reinterpret_cast<const float4*>(gt_boxes), gt_counts, G, iou_min, cap, pair_keys,
      reinterpret_cast<float4*>(pair_boxes), counts, status);
  return check_launch("hdy_match_pairs");
}

int hdy_box_iou(const float* box1, int64_t n, const float* box2, int64_t m, float* out, hdy_stream_t stream) {
  using namespace hdy;
  HDY_REQUIRE(n >= 0 && m >= 0, "box_iou: negative size");
  if (n == 0 || m == 0) return HDY_OK;
  HDY_REQUIRE(box1 && box2 && out, "box_iou: NULL pointer");
  HDY_REQUIRE((((uintptr_t)box1 | (uintptr_t)box2) & 15) == 0, "box_iou: box arrays must be 16-byte aligned");
  HDY_REQUIRE(n * m < (1ll << 38), "box_iou: matrix too large");
  const long long total = n * m;
  box_iou_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(box1), n, reinterpret_cast<const float4*>(box2), m, out);
  return check_launch("hdy_box_iou");
}

}  // extern "C"
