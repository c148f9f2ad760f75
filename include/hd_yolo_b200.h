/*
 * hd_yolo_b200 -- C-ABI of the B200 (sm_100a) post-processing hot path.
 *
 * This is the drop-in boundary: plain pointers, sizes and scalars, no torch
 * types.  The reference (impromptuRong/hd_yolo) has no FFI layer of its own --
 * its boundary is a set of Python functions -- so every entry point below
 * names the reference function (file:line, relative to the reference root)
 * whose arithmetic it replaces.  The Python mirror with the reference's
 * call signatures is hd_yolo_b200/ops.py; INTEGRATION.md shows the ctypes
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - every call enqueues work on `stream` and returns without synchronising,
 *     never allocates, never throws;
 *   - return value: HDY_OK, or a negative HDY_ERR_* (argument errors are
 *     detected on the host before anything is launched);
 *   - capacity overflow is reported asynchronously: the kernel sets bit
 *     HDY_STATUS_OVERFLOW in *status (device int32) and `counts` holds the
 *     size that would have been needed;
 *   - fp32 arithmetic in the reference's operation order (no FMA contraction,
 *     IEEE division), int32 indices on device (widened to int64 by the host
 *     mirror where the reference returns int64).
 */
#ifndef HD_YOLO_B200_H_
#define HD_YOLO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HDY_OK 0
#define HDY_ERR_INVALID (-1)   /* bad argument                                  */
#define HDY_ERR_CAPACITY (-2)  /* host-detectable capacity / workspace problem  */
#define HDY_ERR_CUDA (-3)      /* a CUDA runtime call failed (see hdy_last_error) */

#define HDY_STATUS_OVERFLOW 1  /* device status bit: a per-tile candidate list overflowed */
#define HDY_STATUS_ROUNDS 2    /* device status bit: merge rounds budget exhausted        */

#define HDY_MAX_LEVELS 8
#define HDY_MAX_ANCHORS 8
#define HDY_MAX_SCORES 96      /* 1 + nc must not exceed this */

typedef void* hdy_stream_t;    /* a cudaStream_t */

#if defined(__GNUC__)
#define HDY_API __attribute__((visibility("default")))
#else
#define HDY_API
#endif

/* Element type of the head's raw outputs (logits, prototypes).  The reference's GPU default is a half() model
 * (val_nuclei.py:109, 115-116): HDY_F16 inputs are widened to fp32 on load -- every fp16 value is an fp32 value, so
 * the result is exactly that of the fp32 path fed the same (fp16-rounded) numbers; all arithmetic stays fp32. */
#define HDY_F32 0
#define HDY_F16 1

/* One pyramid level of raw head output (Detect.forward, yolo_head.py:141-145). */
typedef struct {
  const void* logits;   /* layout 0: [bs, na, ny, nx, no]   (the permuted tensor the reference decodes)
                           layout 1: [bs, na*no, ny, nx]     (the 1x1 conv's native output, D0 skipped; fp32 only) */
  int32_t ny, nx;
  float stride;                      /* buffer.stride            yolo_head.py:61   */
  float anchor_w[HDY_MAX_ANCHORS];   /* anchor_grid = anchor*stride, pixels  yolo_head.py:427 */
  float anchor_h[HDY_MAX_ANCHORS];
  int32_t dtype;                     /* HDY_F32 / HDY_F16, the same on every level */
} hdy_level_t;

/* Library / build information. */
HDY_API const char* hdy_version(void);
HDY_API const char* hdy_last_error(void);
HDY_API int hdy_device_sm_count(void);

/* ------------------------------------------------------------------ decode */

/* D1: Detect.compute_proposals (yolo_head.py:185-213) + _make_grid (:419-429).
 * out[l] has the layout and shape of levels[l].logits ([bs,na,ny,nx,no]);
 * layout must be 0.  y = sigmoid(x); xy = (y*2 - 0.5 + grid)*stride;
 * wh = (y*2)^2 * anchor_grid; the remaining channels are sigmoid(x). */
HDY_API int hdy_decode_levels(const hdy_level_t* levels_host, int nl, int bs, int na, int no,
                      float* const* out_host, hdy_stream_t stream);

/* D1+D2: decode + level-id column + concat over levels (yolo_head.py:311-312).
 * out: [bs, N, no+1] with N = na * sum(ny*nx); last column = level index. */
HDY_API int hdy_decode_concat(const hdy_level_t* levels_host, int nl, int bs, int na, int no, int layout,
                      float* out, hdy_stream_t stream);

/* ------------------------------------------------- filter + stream compaction */

/* D0..D2 + B1 + the front half of nms_per_image (utils_general.py:327-338), fused:
 * reads raw logits once, keeps rows with sigmoid(obj) > conf_thres whose decoded
 * xyxy box has (x2-x1) >= min_size and (y2-y1) >= min_size, and appends them to the
 * tile's candidate list (unordered; the key carries the row index).
 *   cand_keys  [bs, cap] u64 : (~orderable(score) << 32) | row   -- ascending key == reference order
 *   cand_boxes [bs, cap] f32x4 : xyxy
 *   counts     [bs] i32 : number of candidates found (may exceed cap -> HDY_STATUS_OVERFLOW)
 * Rows have `no` >= 5+nc channels (box 4, obj 1, cls nc, then extra channels such as mask
 * coefficients, which this call ignores).  counts and status must be zeroed by the caller
 * (hdy_zero_i32). */
HDY_API int hdy_filter_compact_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no, int layout,
                              float conf_thres, float min_size, int cap,
                              uint64_t* cand_keys, float* cand_boxes, int32_t* counts, int32_t* status,
                              hdy_stream_t stream);

/* Front half of nms_per_image (utils_general.py:325-338) on already decoded rows
 * preds [bs, N, row_len] = (cx, cy, w, h, obj, cls[nc], extra...). Same outputs as above. */
HDY_API int hdy_filter_compact_preds(const float* preds, int bs, int N, int row_len,
                             float conf_thres, float min_size, int cap,
                             uint64_t* cand_keys, float* cand_boxes, int32_t* counts, int32_t* status,
                             hdy_stream_t stream);

/* Front half of non_max_suppression (utils_general.py:439-491): obj > conf, conf = obj*cls,
 * best class (multi_label == 0: one candidate per row, key index = row) or every class with
 * conf > conf_thres (multi_label != 0: key index = row*nc + cls), optional class filter
 * (class_mask[c] != 0 keeps class c; NULL keeps all).  cand_cls [bs,cap] receives the class
 * as float, cand_boxes the un-offset xyxy box. */
HDY_API int hdy_filter_compact_yolo(const float* prediction, int bs, int N, int nc,
                            float conf_thres, int multi_label, const uint8_t* class_mask, int cap,
                            uint64_t* cand_keys, float* cand_boxes, float* cand_cls,
                            int32_t* counts, int32_t* status, hdy_stream_t stream);

/* ------------------------------------------------------------ per-tile NMS */

/* Scratch bytes hdy_nms_tiles needs for (bs, cap). */
HDY_API size_t hdy_nms_workspace_bytes(int bs, int cap);

/* torchvision.ops.nms semantics per tile (called at utils_general.py:342 and :507):
 * stable descending score order (ties -> lower index first), greedy suppression with
 * iou = inter/(area_a+area_b-inter) > iou_thres in fp32, first max_det survivors.
 * cand_cls may be NULL; otherwise boxes are shifted by cls*class_offset (fp32) before
 * the IoU test (utils_general.py:505-506).
 * max_nms > 0: only the max_nms best-scored candidates enter NMS (utils_general.py:501-502).
 *   keep_idx   [bs, max_det] i32 : key index (row, or row*nc+cls) of survivors, score-descending
 *   keep_slot  [bs, max_det] i32 : candidate slot of each survivor (into cand_* arrays)
 *   keep_box   [bs, max_det] f32x4 : un-offset box of each survivor (may be NULL)
 *   keep_score [bs, max_det] f32 : NMS score of each survivor (may be NULL)
 *   keep_cls   [bs, max_det] f32 : cand_cls of each survivor (may be NULL)
 *   keep_counts[bs] i32
 * Gray zone (keep_fragile non-NULL and gray_eps > 0; used by the whole-slide pipeline): keep_fragile [bs, max_det] u8
 * is set for every survivor that has a neighbour with IoU <= iou_thres here, but whose IoU could exceed iou_thres if
 * every coordinate of both boxes moved by up to gray_eps -- which is what Detect.merge_outputs' `boxes + roi origin`
 * does to them in fp32 (yolo_head.py:455) before Ensemble.merge runs NMS again (yolo.py:195).  Survivors without the
 * flag can never be suppressed by a survivor of their own tile in slide coordinates.  Tiles with more than 4096
 * candidates report every survivor fragile. */
HDY_API int hdy_nms_tiles(const uint64_t* cand_keys, const float* cand_boxes, const float* cand_cls,
                  const int32_t* counts, int bs, int cap, float iou_thres, float class_offset, int max_nms,
                  int max_det, int32_t* keep_idx, int32_t* keep_slot, float* keep_box, float* keep_score,
                  float* keep_cls, int32_t* keep_counts, float gray_eps, uint8_t* keep_fragile, void* workspace,
                  size_t workspace_bytes, hdy_stream_t stream);

/* Debug: when device_buf8 (8 x u64, zeroed by the caller) is non-NULL, the following hdy_nms_tiles calls accumulate
 * into it, over the tiles with at most 4096 candidates: 0 sweeps of the fixed point, SM cycles of 1 sort, 3 binning,
 * 4 pairs, 5 resolve, 6 emit (2 stays 0), and 7 the number of such tiles.  Pass NULL to switch it off (the default).
 * Only records the pointer: nothing is launched or synchronised. */
HDY_API int hdy_debug_nms_phases(uint64_t* device_buf8);

/* Keys for a plain torchvision.ops.nms(boxes, scores, thr) call: scores [bs, seg_len] ->
 * keys [bs, seg_len] with index = position inside the segment. */
HDY_API int hdy_make_keys(const float* scores, int bs, int seg_len, uint64_t* keys, hdy_stream_t stream);

/* ---------------------------------------------------------------- epilogues */

/* Tail of nms_per_image (utils_general.py:343): gather surviving rows of preds.
 *   out_scores [bs, max_det, 1+nc], out_extra [bs, max_det, row_len-5-nc] (may be NULL if no extra) */
HDY_API int hdy_gather_preds(const float* preds, int bs, int N, int row_len, int nc,
                     const int32_t* keep_idx, const int32_t* keep_counts, int max_det,
                     float* out_scores, float* out_extra, hdy_stream_t stream);

/* Scores of surviving rows recomputed from raw logits (sigmoid), + level id + raw extra channels:
 *   out_scores [bs, max_det, 1+nc], out_level [bs, max_det] f32 (may be NULL),
 *   out_extra [bs, max_det, no-5-nc] raw (may be NULL) */
HDY_API int hdy_gather_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no, int layout,
                      const int32_t* keep_idx, const int32_t* keep_counts, int max_det,
                      float* out_scores, float* out_level, float* out_extra, hdy_stream_t stream);

/* S1: Detect.hierarchical_scores (yolo_head.py:473-479) + score/label select (:336-345), in place
 * on scores [bs, max_det, 1+nc].  hier_ops_host = n_ops pairs (dst, src): scores[dst] *= scores[src]
 * applied in order (default tree: (c,0) for c=1..nc).
 *   out_score [bs,max_det] f32, out_label [bs,max_det] i64 (cls+1, or -100 if cls_score <= conf) */
HDY_API int hdy_select_scores(float* scores, const int32_t* keep_counts, int bs, int max_det, int nc,
                      const int32_t* hier_ops_host, int n_ops, float conf_thres,
                      float* out_score, int64_t* out_label, hdy_stream_t stream);

/* hdy_gather_logits + hdy_select_scores in one launch (one warp per survivor, coalesced), for 1 + nc <= 32:
 * out_scores receives the scores AFTER hierarchical_scores, exactly what the two-call sequence leaves there. */
HDY_API int hdy_gather_select_logits(const hdy_level_t* levels_host, int nl, int bs, int na, int nc, int no,
                                     int layout, const int32_t* keep_idx, const int32_t* keep_counts, int max_det,
                                     const int32_t* hier_ops_host, int n_ops, float conf_thres, float* out_scores,
                                     float* out_level, float* out_extra, float* out_score, int64_t* out_label,
                                     hdy_stream_t stream);

/* -------------------------------------------------------------------- masks */

/* M1: mask tail of Detect.compute_outputs (yolo_head.py:332, 346-353) for K detections:
 * out[i] = sigmoid(logits[i, mask_indices[max(labels[i],0)]]), or 0 when that index is < 0.
 *   logits [K, C, M, M] f32, labels [K] i64, mask_indices [nc+1] i64 -> out [K, 1, M, M] f32 */
HDY_API int hdy_mask_select(const float* logits, const int64_t* labels, const int64_t* mask_indices, int K, int C,
                            int M, float* out, hdy_stream_t stream);

/* M2: torchvision paste_masks_in_image(masks, boxes, (H,W), padding) as called at val_nuclei.py:169-176 and
 * evaluation.py:122-123, dense output identical in layout to the reference ([K,1,H,W] f32).
 *   src [K, C, M, M] f32; channel [K] i32 picks the channel per mask (NULL: channel 0; < 0: all-zero mask);
 *   apply_sigmoid != 0 fuses M1's sigmoid (src holds logits). */
HDY_API int hdy_paste_masks(const float* src, const int32_t* channel, const float* boxes, int K, int C, int M,
                            int padding, int apply_sigmoid, int H, int W, float* out, hdy_stream_t stream);

/* Cropped bit-packed layout (M2 + M3 "> 0.5"): geom [K,4] i32 = paste window {x0, y0, w, h} in image pixels,
 * offsets [K+1] i64 = first 32-bit word of each mask (row r of mask i = ceil(w/32) words; bit (x-x0)&31 of
 * word (x-x0)>>5).  hdy_paste_geometry fills geom/offsets (offsets[K] = total words); the caller sizes `bits`
 * from it (or passes an upper bound: masks that do not fit set HDY_STATUS_OVERFLOW in *status). */
HDY_API int hdy_paste_geometry(const float* boxes, const int32_t* channel, int K, int M, int padding, int H, int W,
                               int32_t* geom, int64_t* offsets, hdy_stream_t stream);
HDY_API int hdy_paste_masks_packed(const float* src, const int32_t* channel, const float* boxes,
                                   const int64_t* offsets, int K, int C, int M, int padding, int apply_sigmoid,
                                   int H, int W, uint32_t* bits, int64_t capacity_words, int32_t* status,
                                   hdy_stream_t stream);
/* Expand cropped bit planes to a dense [K, H, W] u8 canvas (verification / visualisation). */
HDY_API int hdy_unpack_masks(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int H,
                             int W, uint8_t* out, hdy_stream_t stream);

/* Boundary polygons of cropped bit planes (PackedMasks.contours, csrc/contours.cu).  Coordinates are canvas pixel
 * corners: pixel (x, y) is the unit square [x, x+1] x [y, y+1], x to the right, y down.  Pixels outside a mask's
 * window are unset; padding bits beyond w are ignored, whatever they hold (as in hdy_mask_areas).
 *   edges     a boundary edge is a unit edge between a set and an unset pixel, directed so that the set pixel lies on
 *             its right as drawn on screen (y down): a top edge runs toward +x;
 *   saddles   at a corner whose 2 x 2 pixels are set only on one diagonal a ring turns right, hugging the pixel it
 *             walks along: set pixels are 4-connected, background pixels 8-connected;
 *   vertices  only the corners where the direction changes, the closing vertex not repeated;
 *   order     each ring starts at its least vertex in (y, x) order (unique within the ring); a mask's rings are
 *             ordered by that start, and no two share one;
 *   sign      the shoelace sum 1/2 sum(x_i y_i+1 - x_i+1 y_i) is positive for exterior rings and negative for holes
 *             (counter-clockwise exteriors read with y up, RFC 7946);
 *   parent    every ring hugs one 4-connected component, which has exactly one exterior ring; parent[r] = -1 for an
 *             exterior ring, else the global index of its component's exterior ring.
 * hdy_mask_contour_sizes: ring_off [K+1], vert_off [K+1] = exclusive scans of each mask's ring and vertex counts, the
 * totals R and V at [K].  hdy_mask_contours then fills ring_verts [R+1] (first vertex of each ring, ring_verts[R] = V),
 * parent [R] (R < 2^31) and xy [V, 2] i32 (8-byte aligned); ring r of mask i is one of ring_off[i] .. ring_off[i+1]-1.
 * A mask is addressed through geom[i] (16-byte aligned) and offsets[i] only.  Any window size works: windows up to
 * 64 x 64 are traced one thread per mask, larger ones one CTA per mask. */
HDY_API int hdy_mask_contour_sizes(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K,
                                   int64_t* ring_off, int64_t* vert_off, hdy_stream_t stream);
HDY_API int hdy_mask_contours(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K,
                              const int64_t* ring_off, const int64_t* vert_off, int64_t* ring_verts, int32_t* parent,
                              int32_t* xy, hdy_stream_t stream);

/* Morphometry of cropped bit planes (PackedMasks.measure, csrc/measure.cu; DESIGN §3.10b).  Pixels, windows and padding
 * bits as for the contours above; (gx, gy, w, h) = geom[i], dx = x - gx and dy = y - gy window-relative pixel indices.
 * Exact fields of mask i (all integers but the two f64 values, whose operation order is fixed):
 *   area [K] i32          set pixels (= hdy_mask_areas)
 *   bbox [K,4] i32        tight box of the set pixels (x0, y0, x1, y1), canvas corners, x1 / y1 exclusive
 *   moments [K,5] i64     sum dx, sum dy, sum dx^2, sum dy^2, sum dx*dy over the set pixels
 *   quads [K,4] i32       over the (w+1)(h+1) corners of the window, the 2 x 2 pixel patterns around the corner
 *                         (outside the window = unset): n1 (one set), n2 (two sharing an edge), n3 (three set), nD (two
 *                         on a diagonal)
 *   hull [K,3] i64        convex_area2 (twice the area of the convex hull of the set pixels' unit squares), feret_max2
 *                         (largest squared distance between two hull vertices), hull_verts (vertices: pixel corners,
 *                         collinear points dropped)
 *   hull_len [K,2] f64    convex_perimeter = sum of sqrt((double)(dx^2 + dy^2)) over the hull's edges in order, starting
 *                         at the least hull vertex in (y, x) order and going in the exterior rings' rotational sense;
 *                         feret_min = min over hull edges e = b - a of (double)max_v |cross(e, v - a)| / sqrt((double)e.e)
 * Empty masks (w or h <= 0, or no set pixel) give 0 in every field.  Window sides up to 32 768 keep every sum exact; a
 * larger window gets area -1 and 0 in every other field.  geom is 16-byte aligned; K = 0 is a no-op.  Windows up to
 * 64 x 64 are measured one warp per mask, larger ones one CTA per mask. */
HDY_API int hdy_mask_measure(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int32_t* area,
                             int32_t* bbox, int64_t* moments, int32_t* quads, int64_t* hull, double* hull_len,
                             hdy_stream_t stream);

/* North-star process_mask (ultralytics/yolov5 v7 utils/segment/general.py::process_mask + crop_mask; the
 * reference itself has no such function): mask = sigmoid(coef . protos), zero outside the box scaled by
 * (mw/iw, mh/ih), optional bilinear upsample (align_corners=False) to (ih, iw), > 0.5.  Batched over tiles:
 *   protos [bs, nm, mh, mw] (proto_dtype: HDY_F32 or HDY_F16), coef [bs, max_det, nm] f32, boxes [bs, max_det, 4]
 *   (image pixels), counts [bs]
 *   dense out [bs, max_det, oh, ow] f32 in {0,1} with (oh,ow) = upsample ? (ih,iw) : (mh,mw).
 * workspace (hdy_process_mask_workspace_bytes(bs, max_det) bytes, may be NULL) enables the two-phase path
 * (csrc/mask_regions.cu: TMA-staged prototypes -> sigmoid patches -> upsample + pack) when nm == 32, mw % 4 == 0 and
 * protos is 16-byte aligned; otherwise, and for boxes wider than 16 proto pixels, the per-detection kernel runs. */
HDY_API size_t hdy_process_mask_workspace_bytes(int bs, int max_det);
HDY_API int hdy_process_mask(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                             const int32_t* counts, int bs, int max_det, int nm, int mh, int mw, int ih, int iw,
                             int upsample, float* out, void* workspace, size_t workspace_bytes, hdy_stream_t stream);
/* Cropped bit-packed variant; geom [bs*max_det, 4], offsets [bs*max_det + 1] as above (slots >= counts are empty).
 * hdy_process_mask_packed takes the geom array hdy_process_mask_geometry wrote; the two-phase path needs it (NULL:
 * the per-detection kernel runs and recomputes the windows).
 * Slide form (row_state / tile_offsets non-NULL): slot d of tile t is row tile_offsets[t] + d of the slide-level
 * arrays (hdy_merge_append); only rows whose verdict row_state[row] is HDY_STATE_KEPT get a window -- Ensemble.merge
 * returns masks[keep] (yolo.py:197-202), so the masks of suppressed duplicates are never computed. */
HDY_API int hdy_process_mask_geometry(const float* boxes, const int32_t* counts, int bs, int max_det, int mh, int mw,
                                      int ih, int iw, int upsample, const uint8_t* row_state,
                                      const int64_t* tile_offsets, int32_t* geom, int64_t* offsets,
                                      hdy_stream_t stream);
/* Slide form, second step: the batch's offsets are moved behind the words of the earlier batches (cursor2: two device
 * int64, read at [parity & 1], the advanced value written to [(parity + 1) & 1]) and every live slot's window and
 * offset are copied to its slide row: geom_rows [n, 4] (window origin shifted by the tile origin rois[t] to slide
 * pixels), off_rows [n].  Run hdy_process_mask_packed afterwards with `bits` = the slide-wide word buffer. */
HDY_API int hdy_process_mask_rows(int32_t* geom, int64_t* offsets, const int32_t* counts, const int64_t* tile_offsets,
                                  const float* rois, int bs, int max_det, int64_t* cursor2, int parity,
                                  int32_t* geom_rows, int64_t* off_rows, hdy_stream_t stream);
HDY_API int hdy_process_mask_packed(const void* protos, int proto_dtype, const float* coef, const float* boxes,
                                    const int32_t* counts, const int32_t* geom, const int64_t* offsets, int bs, int max_det, int nm,
                                    int mh, int mw, int ih, int iw, int upsample, uint32_t* bits,
                                    int64_t capacity_words, int32_t* status, void* workspace, size_t workspace_bytes,
                                    hdy_stream_t stream);

/* ------------------------------------------------------------- coordinates */

/* C1: scale_coords + clip_coords (utils_general.py:161-190), Detect.rescale_outputs (yolo_head.py:465-471) and the
 * `.round()` of evaluation.py:109, IN PLACE on rows [n, row_len] whose first four columns are xyxy.  flags:
 *   1: x -= pad_x, y -= pad_y, then /= gain      2: *= scale      4: clamp x to [0, clip_w], y to [0, clip_h]
 *   8: round half to even.   Steps run in that order, each a separate fp32 operation. */
#define HDY_AFFINE_UNPAD 1
#define HDY_AFFINE_SCALE 2
#define HDY_AFFINE_CLIP 4
#define HDY_AFFINE_ROUND 8
HDY_API int hdy_affine_boxes(float* rows, int64_t n, int row_len, float pad_x, float pad_y, float gain, float scale,
                             float clip_w, float clip_h, int flags, hdy_stream_t stream);

/* -------------------------------------------------------- whole-slide merge */

#define HDY_STATE_UNKNOWN 0     /* only after HDY_STATUS_ROUNDS: not resolved within the round budget */
#define HDY_STATE_KEPT 1
#define HDY_STATE_SUPPRESSED 2
#define HDY_STATE_DROPPED 3     /* score <= conf_thres */

/* T2: Detect.merge_outputs (yolo_head.py:450-463) [+ rescale_outputs (:465-471) when scale != 1]: the detections
 * of a batch of tiles (slot d < counts[t] of tile t) are shifted by the tile origin rois[t] = (x0, y0, x1, y1) and
 * appended, tile by tile in order, to flat slide-level arrays at *cursor (device int64, advanced by the call).
 *   boxes [bs,max_det,4] f32, scores [bs,max_det] f32, labels [bs,max_det] i64, counts [bs] i32, rois [bs,4] f32
 *   out_boxes [capacity,4], out_scores/out_labels/out_tile [capacity] (the last three may be NULL)
 *   tile_offsets [bs+1] i64: first output row of every tile, total in [bs]; out_tile[i] = tile_base + t, or
 *   ~(tile_base + t) (negative) when fragile [bs,max_det] u8 (may be NULL) flags the detection: such rows never take
 *   the interior shortcut of hdy_merge_nms.
 * Rows that do not fit set HDY_STATUS_OVERFLOW in *status. */
HDY_API int hdy_merge_append(const float* boxes, const float* scores, const int64_t* labels, const uint8_t* fragile,
                             const int32_t* counts, const float* rois, int bs, int max_det, int tile_base, float scale,
                             int64_t capacity,
                             float* out_boxes, float* out_scores, int64_t* out_labels, int32_t* out_tile,
                             int64_t* cursor, int64_t* tile_offsets, int32_t* status, hdy_stream_t stream);

/* Largest distance by which a box sticks out of its own tile (atomic max into *margin, which the caller zeroes).
 * n_dev (device int64, may be NULL) holds the live row count; n_max bounds it.  tile_id may hold ~tile for fragile
 * rows.  With far_count non-NULL (device int32, zeroed by the caller), boxes sticking out by more than far_cap are
 * not folded into the margin but listed (far_boxes [far_capacity,4], far_tile [far_capacity]; *far_count may exceed
 * far_capacity: overflow): one huge false positive would otherwise shrink every tile's core. */
HDY_API int hdy_merge_overhang(const float* boxes, const int32_t* tile_id, const float* tile_rois,
                               const int64_t* n_dev, int64_t n_max, float far_cap, const float* far_cap_dev,
                               float* margin, float* far_boxes, int32_t* far_tile, int32_t* far_count,
                               int far_capacity, hdy_stream_t stream);
/* Picks far_cap from the data: *cap_out (device float) = the smallest whole-pixel cap in [min_cap, max_cap] that
 * leaves at most max_far boxes sticking out of their tiles by more than it (max_cap if there is none).  Pass cap_out
 * as far_cap_dev above (it overrides far_cap).  hist: 256 device uint32 of scratch. */
HDY_API int hdy_merge_overhang_cap(const float* boxes, const int32_t* tile_id, const float* tile_rois,
                                   const int64_t* n_dev, int64_t n_max, int max_far, float min_cap, float max_cap,
                                   uint32_t* hist, float* cap_out, hdy_stream_t stream);
/* dirty [n_tiles] u8: 1 for every tile whose window is touched by a listed far-reaching box of another tile (all
 * tiles if the list overflowed).  Rows of dirty tiles never take the interior shortcut. */
HDY_API int hdy_merge_dirty_tiles(const float* far_boxes, const int32_t* far_tile, const int32_t* far_count,
                                  int far_capacity, const float* tile_rois, int n_tiles, uint8_t* dirty,
                                  hdy_stream_t stream);

/* T3: Ensemble.merge (yolo.py:165-204): keep scores > conf_thres, class-agnostic greedy NMS
 * (torchvision.ops.nms semantics: score-descending, ties by lower index, IoU > iou_thres in fp32) over all n rows.
 * Sparse and exact: boxes are binned by centre, verdicts are resolved as a fixed point in at most max_rounds
 * rounds (HDY_STATUS_ROUNDS in *status if the budget was too small; call again with more).
 *   state [n] u8 receives HDY_STATE_* per row.
 * Optional shortcut (tile_id, tile_cores [n_tiles,4], margin all non-NULL; tile_dirty [n_tiles] optional): a row
 * with tile_id >= 0 whose box lies strictly inside its tile's core shrunk by *margin, in a tile that is not dirty, is
 * KEPT without any pair test.  Exact when the rows that can be suppressed by a survivor of their OWN tile in slide
 * coordinates carry a negative tile_id (hdy_nms_tiles' gray-zone flags -> hdy_merge_append) -- see DESIGN.md 3.5;
 * pass NULL for the unconditional path. */
HDY_API size_t hdy_merge_workspace_bytes(int64_t n_max);
HDY_API int hdy_merge_nms(const float* boxes, const float* scores, const int32_t* tile_id, const float* tile_cores,
                          const uint8_t* tile_dirty, const float* margin, const int64_t* n_dev, int64_t n_max,
                          float conf_thres,
                          float iou_thres, int max_rounds, uint8_t* state, int32_t* status, void* workspace,
                          size_t workspace_bytes, hdy_stream_t stream);

/* hdy_merge_nms in steps, for the multi-GPU seam exchange below: after hdy_seam_build, hdy_merge_rounds runs rounds
 * [first_round, first_round + n_rounds) of the fixed point (at most 64 in all) on the workspace, and hdy_merge_finish
 * writes state [n_max] (rows not resolved by then: HDY_STATE_UNKNOWN and HDY_STATUS_ROUNDS in *status). */
HDY_API int hdy_merge_rounds(void* workspace, int64_t n_max, float iou_thres, int first_round, int n_rounds,
                             hdy_stream_t stream);
HDY_API int hdy_merge_finish(void* workspace, const int64_t* n_dev, int64_t n_max, uint8_t* state, int32_t* status,
                             hdy_stream_t stream);

/* Multi-GPU form of T3 (the reference runs Ensemble.merge, yolo.py:165-204, on one device; here every rank owns a band
 * of tile rows and only detections near a band boundary are exchanged).  Everything variable-sized travels in
 * FIXED-SIZE blocks whose fill counts stay on the device, so the host issues
 *     summary -> [all-gather] -> select -> [all-gather] -> scatter, dirty_tiles, build
 *     -> { rounds -> export -> [all-gather] -> import } x 2 -> rounds -> finish
 * without reading anything back in between (hd_yolo_b200/dist.py).  Blocks are arrays of 32-bit words:
 *   summary block  [HDY_SEAM_HDR_WORDS + far_cap * HDY_SEAM_FAR_WORDS]:
 *       [0..3] bounding rectangle of the rank's detections (f32 x1,y1,x2,y2; inverted when there are none)
 *       [4] largest overhang of a non-far box over its tile (f32)   [5] far-list length (> far_cap: overflowed)
 *       [6..7] number of own rows (i64)   then per far-reaching box: f32 box x4, i32 GLOBAL tile, 3 pad words
 *   payload block  [HDY_SEAM_HDR_WORDS + seam_cap * HDY_SEAM_ROW_WORDS]:
 *       [0] number of seam rows (> seam_cap: overflowed)   then per seam row (ascending own row): box bits x4, score
 *       bits, index in the slide-wide concatenation (low 32 bits)
 *   meta [HDY_SEAM_META_WORDS] i32, written by hdy_seam_scatter: [0..1] own rows + replicas (i64), [2] largest margin of
 *       any rank (f32), [3] global index of own row 0, [4] flags (1: a payload overflowed, 2: replicas did not fit,
 *       4: a far list overflowed -- all tiles dirty, 8: 2^32 rows or more), [5] far boxes listed, [6..7] spare (the
 *       host mirror parks hdy_merge_finish's status and the survivor count there), [8..15] "a seam row is still
 *       undecided" per exchange (index mod 8), [16..16+world] first replica slot of every rank, [88] own seam rows. */
#define HDY_SEAM_HDR_WORDS 16
#define HDY_SEAM_FAR_WORDS 8
#define HDY_SEAM_ROW_WORDS 6
#define HDY_SEAM_META_WORDS 96
#define HDY_SEAM_MAX_WORLD 64
#define HDY_SEAM_FLAG_PAYLOAD_OVERFLOW 1
#define HDY_SEAM_FLAG_REPLICA_OVERFLOW 2
#define HDY_SEAM_FLAG_FAR_OVERFLOW 4
#define HDY_SEAM_FLAG_TOO_MANY_ROWS 8
/* This rank's summary block.  margin / far_* are what hdy_merge_overhang wrote (far_tile local: tile_base is added). */
HDY_API int hdy_seam_summary(const float* boxes, int64_t n_local, const float* margin, const float* far_boxes,
                             const int32_t* far_tile, const int32_t* far_count, int far_list_capacity, int tile_base,
                             int far_cap, int32_t* block, hdy_stream_t stream);
/* Own rows whose box touches (closed intervals) the rectangle of another rank that has rows: sel [seam_cap] i32 (own
 * row of payload row k) and this rank's payload block.  summaries = the all-gathered summary blocks [world][..];
 * block_scratch: 4097 device int32. */
HDY_API int hdy_seam_select(const float* boxes, const float* scores, int64_t n_local, const int32_t* summaries,
                            int world, int rank, int far_cap, int seam_cap, int32_t* sel, int32_t* block,
                            int32_t* block_scratch, hdy_stream_t stream);
/* The other ranks' seam rows become replicas behind the own rows: boxes / scores rows [n_local, n_local + R) (R <=
 * rep_cap), rep_gidx [rep_cap]; fills meta.  payloads = the all-gathered payload blocks. */
HDY_API int hdy_seam_scatter(const int32_t* payloads, const int32_t* summaries, int world, int rank, int far_cap,
                             int seam_cap, int64_t n_local, int64_t rep_cap, float* boxes, float* scores,
                             uint32_t* rep_gidx, int32_t* meta, hdy_stream_t stream);
/* hdy_merge_dirty_tiles over every rank's far list (global tile ids, tile_rois of the whole slide). */
HDY_API int hdy_seam_dirty_tiles(const int32_t* summaries, int world, int far_cap, const float* tile_rois, int n_tiles,
                                 uint8_t* dirty, hdy_stream_t stream);
/* First step of the merge (as hdy_merge_nms, with its conf_thres / iou_thres / interior shortcut) over the own rows
 * [0, n_local) and the replicas behind them; the replicas take part in every pair test, but their verdicts are only
 * ever imported.  Row count, margin and the global index of own row 0 are read from meta; a row's global index
 * (replicas: rep_gidx) breaks score ties exactly as the single-device call does.  tile_id [n_local] holds LOCAL tile
 * ids (tile_id + tile_base indexes tile_cores / tile_dirty, which cover the whole slide).  workspace:
 * hdy_merge_workspace_bytes(n_max) bytes, kept for the later steps. */
HDY_API int hdy_seam_build(const float* boxes, const float* scores, const uint32_t* rep_gidx, const int32_t* meta,
                           const int32_t* tile_id, int tile_base, const float* tile_cores, const uint8_t* tile_dirty,
                           int64_t n_max, int64_t n_local, float conf_thres, float iou_thres, uint8_t* state,
                           void* workspace, size_t workspace_bytes, hdy_stream_t stream);
/* Verdicts of the own seam rows (out [seam_cap] u8, payload order) / of the replicas from the all-gathered verdicts
 * (states [world][seam_cap]); import also raises meta[8 + exchange % 8] while any rank's seam row is undecided. */
HDY_API int hdy_seam_export(void* workspace, int64_t n_max, const uint8_t* state, const int32_t* sel,
                            const int32_t* my_block, int seam_cap, uint8_t* out, hdy_stream_t stream);
HDY_API int hdy_seam_import(void* workspace, int64_t n_max, int64_t n_local, const uint8_t* states,
                            const int32_t* payloads, int32_t* meta, int world, int rank, int seam_cap, int exchange,
                            hdy_stream_t stream);

/* Survivors in the reference's order (`nms(...)[:max_det]`, yolo.py:195): select_ordered -> sort_keys_bytes ->
 * gather.  select_ordered writes one 64-bit order key (~orderable(score) << 32 | row) per KEPT row, in ROW order, and
 * their number (block_scratch: 4096 device int32).  sort_keys_bytes is a stable ascending LSD radix sort of the bytes
 * [first_byte, first_byte + n_bytes) of each key (one pass of 8 bits per byte; n_bytes even; result in `keys`, `tmp`
 * is scratch of the same size): first_byte = 4, n_bytes = 4 sorts the score half alone and leaves ties in row order,
 * i.e. score-descending, ties by lower row.  gather emits the first max_det rows. */
HDY_API int hdy_merge_select_ordered(const uint8_t* state, const float* scores, const int64_t* n_dev, int64_t n_max,
                                     uint64_t* keys, int32_t* count, int32_t* block_scratch, hdy_stream_t stream);
HDY_API size_t hdy_sort_workspace_bytes(int64_t n_max);
HDY_API int hdy_sort_keys_bytes(uint64_t* keys, uint64_t* tmp, const int32_t* n_dev, int64_t n_max, int first_byte,
                                int n_bytes, void* workspace, size_t workspace_bytes, hdy_stream_t stream);
HDY_API int hdy_merge_gather(const uint64_t* keys, const int32_t* count, int64_t max_det, const float* boxes,
                             const float* scores, const int64_t* labels, int64_t* out_idx, float* out_boxes,
                             float* out_scores, int64_t* out_labels, int32_t* out_count, hdy_stream_t stream);

/* ------------------------------------------------- hnet multi-level heads (H1-H3) */

/* H1: torchvision BoxCoder.decode_single, as reached from hnet/detection/mask_rcnn.py:67 (RPN, weights 1,1,1,1) and
 * :192 (RoIHeads.postprocess_detections, weights 10,10,5,5).  deltas [R, C*4], boxes [boxes_rows, 4] (row r of the
 * deltas uses boxes[r % boxes_rows]: the anchors are shared by the images of a batch) -> out [R, C, 4] xyxy.
 * xform_clip = log(1000/16).  All three arrays 16-byte aligned. */
HDY_API int hdy_rcnn_decode(const float* deltas, const float* boxes, int64_t R, int C, int64_t boxes_rows, float wx,
                            float wy, float ww, float wh, float xform_clip, float* out, hdy_stream_t stream);

/* F.softmax(class_logits, -1) of RoIHeads.postprocess_detections: [R, C] -> [R, C]. */
HDY_API int hdy_softmax_rows(const float* logits, int64_t R, int C, float* out, hdy_stream_t stream);

/* H3 front half (torchvision roi_heads.py postprocess_detections): clip to the image, drop the background column,
 * one candidate per (row, class >= 1) with score > score_thresh whose clipped box has both sides >= min_size.
 *   pred_boxes [R, C, 4], scores [R, C], row_offsets [bs+1] i32 (rows of image i = [row_offsets[i], row_offsets[i+1])),
 *   img_wh [bs, 2] f32 (width, height).  Candidate lists as for hdy_nms_tiles; key index = position in torchvision's
 *   flattened arrays ((row - row0) * (C-1) + class - 1), cand_cls = class.
 *   per_class_tiles != 0: list of (image i, class c) is tile i*(C-1) + c-1 (class-separated NMS, the "vanilla"
 *   batched_nms); 0: one list per image (use hdy_nms_tiles' class_offset for the coordinate trick). */
HDY_API int hdy_rcnn_filter_compact(const float* pred_boxes, const float* scores, const int32_t* row_offsets,
                                    const float* img_wh, int bs, int64_t R, int C, float score_thresh, float min_size,
                                    int per_class_tiles, int cap, uint64_t* cand_keys, float* cand_boxes,
                                    float* cand_cls, int32_t* counts, int32_t* status, hdy_stream_t stream);

/* H2 (torchvision rpn.py filter_proposals), step 1: one 64-bit key per anchor so that ONE ascending sort
 * (hdy_sort_keys_bytes over all eight bytes) leaves every (image, level) segment in place, best objectness logit first, ties by lower anchor.
 *   objectness [N, A] logits, level_sizes_host [nl] anchors per level (sum = A, each <= 262144). */
HDY_API int hdy_rpn_level_keys(const float* objectness, int N, int A, const int32_t* level_sizes_host, int nl,
                               uint64_t* keys, hdy_stream_t stream);
/* step 2: the first pre_nms_top_n keys of every segment -> sigmoid, clip, remove_small_boxes(min_size),
 * score >= score_thresh -> candidate lists (key index = position in the image's top-k concatenation, cand_cls = level).
 *   proposals [N, A, 4]; per_level_tiles as above (tile = image*nl + level). */
HDY_API int hdy_rpn_topk_compact(const uint64_t* sorted_keys, const float* proposals, int N, int A,
                                 const int32_t* level_sizes_host, int nl, int pre_nms_top_n, const float* img_wh,
                                 float min_size, float score_thresh, int per_level_tiles, int cap,
                                 uint64_t* cand_keys, float* cand_boxes, float* cand_cls, int32_t* counts,
                                 int32_t* status, hdy_stream_t stream);

/* Survivors of `group` consecutive class/level tiles (outputs of hdy_nms_tiles) -> one candidate list per image, for
 * the final score-ordered cut (`keep[:post_nms_top_n]` / `[:detections_per_img]`): run hdy_nms_tiles on it with
 * iou_thres = 2, which suppresses nothing and only sorts and caps. */
HDY_API int hdy_regroup_kept(const int32_t* keep_idx, const float* keep_box, const float* keep_score,
                             const float* keep_cls, const int32_t* keep_counts, int n_tiles, int group, int max_det,
                             int cap, uint64_t* cand_keys, float* cand_boxes, float* cand_cls, int32_t* counts,
                             int32_t* status, hdy_stream_t stream);

/* ------------------------------------------------- next rows (SURVEY 8f): RoIAlign in front of the mask head */

/* One pyramid level of mask features (the `features` list of Detect.compute_outputs, yolo_head.py:301, after the
 * `seg` convs): [bs, channels, h, w] fp32, spatial_scale = 1 / stride. */
typedef struct {
  const float* data;
  int32_t h, w;
  float spatial_scale;
} hdy_feature_level_t;

/* f1: Detect.multiscale_roi_align (yolo_head.py:279-299) = torchvision.ops.roi_align per level + scatter, in one
 * launch.  rois [K, 5] = (batch index, x1, y1, x2, y2) in image pixels; level_of [K] = the level id column nms_per_image
 * carries in 'extra' (float; NULL with nl == 1: plain roi_align); out [K, channels, pooled, pooled].  RoIs whose level
 * id is not an integer in [0, nl) stay zero, as rows of the reference's zero-initialised `result` do.
 * sampling_ratio in [1, 4] (reference: 2), pooled in [1, 16] (reference: mask_output_size // 2 = 14), aligned as in
 * torchvision (reference: False).  fp32, torchvision's CPU operation order, no FMA contraction. */
HDY_API int hdy_multiscale_roi_align(const hdy_feature_level_t* levels_host, int nl, int bs, int channels,
                                     const float* rois, const float* level_of, int64_t K, int pooled,
                                     int sampling_ratio, int aligned, float* out, hdy_stream_t stream);

/* f1 on the tensor cores (tcgen05.mma.kind::tf32, accumulators in TMEM): same arguments and result layout, but the
 * bilinear sampling + averaging of a RoI is evaluated as the [pooled^2 x 36] x [36 x channels] product of its tap
 * weights with its <= 6 x 6 feature window, in 3xTF32 (split operands, fp32 accumulation): results agree with
 * hdy_multiscale_roi_align to ~1e-6 relative to the window's magnitude instead of bit for bit (the north star's
 * tolerance for box-derived quantities is 1e-5).  RoIs whose taps span more than 6 x 6 feature pixels, and rows the
 * reference leaves zero, are listed in `fallback` and computed by the exact kernel in the same call.
 *   channels_last != 0: the feature maps are [bs][h][w][channels] in memory (torch.channels_last) -- the faster form:
 *   a window row is contiguous, one TMA request per 128 bytes.  channels must be a multiple of 64; pooled <= 14 (larger outputs run the exact kernel); fallback [K + 1] int32 scratch ([0] = number of listed RoIs afterwards). */
HDY_API int hdy_multiscale_roi_align_tf32x3(const hdy_feature_level_t* levels_host, int nl, int bs, int channels,
                                            int channels_last, const float* rois, const float* level_of, int64_t K,
                                            int pooled, int sampling_ratio, int aligned, float* out, int32_t* fallback,
                                            hdy_stream_t stream);

/* f2: the matching step of APMeter.add (metayolo/models/metrics.py:270-303) without the dense k x g matrix.
 *   pred_boxes [bs, P, 4], pred_order [bs, P] i32 (rank in score order -> row; NULL: rows are already in order),
 *   pred_counts [bs], gt_boxes [bs, G, 4], gt_counts [bs]; every pair with box_iou >= iou_min (utils_general.py:
 *   247-265 arithmetic) is appended to image i's list: pair_keys [bs, cap] = ~orderable(iou) << 32 | (rank * g_i + j),
 *   pair_boxes [bs, cap, 4] (the prediction's box), counts [bs] (zeroed by the caller; holds the needed size on
 *   overflow, *status gets HDY_STATUS_OVERFLOW).  Sorting a list ascending (hdy_nms_tiles with iou_thres = 2) yields
 *   `sort(ious[where(ious >= iou_min)], descending=True)` with ties in row-major order.  P * G < 2^32. */
HDY_API int hdy_match_pairs(const float* pred_boxes, const int32_t* pred_order, const int32_t* pred_counts, int bs,
                            int P, const float* gt_boxes, const int32_t* gt_counts, int G, float iou_min, int cap,
                            uint64_t* pair_keys, float* pair_boxes, int32_t* counts, int32_t* status,
                            hdy_stream_t stream);

/* box_iou (metayolo/models/utils_general.py:247-265): out [n, m] fp32, 0/0 = NaN as in the reference. */
HDY_API int hdy_box_iou(const float* box1, int64_t n, const float* box2, int64_t m, float* out, hdy_stream_t stream);

/* f2 by mask IoU (APMeter.add(..., iou_type='masks'), metrics.py:270-303), over the cropped bit-packed layout above.
 * A pixel is set iff its value is > 0.5 (HDY_F32, HDY_F16) or nonzero (HDY_U8: uint8 or bool masks).
 * Dense [K, H, W] masks (H * W < 2^31) -> bit planes with TIGHT windows (bounding rectangle of the set pixels; an empty
 * mask gets w = h = 0): hdy_pack_masks_geometry fills geom [K,4] (16-byte aligned) and offsets [K+1] (offsets[K] =
 * total words), hdy_pack_masks writes `bits` (padding bits beyond w are zero; masks that do not fit capacity_words set
 * HDY_STATUS_OVERFLOW in *status). */
#define HDY_U8 2
HDY_API int hdy_pack_masks_geometry(const void* masks, int dtype, int K, int H, int W, int32_t* geom, int64_t* offsets,
                                    hdy_stream_t stream);
HDY_API int hdy_pack_masks(const void* masks, int dtype, int K, int H, int W, const int32_t* geom,
                           const int64_t* offsets, uint32_t* bits, int64_t capacity_words, int32_t* status,
                           hdy_stream_t stream);
/* areas [K] i32: set pixels per mask.  The bits beyond w in each row's last word are ignored, whatever they hold. */
HDY_API int hdy_mask_areas(const int32_t* geom, const int64_t* offsets, const uint32_t* bits, int K, int32_t* areas,
                           hdy_stream_t stream);
/* The mask form of hdy_match_pairs for one image.  Both mask sets lie on one canvas (the caller checks); areas from
 * hdy_mask_areas; pred_order [P] i32 (rank in score order -> row; NULL: rows are already in order).  inter = pixels
 * set in both, union = area_p + area_g - inter, iou = float(inter) / float(union) (round to nearest, 0/0 = NaN).
 * Two phases: the pairs whose windows overlap and whose IoU bound float(min(overlap, area_p, area_g)) / float(union)
 * reaches iou_min go to cand [cand_cap] (u32 rank * G + j; counts[1] = their number), then every candidate's
 * intersection is counted exactly and the pairs with iou >= iou_min are appended to pair_keys [cap] as in
 * hdy_match_pairs (counts[0]).  counts [2] is zeroed by the caller; either list overflowing sets HDY_STATUS_OVERFLOW
 * in *status and its count holds the size needed (call again: cand_cap >= counts[1] and cap >= counts[0]).
 * iou_min > 0 (pairs of disjoint masks are never listed); P * G < 2^32.  Cost O(P * G) window tests per image. */
HDY_API int hdy_match_mask_pairs(const int32_t* pred_geom, const int64_t* pred_offsets, const uint32_t* pred_bits,
                                 const int32_t* pred_areas, const int32_t* pred_order, int P, const int32_t* gt_geom,
                                 const int64_t* gt_offsets, const uint32_t* gt_bits, const int32_t* gt_areas, int G,
                                 float iou_min, int cand_cap, uint32_t* cand, int cap, uint64_t* pair_keys,
                                 int32_t* counts, int32_t* status, hdy_stream_t stream);

/* f2 at region and slide scale (match_predictions(..., binned=True)): the pairs of hdy_match_pairs /
 * hdy_match_mask_pairs, bit for bit, without their P * G < 2^32 limit or their O(P * G) work: P, G < 2^31 and fewer
 * than 2^31 pairs (candidates, for masks).  iou_min > 0.  The ground truth is binned into a uniform grid; a pair is
 * tested only in the cell holding (max(x0_p, x0_g), max(y0_p, y0_g)), so each pair is seen exactly once.  Rectangles:
 * boxes [n, 4] xyxy fp32 (rows with a non-finite coordinate or without positive width and height match nothing and are
 * never binned) or mask windows geom [n, 4] {x0, y0, w, h} (empty windows likewise).  All arrays 16-byte aligned where
 * they hold rectangles.  Grid: cell (cx, cy) of a point is clamp(floor((x - ox) * inv_cell), 0, nx - 1) (same in y),
 * evaluated in fp32; any grid gives the same pairs, the grid only sets the cost.
 *
 * bin_stats: stats [6] u64 = orderable_u32 of min x0, min y0, max x1, max y1 of the valid ground truth (x1, y1: the last
 * pixel of a window), their number, and the sum of their sides max(w, h) in 1/16 px -- what the caller picks the grid
 * from.  Pass exactly one of gt_boxes / gt_geom.
 * bin_entries, count pass (cell_keys NULL): ent_off [G+1] = exclusive scan of the cells each ground truth covers
 * (ent_off[G] = E entries).  Emit pass: cell_keys [E] = cell << 32 | j, in ascending j.  The caller then sorts
 * cell_keys by the cell (hdy_sort_keys_bytes, first_byte 4: stable, so every cell lists ascending j) and
 * bin_cells writes cell_start [n_cells + 1] (n_cells = nx * ny): the first entry of every cell.
 * boxes_binned, count pass (pair_rank / pair_j / pair_iou NULL): pair_off [P+1] = exclusive scan of the pairs with
 * box_iou >= iou_min of every prediction rank (pred_order [P] i32: rank -> row; NULL: identity).  Emit pass: the pairs
 * of rank r go to [pair_off[r], pair_off[r+1]) of pair_rank / pair_j / pair_iou, sorted by j: the whole list is in
 * row-major (rank, j) order.
 * mask_candidates_binned: the same two passes over windows; a pair is a candidate when its windows overlap and its
 * IoU bound (hdy_match_mask_pairs) reaches iou_min.  areas from hdy_mask_areas.
 * mask_exact_list: counts every candidate's intersection exactly (cand_iou [n_cand] scratch) and compacts the pairs
 * with iou >= iou_min, in candidate order, into pair_rank / pair_j / pair_iou; *pair_count (device) = their number
 * (block_scratch: 4096 int32).
 * order_keys: keys [n] = ~orderable(ious[i]) << 32 | i; sorting their high half (hdy_sort_keys_bytes, first_byte 4,
 * n_bytes 4) orders a (rank, j)-ordered list by IoU, descending, with ties in (rank, j) order. */
HDY_API int hdy_match_bin_stats(const float* gt_boxes, const int32_t* gt_geom, int G, uint64_t* stats,
                                hdy_stream_t stream);
HDY_API int hdy_match_bin_entries(const float* gt_boxes, const int32_t* gt_geom, int G, float ox, float oy,
                                  float inv_cell, int nx, int ny, int64_t* ent_off, uint64_t* cell_keys,
                                  hdy_stream_t stream);
HDY_API int hdy_match_bin_cells(const uint64_t* cell_keys, int64_t E, int64_t n_cells, int64_t* cell_start,
                                hdy_stream_t stream);
HDY_API int hdy_match_boxes_binned(const float* pred_boxes, const int32_t* pred_order, int P, const float* gt_boxes,
                                   int G, float ox, float oy, float inv_cell, int nx, int ny, const int64_t* cell_start,
                                   const uint64_t* cell_keys, float iou_min, int64_t* pair_off, int32_t* pair_rank,
                                   int32_t* pair_j, float* pair_iou, hdy_stream_t stream);
HDY_API int hdy_match_mask_candidates_binned(const int32_t* pred_geom, const int32_t* pred_areas,
                                             const int32_t* pred_order, int P, const int32_t* gt_geom,
                                             const int32_t* gt_areas, int G, float ox, float oy, float inv_cell,
                                             int nx, int ny, const int64_t* cell_start, const uint64_t* cell_keys,
                                             float iou_min, int64_t* cand_off, int32_t* cand_rank, int32_t* cand_j,
                                             hdy_stream_t stream);
HDY_API int hdy_match_mask_exact_list(const int32_t* pred_geom, const int64_t* pred_offsets, const uint32_t* pred_bits,
                                      const int32_t* pred_areas, const int32_t* pred_order, const int32_t* gt_geom,
                                      const int64_t* gt_offsets, const uint32_t* gt_bits, const int32_t* gt_areas,
                                      const int32_t* cand_rank, const int32_t* cand_j, int64_t n_cand, float iou_min,
                                      float* cand_iou, int32_t* pair_rank, int32_t* pair_j, float* pair_iou,
                                      int32_t* pair_count, int32_t* block_scratch, hdy_stream_t stream);
HDY_API int hdy_match_order_keys(const float* ious, int64_t n, uint64_t* keys, hdy_stream_t stream);

/* Utility: zero n int32 words (keeps the host mirror free of extra torch launches). */
HDY_API int hdy_zero_i32(int32_t* p, size_t n, hdy_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* HD_YOLO_B200_H_ */
