"""Whole-slide tiling and tile-merge: host-side mirror of the reference functions over csrc/merge.cu, csrc/coords.cu.

* ``sliding_window_scanner``  -- hnet/utils.py:37-62 (== metayolo/models/utils_o.py:37-62)          (T1, host side)
* ``merge_outputs``           -- Detect.merge_outputs, metayolo/models/yolo_head.py:450-463             (T2)
* ``rescale_outputs``         -- Detect.rescale_outputs, yolo_head.py:465-471 (in place)               (T2)
* ``Ensemble.merge`` / ``ensemble_merge`` -- metayolo/models/yolo.py:165-204                           (T3)
* ``scale_coords`` / ``clip_coords``      -- metayolo/models/utils_general.py:161-190 (in place)       (C1)
* ``SlideAccumulator``        -- the struct-of-arrays form the slide pipeline uses: DetectBatch results are appended
                                 in slide coordinates without leaving the device, then merged once.

The merge NMS is sparse (spatial hash + fixed-point rounds) but returns exactly what torchvision.ops.nms returns on
the concatenated detections.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import HdyError, ptr
from .ops import DetectBatch, _Scratch, _aligned16, _call, _conf_thr_f32, _iou_thr_f32, _need_cuda, _stream

__all__ = ["sliding_window_scanner", "tile_cores", "merge_outputs", "rescale_outputs", "scale_coords", "clip_coords",
           "merge_nms", "ensemble_merge", "Ensemble", "SlideAccumulator", "sort_keys", "kept_digest", "fold_digest",
           "mask_digest",
           "STATE_KEPT", "STATE_SUPPRESSED", "STATE_DROPPED"]

STATE_UNKNOWN, STATE_KEPT, STATE_SUPPRESSED, STATE_DROPPED = 0, 1, 2, 3
AFFINE_UNPAD, AFFINE_SCALE, AFFINE_CLIP, AFFINE_ROUND = 1, 2, 4, 8
_ws = _Scratch()


def _pair(v):
    return (v, v) if isinstance(v, (int, float)) else (v[0], v[1])


# ------------------------------------------------------------------------------------------------ T1
def sliding_window_scanner(image_size, roi_size=None, overlap=0) -> torch.Tensor:
    """hnet/utils.py:37-62: window origins every (roi - overlap) pixels, x fastest; windows are clipped to the
    image, so the last row / column are slivers.  Returns [n, 4] fp32 (x0, y0, x1, y1) on the host (this is
    control-plane data: 11 025 rows for a 100k x 100k px slide)."""
    if roi_size is None:
        return torch.tensor([[0., 0., image_size[0], image_size[1]]], dtype=torch.float32)
    h, w = _pair(image_size)
    roi_h, roi_w = _pair(roi_size)
    xs = torch.arange(0, w, roi_w - overlap, dtype=torch.float32) if w > roi_w else torch.zeros(1)
    ys = torch.arange(0, h, roi_h - overlap, dtype=torch.float32) if h > roi_h else torch.zeros(1)
    x0 = xs.repeat(len(ys))
    y0 = ys.repeat_interleave(len(xs))
    out = torch.stack((x0, y0, x0 + roi_w, y0 + roi_h), 1)
    out[:, 0::2] = out[:, 0::2].clamp(min=0, max=w)   # clip_boxes_to_image
    out[:, 1::2] = out[:, 1::2].clamp(min=0, max=h)
    return out


def tile_cores(rois: torch.Tensor) -> torch.Tensor:
    """For every tile the rectangle no OTHER tile of a grid tiling reaches: x from the right edge of the previous
    column to the left edge of the next one (unbounded at the border), same in y.  Host side, [n, 4] fp32."""
    r = rois.detach().cpu().to(torch.float64)
    big = 3.0e38
    out = torch.empty((len(r), 4), dtype=torch.float64)
    for lo, hi in ((0, 2), (1, 3)):
        starts = torch.unique(r[:, lo])                    # sorted column / row origins
        ends = torch.stack([r[r[:, lo] == s, hi].max() for s in starts])
        idx = torch.searchsorted(starts, r[:, lo].contiguous())
        prev_end = torch.cat([torch.tensor([-big], dtype=torch.float64), ends[:-1]])
        # several columns before this one may reach into it: take the furthest
        prev_end = torch.cummax(prev_end, 0).values
        next_start = torch.cat([starts[1:], torch.tensor([big], dtype=torch.float64)])
        out[:, lo] = prev_end[idx]
        out[:, hi] = next_start[idx]
    return out.to(torch.float32)


# ------------------------------------------------------------------------------------------------ C1
def _affine(rows: torch.Tensor, pad_x, pad_y, gain, scale, clip_w, clip_h, flags):
    _need_cuda(rows, "coords")
    if rows.dim() != 2 or rows.shape[1] < 4 or rows.stride(1) != 1:
        raise HdyError("coords must be [n, >=4] with unit stride along columns")
    if rows.shape[0]:
        _call("hdy_affine_boxes", ptr(rows), rows.shape[0], rows.stride(0), float(pad_x), float(pad_y), float(gain),
              float(scale), float(clip_w), float(clip_h), flags, _stream())
    return rows


def clip_coords(boxes: torch.Tensor, shape) -> None:
    """utils_general.py:181-190 (tensor branch), in place: x to [0, shape[1]], y to [0, shape[0]]."""
    _affine(boxes, 0, 0, 1, 1, shape[1], shape[0], AFFINE_CLIP)


def scale_coords(img1_shape, coords: torch.Tensor, img0_shape, ratio_pad=None, round_: bool = False) -> torch.Tensor:
    """utils_general.py:161-178, in place on coords [n, >=4]: undo the letterbox (subtract pad, divide by gain),
    clip to img0_shape.  round_=True fuses the ``.round()`` of evaluation.py:109."""
    img1_shape, img0_shape = _pair(img1_shape), _pair(img0_shape)
    if ratio_pad is None:
        gain = min(img1_shape[0] / img0_shape[0], img1_shape[1] / img0_shape[1])
        pad = (img1_shape[1] - img0_shape[1] * gain) / 2, (img1_shape[0] - img0_shape[0] * gain) / 2
    else:
        gain = ratio_pad[0][0]
        pad = ratio_pad[1]
    return _affine(coords, pad[0], pad[1], gain, 1, img0_shape[1], img0_shape[0],
                   AFFINE_UNPAD | AFFINE_CLIP | (AFFINE_ROUND if round_ else 0))


def rescale_outputs(r: Dict[str, torch.Tensor], scale: float = 1.0) -> Dict[str, torch.Tensor]:
    """Detect.rescale_outputs (yolo_head.py:465-471): r['boxes'] *= scale, in place."""
    if scale != 1.0:
        _affine(r['boxes'], 0, 0, 1, scale, 0, 0, AFFINE_SCALE)
    return r


# ------------------------------------------------------------------------------------------------ T3 core
def merge_nms(boxes: torch.Tensor, scores: torch.Tensor, conf_thres: float, iou_thres: float,
              tile_id: Optional[torch.Tensor] = None, cores: Optional[torch.Tensor] = None,
              margin: Optional[torch.Tensor] = None, n_dev: Optional[torch.Tensor] = None,
              max_rounds: int = 8, dirty: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Verdict per row of the slide-level greedy NMS of Ensemble.merge (yolo.py:189-195):
    uint8 [n] of STATE_KEPT / STATE_SUPPRESSED / STATE_DROPPED (score <= conf_thres).
    tile_id + cores + margin enable the interior shortcut (see include/hd_yolo_b200.h)."""
    _need_cuda(boxes, "boxes")
    _need_cuda(scores, "scores")
    n = boxes.shape[0]
    if boxes.dim() != 2 or boxes.shape[1] != 4 or scores.shape != (n,):
        raise HdyError("boxes must be [n,4] and scores [n]")
    dev = boxes.device
    state = torch.empty((n,), dtype=torch.uint8, device=dev)
    if n == 0:
        return state
    boxes = _aligned16(boxes.contiguous())
    scores = scores.contiguous()
    lib = _lib.load()
    wbytes = lib.hdy_merge_workspace_bytes(n)
    ws = _ws.get(dev, "merge", wbytes)
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    use_cores = cores is not None
    if use_cores and (tile_id is None or margin is None):
        raise HdyError("the interior shortcut needs tile_id, cores and margin")
    rounds = max_rounds
    while True:
        _call("hdy_merge_nms", ptr(boxes), ptr(scores), ptr(tile_id) if use_cores else None,
              ptr(cores) if use_cores else None, ptr(dirty) if use_cores else None,
              ptr(margin) if use_cores else None, ptr(n_dev), n,
              _conf_thr_f32(conf_thres), _iou_thr_f32(iou_thres), rounds, ptr(state), ptr(status), ptr(ws), wbytes,
              _stream(), launches=8 + 3 * rounds)
        if not int(status.item()) & _lib.HDY_STATUS_ROUNDS:
            return state
        if rounds >= 64:
            raise HdyError("merge NMS did not converge in 64 rounds")
        rounds, _ = min(64, rounds * 2), status.zero_()


def dirty_tiles(far_boxes: torch.Tensor, far_tile: torch.Tensor, far_count: torch.Tensor,
                rois: torch.Tensor) -> torch.Tensor:
    """uint8 [n_tiles]: tiles whose window is touched by a far-reaching box of another tile (hdy_merge_dirty_tiles)."""
    n_tiles = int(rois.shape[0])
    dirty = torch.empty((max(n_tiles, 1),), dtype=torch.uint8, device=rois.device)
    _call("hdy_merge_dirty_tiles", ptr(far_boxes), ptr(far_tile), ptr(far_count), int(far_boxes.shape[0]),
          ptr(_aligned16(rois.contiguous())), n_tiles, ptr(dirty), _stream())
    return dirty


def sort_keys(keys: torch.Tensor, n_dev: Optional[torch.Tensor] = None, first_byte: int = 0,
              n_bytes: int = 8) -> torch.Tensor:
    """Ascending in-place LSD radix sort of int64-typed 64-bit keys (bit pattern treated as unsigned); stable, and
    restricted to the bytes [first_byte, first_byte + n_bytes) of the key when asked (n_bytes even)."""
    if not keys.is_cuda or keys.dtype != torch.int64 or not keys.is_contiguous():
        raise HdyError("keys must be a contiguous CUDA int64 tensor")
    n = keys.numel()
    if n:
        lib = _lib.load()
        wbytes = lib.hdy_sort_workspace_bytes(n)
        ws = _ws.get(keys.device, "sort", wbytes)
        tmp = _ws.get(keys.device, "sort_tmp", n * 8)
        # per pass: histogram, its scan (one launch while the histogram fits one scan tile: n <= 16 384), scatter
        _call("hdy_sort_keys_bytes", ptr(keys), ptr(tmp), ptr(n_dev), n, int(first_byte), int(n_bytes), ptr(ws), wbytes,
              _stream(), launches=int(n_bytes) * (3 if n <= 16384 else 5))
    return keys


def _order_keys(state, scores, n: int, count: torch.Tensor) -> torch.Tensor:
    """Enqueues select + sort: one order key per KEPT row of state[:n], ascending (== score-descending, ties by the
    lower row); their number lands in `count` (device int32 [1]).  Returns the key buffer [n] (valid up to *count)."""
    dev = scores.device
    keys = torch.empty((max(n, 1),), dtype=torch.int64, device=dev)
    if n == 0:
        count.zero_()
        return keys
    # keys in row order + a stable sort of the score half only: same order as sorting the whole 64-bit key, in four
    # radix passes instead of eight
    blk = _ws.get(dev, "select_blocks", 4096 * 4)
    _call("hdy_merge_select_ordered", ptr(state), ptr(scores), None, n, ptr(keys), ptr(count), ptr(blk), _stream(),
          launches=3)
    sort_keys(keys, n_dev=count, first_byte=4, n_bytes=4)
    return keys


def _gather_ordered(keys, count, k_all: int, max_det: int, boxes, scores, labels):
    dev = boxes.device
    k = min(int(k_all), int(max_det))
    idx = torch.empty((k,), dtype=torch.int64, device=dev)
    ob = torch.empty((k, 4), dtype=torch.float32, device=dev)
    os_ = torch.empty((k,), dtype=torch.float32, device=dev)
    ol = torch.empty((k,), dtype=torch.int64, device=dev) if labels is not None else None
    oc = torch.empty((1,), dtype=torch.int32, device=dev)
    if k:
        _call("hdy_merge_gather", ptr(keys), ptr(count), k, ptr(boxes), ptr(scores), ptr(labels), ptr(idx), ptr(ob),
              ptr(os_), ptr(ol), ptr(oc), _stream())
    return idx, ob, os_, ol


def _kept_in_order(state, boxes, scores, labels, max_det: int, n_dev=None):
    """`keep = nms(...)[:max_det]; boxes[keep] ...` (yolo.py:195-196) from the verdicts."""
    n = boxes.shape[0]
    count = torch.empty((1,), dtype=torch.int32, device=boxes.device)
    keys = _order_keys(state, scores, n, count)
    return _gather_ordered(keys, count, int(count.item()), max_det, boxes, scores, labels)


def kept_digest(state: torch.Tensor, base: int = 0) -> torch.Tensor:
    """Order-independent digest of the KEPT global row indices: int64 [3] = (count, low 32 bits of the sum of a 64-bit
    mix of every index, high 32 bits of it), each a plain sum -- add the tensors of all ranks (all_reduce) and fold with
    ``fold_digest``.  Two runs kept the same rows iff (up to hash collisions) their digests agree, whatever the number
    of ranks.  Diagnostics: not part of the timed path."""
    idx = torch.nonzero(state == STATE_KEPT).flatten().to(torch.int64) + int(base)
    h = idx * -7046029254386353131            # 0x9E3779B97F4A7C15 (wraps: int64 arithmetic is mod 2^64)
    h = h ^ (h >> 31)
    h = h * -4658895280553007687              # 0xBF58476D1CE4E5B9
    h = h ^ (h >> 29)
    lo = (h & 0xffffffff).sum()
    hi = ((h >> 32) & 0xffffffff).sum()
    return torch.stack([torch.tensor(idx.numel(), dtype=torch.int64, device=state.device), lo, hi])


def fold_digest(t: torch.Tensor) -> Dict[str, object]:
    c, lo, hi = [int(v) for v in t.tolist()]
    return {"kept": c, "hash": f"{(lo + (hi << 32)) & 0xffffffffffffffff:016x}"}


def mask_digest(masks, state: torch.Tensor, base: int = 0, chunk_rows: int = 1 << 19) -> torch.Tensor:
    """The same for the mask bits of the KEPT rows: every mask word is mixed with (global row, word position inside
    the mask), so the digest does not depend on where a rank's words sit in its buffer.  int64 [3] like kept_digest,
    the count being the number of set mask pixels.  Diagnostics (chunked torch ops), not part of the timed path."""
    dev = state.device
    all_rows = torch.nonzero(state == STATE_KEPT).flatten()
    acc = torch.zeros((3,), dtype=torch.int64, device=dev)
    for c0 in range(0, int(all_rows.numel()), chunk_rows):
        rows = all_rows[c0:c0 + chunk_rows]
        g = masks.geom[rows].to(torch.int64)
        words = ((g[:, 2] + 31) >> 5) * g[:, 3]
        total = int(words.sum())
        if total == 0:
            continue
        owner = torch.repeat_interleave(torch.arange(rows.numel(), device=dev), words)
        start = torch.cumsum(words, 0) - words
        j = torch.arange(total, device=dev) - start[owner]
        w = masks.bits[masks.offsets[rows][owner] + j].to(torch.int64) & 0xffffffff
        h = ((rows[owner] + int(base)) * 1000003 + j) * -7046029254386353131
        h = (h ^ (h >> 31)) + w * -4658895280553007687
        h = h ^ (h >> 29)
        pop = w - ((w >> 1) & 0x55555555)
        pop = (pop & 0x33333333) + ((pop >> 2) & 0x33333333)
        pop = ((((pop + (pop >> 4)) & 0x0f0f0f0f) * 0x01010101) >> 24) & 0xff
        acc += torch.stack([pop.sum(), (h & 0xffffffff).sum(), ((h >> 32) & 0xffffffff).sum()])
    return acc


# ------------------------------------------------------------------------------------------------ T2 / T3 drop-ins
def merge_outputs(r: List[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
    """Detect.merge_outputs (yolo_head.py:450-463): one dict per tile with 'boxes' [k,4] (tile coordinates),
    'labels', 'scores' and 'roi' (x0, y0, ...) -> one dict in slide coordinates, tiles concatenated in order.
    No NMS.  'masks' are concatenated as they are."""
    if not len(r):
        raise HdyError("merge_outputs needs at least one tile")
    dev = r[0]['boxes'].device
    _need_cuda(r[0]['boxes'], "boxes")
    counts_h = [int(t['boxes'].shape[0]) for t in r]
    bs, md = len(r), max(max(counts_h), 1)
    n = sum(counts_h)
    res = {'labels': torch.cat([t['labels'] for t in r]), 'scores': torch.cat([t['scores'] for t in r])}
    cat = _aligned16(torch.cat([t['boxes'] for t in r]).contiguous())
    rois = torch.stack([torch.as_tensor(t['roi'], dtype=torch.float32).reshape(-1)[:4].cpu() for t in r]).to(dev)
    out = torch.empty((n, 4), dtype=torch.float32, device=dev)
    if n:
        # one launch per call: every tile is a "batch row" of its own length, addressed through tile_offsets
        counts = torch.tensor(counts_h, dtype=torch.int32).to(dev)
        # pad to [bs, md, 4] without a Python loop
        offs = torch.tensor([0] + counts_h[:-1], dtype=torch.int64).cumsum(0).to(dev)
        tile_of = torch.repeat_interleave(torch.arange(bs, device=dev), counts.long())
        slot = torch.arange(n, device=dev) - offs[tile_of]
        padded = torch.zeros((bs, md, 4), dtype=torch.float32, device=dev)
        padded[tile_of, slot] = cat
        cursor = torch.zeros((1,), dtype=torch.int64, device=dev)
        tile_offsets = torch.empty((bs + 1,), dtype=torch.int64, device=dev)
        status = torch.zeros((1,), dtype=torch.int32, device=dev)
        for b0 in range(0, bs, 65535):
            b1 = min(bs, b0 + 65535)
            _call("hdy_merge_append", ptr(padded[b0:b1]), None, None, None, ptr(counts[b0:b1]), ptr(rois[b0:b1]), b1 - b0, md,
                  b0, 1.0, n, ptr(out), None, None, None, ptr(cursor), ptr(tile_offsets[b0:]), ptr(status), _stream(),
                  launches=2)
    res = {'boxes': out, **res}
    if 'masks' in r[0]:
        res['masks'] = torch.cat([t['masks'] for t in r])
    return res


def ensemble_merge(x: List[Dict[str, Dict[str, torch.Tensor]]], nms_params: Dict[str, float]):
    """Ensemble.merge (yolo.py:165-204): per task id, concatenate the members' detections, keep scores >
    conf_thres, class-agnostic NMS on the final scores, first max_det, gather boxes / scores / labels / masks."""
    task_ids = set().union(*x)
    res: Dict[str, Dict[str, torch.Tensor]] = {}
    conf, iou, max_det = nms_params['conf_thres'], nms_params['iou_thres'], int(nms_params['max_det'])
    for task_id in task_ids:
        parts = [r[task_id] for r in x if task_id in r]
        boxes = torch.cat([p['boxes'] for p in parts])
        scores = torch.cat([p['scores'] for p in parts])
        labels = torch.cat([p['labels'] for p in parts])
        masks = None
        if any('masks' in p for p in parts):
            ref = [p['masks'] for p in parts if 'masks' in p][0]
            masks = torch.cat([p['masks'] if 'masks' in p else torch.zeros(ref.shape[1:]).to(ref.device, ref.dtype)
                               for p in parts])
        if scores.dim() != 1:
            raise HdyError("Ensemble.merge handles single-label outputs (scores [n]); the reference's multi-label "
                           "merge is unfinished (yolo.py:145)")
        lab64 = labels.to(torch.int64).contiguous()
        boxes = _aligned16(boxes.contiguous().float())
        state = merge_nms(boxes, scores.contiguous(), conf, iou)
        idx, ob, os_, ol = _kept_in_order(state, boxes, scores.contiguous(), lab64, max_det)
        out = {'boxes': ob, 'scores': os_, 'labels': ol.to(labels.dtype)}
        if masks is not None:
            out['masks'] = masks[idx]
        res[task_id] = out
    return res


class Ensemble:
    """The merge half of metayolo.models.yolo.Ensemble (yolo.py:144-204); the member models stay PyTorch."""

    def __init__(self, models=(), nms_params: Dict[str, float] = {}):
        self.models = list(models)
        self.nms_params = self.get_nms_params(nms_params)

    def get_nms_params(self, args={}):
        default_args = {'conf_thres': 0.15, 'iou_thres': 0.45, 'max_det': 300}
        return {k: float(args.get(k, v)) for k, v in default_args.items()}

    def merge(self, x):
        return ensemble_merge(x, self.nms_params)


# ------------------------------------------------------------------------------------------------ slide pipeline
class SlideAccumulator:
    """Slide-level struct-of-arrays store: DetectBatch results are appended in slide coordinates (T2) as the tile
    batches finish, entirely on the device; ``merge`` then runs T3 once.  Row order == the order
    ``merge_outputs`` would concatenate the tiles in, so results are identical to the list-of-dicts route."""

    def __init__(self, capacity: int, device, with_labels: bool = True):
        self.capacity = int(capacity)
        self.device = torch.device(device)
        d = self.device
        self.boxes = torch.empty((self.capacity, 4), dtype=torch.float32, device=d)
        self.scores = torch.empty((self.capacity,), dtype=torch.float32, device=d)
        self.labels = torch.empty((self.capacity,), dtype=torch.int64, device=d) if with_labels else None
        self.tile = torch.empty((self.capacity,), dtype=torch.int32, device=d)
        self.cursor = torch.zeros((1,), dtype=torch.int64, device=d)
        self.status = torch.zeros((1,), dtype=torch.int32, device=d)
        self.tile_offsets: List[torch.Tensor] = []
        self.rois: List[torch.Tensor] = []
        self.n_tiles = 0
        self.gray_ok = True        # every batch so far came with gray-zone flags (DetectBatch.fragile) and scale 1
        self.gray_eps = float("inf")   # smallest gray_eps / largest tile IoU threshold the flags were produced with
        self.gray_iou = 0.0
        self._cores = self._cores_rois = self._cores_key = None
        self._top = 0.0
        self._rois_key: Optional[List[bytes]] = []   # host bytes of the appended windows (None: not all were given)

    def reset(self):
        self.cursor.zero_()
        self.status.zero_()
        self.tile_offsets.clear()
        self.rois.clear()
        self.n_tiles = 0
        self.gray_ok = True
        self.gray_eps, self.gray_iou = float("inf"), 0.0
        self._rois_key = []          # the core rectangles stay cached: they are keyed on the windows' contents

    def append(self, batch: DetectBatch, rois: torch.Tensor, scale: float = 1.0,
               rois_host: Optional[torch.Tensor] = None) -> None:
        """rois [bs, 4] fp32 on the device: the windows (x0, y0, x1, y1) of the batch's tiles.  rois_host: the same
        windows on the host, if the caller has them (keys the core-rectangle cache without a device read)."""
        bs = batch.counts.shape[0]
        if self._rois_key is not None:
            self._rois_key = self._rois_key + [rois_host.contiguous().numpy().tobytes()] if rois_host is not None \
                else None
        if rois.shape != (bs, 4) or not rois.is_cuda or rois.dtype != torch.float32:
            raise HdyError("rois must be a CUDA fp32 tensor [bs, 4]")
        rois = _aligned16(rois.contiguous())
        offs = torch.empty((bs + 1,), dtype=torch.int64, device=self.device)
        fragile = batch.fragile if scale == 1.0 else None
        if fragile is None:
            self.gray_ok = False
        else:
            self.gray_eps = min(self.gray_eps, float(batch.gray_eps))
            self.gray_iou = max(self.gray_iou, float(batch.iou_thres))
        _call("hdy_merge_append", ptr(batch.boxes), ptr(batch.scores), ptr(batch.labels) if self.labels is not None else None,
              ptr(fragile), ptr(batch.counts), ptr(rois), bs, batch.max_det, self.n_tiles, float(scale), self.capacity,
              ptr(self.boxes), ptr(self.scores), ptr(self.labels), ptr(self.tile), ptr(self.cursor), ptr(offs),
              ptr(self.status), _stream(), launches=2)
        self.tile_offsets.append(offs)
        self.rois.append(rois)
        self.n_tiles += bs

    def reserve(self, capacity: int) -> None:
        """Grow the row arrays to `capacity` rows, keeping what was appended (the sharded merge parks the other ranks'
        seam rows behind the own rows and may find that it needs more room than was planned)."""
        capacity = int(capacity)
        if capacity <= self.capacity:
            return
        n = min(int(self.cursor.item()), self.capacity)
        for name in ("boxes", "scores", "labels", "tile"):
            old = getattr(self, name)
            if old is None:
                continue
            new = torch.empty((capacity,) + tuple(old.shape[1:]), dtype=old.dtype, device=old.device)
            new[:n] = old[:n]
            setattr(self, name, new)
        self.capacity = capacity

    def count(self) -> int:
        """Rows appended so far (synchronises); raises on capacity overflow."""
        both = torch.cat([self.cursor, self.status.long()]).cpu()
        if int(both[1]) & _lib.HDY_STATUS_OVERFLOW:
            raise HdyError(f"slide accumulator overflow ({int(both[0])} rows, capacity {self.capacity}), or a tile's "
                           "candidate list outgrew `cap` (detect_postprocess(cap=...))")
        return int(both[0])

    FAR_CAP_PX = 64.0        # boxes sticking out of their tile by more than this are always handled one by one
    FAR_MIN_CAP_PX = 8.0     # ... and never those sticking out by less than this (the cap is picked in between)
    FAR_CAPACITY = 4096

    def overhang(self):
        """(margin [1] fp32, far_boxes [FAR_CAPACITY,4], far_tile [FAR_CAPACITY] i32, far_count [1] i32), all on the
        device: how far the appended boxes stick out of their own tiles at most, not counting the few far-reaching ones
        (huge false positives), which are listed instead (tile indices local to this accumulator)."""
        rois = torch.cat(self.rois)
        d = self.device
        margin = torch.zeros((1,), dtype=torch.float32, device=d)
        far_boxes = torch.empty((self.FAR_CAPACITY, 4), dtype=torch.float32, device=d)
        far_tile = torch.empty((self.FAR_CAPACITY,), dtype=torch.int32, device=d)
        far_count = torch.zeros((1,), dtype=torch.int32, device=d)
        # the cap is picked from the data: as low as possible (every core shrinks by the largest overhang below it)
        # while at most ~1.5 % of the tiles' worth of boxes end up on the far list (their neighbours turn dirty)
        hist = torch.empty((256,), dtype=torch.int32, device=d)
        cap = torch.empty((1,), dtype=torch.float32, device=d)
        max_far = int(min(max(int(rois.shape[0]) // 64, 16), self.FAR_CAPACITY // 4))
        _call("hdy_merge_overhang_cap", ptr(self.boxes), ptr(self.tile), ptr(rois), ptr(self.cursor), self.capacity,
              max_far, float(self.FAR_MIN_CAP_PX), float(self.FAR_CAP_PX), ptr(hist), ptr(cap), _stream(), launches=2)
        _call("hdy_merge_overhang", ptr(self.boxes), ptr(self.tile), ptr(rois), ptr(self.cursor), self.capacity,
              float(self.FAR_CAP_PX), ptr(cap), ptr(margin), ptr(far_boxes), ptr(far_tile), ptr(far_count),
              self.FAR_CAPACITY, _stream())
        return margin, far_boxes, far_tile, far_count

    def check_shortcut(self, iou_thres: float) -> None:
        """The preconditions under which skipping the interior is exact (DESIGN.md 3.5); raises when one fails."""
        import numpy as np
        if not self.gray_ok:
            raise HdyError("interior_shortcut needs gray-zone flags on every appended batch "
                           "(detect_postprocess(gray_eps=...), scale 1)")
        if iou_thres < 0.05:
            raise HdyError("interior_shortcut: iou_thres < 0.05 is not covered by the gray-zone bound")
        if self.gray_iou and iou_thres < self.gray_iou:
            raise HdyError(f"interior_shortcut: merge iou_thres {iou_thres} is below the per-tile NMS threshold "
                           f"{self.gray_iou} the gray-zone flags were produced for (same-tile survivors may overlap more)")
        if self.rois:
            top = self._top
            need = float(np.spacing(np.float32(max(top, 1.0)))) / 2.0
            if self.gray_eps < need:
                raise HdyError(f"interior_shortcut: the gray-zone flags cover a rounding of {self.gray_eps:g} px per "
                               f"coordinate, slide coordinates up to {top:g} round by up to {need:g}")
        if self.rois and self.gray_eps > 0.004:        # (a rank without tiles has appended nothing: nothing to check)
            raise HdyError("interior_shortcut: gray_eps above 0.004 px exceeds the binning margins of the per-tile NMS")

    def verdicts(self, conf_thres: float, iou_thres: float, interior_shortcut: bool = False) -> torch.Tensor:
        """uint8 state per appended row (asynchronous except for the round-budget check).

        interior_shortcut: rows that lie strictly inside their tile's core (the part no other tile's boxes can reach)
        and are not flagged fragile are KEPT without any pair test.  Exact when every batch was produced with
        gray-zone flags (detect_postprocess(gray_eps=...)) for an IoU threshold <= iou_thres: then a survivor of the
        per-tile NMS can only be suppressed by another tile's box or by a flagged neighbour (DESIGN.md 3.5)."""
        n = self.capacity
        kw = {}
        if interior_shortcut:
            rois = torch.cat(self.rois)
            # the core rectangles are cached on the CONTENTS of the windows (host bytes when the caller supplied them,
            # else a device comparison)
            key = b"".join(self._rois_key) if self._rois_key is not None else None
            same = self._cores is not None and (
                (key is not None and key == self._cores_key) or
                (key is None and self._cores_rois.shape == rois.shape and torch.equal(self._cores_rois, rois)))
            if not same:
                self._cores = tile_cores(rois).to(self.device)
                self._cores_rois, self._cores_key = rois, key
                self._top = float(rois.abs().max()) if rois.numel() else 0.0
            self.check_shortcut(iou_thres)
            margin, far_boxes, far_tile, far_count = self.overhang()
            kw = dict(tile_id=self.tile, cores=self._cores, margin=margin,
                      dirty=dirty_tiles(far_boxes, far_tile, far_count, rois))
        return merge_nms(self.boxes, self.scores, conf_thres, iou_thres, n_dev=self.cursor, **kw)

    def merge(self, conf_thres: float, iou_thres: float, max_det: Optional[int] = None,
              interior_shortcut: bool = False) -> Dict[str, torch.Tensor]:
        """Ensemble.merge over everything appended: {'boxes','scores','labels','index'} score-descending;
        'index' is the row in the concatenated (merge_outputs) order."""
        n = self.count()
        state = self.verdicts(conf_thres, iou_thres, interior_shortcut)
        idx, ob, os_, ol = _kept_in_order(state[:n], self.boxes[:n], self.scores[:n],
                                          self.labels[:n] if self.labels is not None else None,
                                          n if max_det is None else max_det)
        out = {'boxes': ob, 'scores': os_, 'index': idx}
        if ol is not None:
            out['labels'] = ol
        return out
