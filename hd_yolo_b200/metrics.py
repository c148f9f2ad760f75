"""Prediction <-> ground-truth matching on the device (SURVEY 8f rank 2): host mirror of ``box_iou``
(metayolo/models/utils_general.py:247-265) and of the matching half of ``APMeter.add``
(metayolo/models/metrics.py:270-303), over ``hdy_box_iou`` / ``hdy_match_pairs``, and by mask IoU over
``hdy_match_mask_pairs`` (bit-packed masks, ``PackedMasks``); at region and slide scale over the binned matchers of
csrc/match_binned.cu (``binned=True``).

The reference moves every image's detections to the host and builds a dense k x g IoU matrix there; here the
matching pairs are produced on the device and only they (a few hundred rows per image) are copied back.
``APMeter`` keeps the reference's accumulator fields (CPU tensors), so the reference's own ``ap_per_class`` /
plotting code runs on it unchanged.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch

from ._lib import HdyError, ptr
from .masks import PackedMasks
from .ops import _Cand, _aligned16, _call, _need_cuda, _run_nms, _stream

__all__ = ["box_iou", "match_predictions", "APMeter"]


def box_iou(box1: torch.Tensor, box2: torch.Tensor) -> torch.Tensor:
    """box_iou (utils_general.py:247-265): [N, 4] x [M, 4] xyxy -> [N, M]."""
    _need_cuda(box1, "box1")
    _need_cuda(box2, "box2")
    if box1.dim() != 2 or box1.shape[1] != 4 or box2.dim() != 2 or box2.shape[1] != 4:
        raise HdyError("box_iou takes [N,4] and [M,4]")
    n, m = int(box1.shape[0]), int(box2.shape[0])
    out = torch.empty((n, m), dtype=torch.float32, device=box1.device)
    if n and m:
        b1, b2 = _aligned16(box1.contiguous()), _aligned16(box2.contiguous())
        _call("hdy_box_iou", ptr(b1), n, ptr(b2), m, ptr(out), _stream())
    return out


def match_predictions(output: Dict[str, torch.Tensor], target: Dict[str, torch.Tensor], iou_min: float = 0.5,
                      cap: Optional[int] = None, iou_type: str = 'boxes', binned: bool = False) -> Dict[str, torch.Tensor]:
    """The device half of APMeter.add (metrics.py:271-284), by box IoU or, with iou_type='masks', by mask IoU.

    Returns (all on the device): 'order' (rows of `output` by score, descending, ties by lower row), 'scores' /
    'labels' in that order, and the matching pairs 'pred_idx' (rank in `order`), 'true_idx', 'ious' sorted by IoU
    descending (ties in row-major (pred, true) order).  One D2H read (the pair count) per pass; a crowded image that
    overflows `cap` is run again with the size the kernel reported.

    iou_type='masks': output['masks'] and target['masks'] are each a CUDA tensor [n, H, W] / [n, 1, H, W] (packed on
    the fly by PackedMasks.from_dense: fp32 / fp16 set iff > 0.5, uint8 / bool iff nonzero) or a PackedMasks, with as
    many rows as the boxes, on one (H, W) canvas.  inter / union are exact pixel counts, iou = float(inter) /
    float(union); iou_min must be > 0.  Every (prediction, ground truth) pair of windows is tested once (O(k * g), as
    the box path): sized for an image, not for region- or slide-scale ground truth (1e5+ nuclei per call).

    binned=True: the same result, bit for bit, for region- and slide-scale inputs (k, g < 2^31, fewer than 2^31
    matching pairs, k * g unrestricted).  The ground truth is put into a uniform grid over its extent and a prediction
    is tested only against the ground truth listed in the cells its box (or mask window) covers; `cap` is not used.
    Needs iou_min > 0 for boxes too (the grid only finds pairs that overlap).  Small D2H reads: three for boxes (grid
    statistics, entry count, pair count), four for masks (+ the matched count), plus what the mask inputs take as
    everywhere (PackedMasks.check's status read per PackedMasks side, from_dense's word count per dense side).  One
    rank's rows only: a ground-truth nucleus on a seam
    between ranks can match predictions of both, so gather a multi-rank slide result to one rank before matching."""
    if iou_type not in ('boxes', 'masks'):
        raise HdyError(f"iou_type must be 'boxes' or 'masks', got {iou_type!r}")
    if binned and not np.float32(iou_min) > 0:
        raise HdyError(f"binned matching needs iou_min > 0 (the grid only finds pairs that overlap), got {iou_min}")
    boxes, scores, gts = output['boxes'], output['scores'], target['boxes']
    _need_cuda(boxes, "output['boxes']")
    _need_cuda(scores, "output['scores']")
    _need_cuda(gts, "target['boxes']")
    dev = boxes.device
    k, g = int(boxes.shape[0]), int(gts.shape[0])
    if iou_type == 'masks':
        _check_mask_inputs(output, target, k, g, iou_min)
    i64 = dict(dtype=torch.int64, device=dev)
    empty = {'pred_idx': torch.empty(0, **i64), 'true_idx': torch.empty(0, **i64),
             'ious': torch.empty(0, dtype=torch.float32, device=dev)}
    if k == 0:
        return {'order': torch.empty(0, **i64), 'scores': scores.reshape(0), 'labels': output['labels'].reshape(0), **empty}
    # 1. predictions by score: one ascending radix sort of the (~score, row) keys (hdy_sort_keys_bytes), row = low word
    from .slide import sort_keys
    scores = scores.contiguous()
    keys = torch.empty(k, dtype=torch.int64, device=dev)
    _call("hdy_make_keys", ptr(scores), 1, k, ptr(keys), _stream())
    sort_keys(keys)
    order = keys & 0xffffffff
    order32 = order.to(torch.int32).contiguous()
    res = {'order': order, 'scores': scores[order], 'labels': output['labels'][order]}
    if g == 0:
        return {**res, **empty}
    if binned:
        if max(k, g) >= 2 ** 31:
            raise HdyError(f"binned matching takes fewer than 2^31 predictions and ground truth (got {k}, {g})")
        return {**res, **_binned_match(output, target, iou_type, order32, k, g, iou_min, empty)}
    # 2. pairs with iou >= iou_min, as order keys (~orderable(iou) << 32 | rank * g + j)
    if iou_type == 'masks':
        launch = _mask_pairs(_packed(output['masks']), _packed(target['masks']), order32, k, g, iou_min)
    else:
        launch = _box_pairs(_aligned16(boxes.contiguous()), order32, _aligned16(gts.contiguous()), k, g, iou_min)
    cap = int(cap) if cap is not None else max(4 * max(k, g), 1024)
    while True:
        pk, needs = launch(cap)
        needs = needs.tolist()                        # the reference's torch.where synchronises here too
        n_match = needs[0]
        if max(needs) <= cap:
            break
        cap = max(needs)                              # a crowded image: retry with the size the kernel reported
    if n_match == 0:
        return {**res, **empty}
    # 3. IoU-descending order of the pairs: a key sort (pairs of one prediction share a box -- as an "NMS that only
    #    sorts" they would all land in one spatial-hash cell); index and IoU are read back out of the key
    pk = pk[:n_match].contiguous()
    sort_keys(pk)
    pidx = pk & 0xffffffff
    res.update({'pred_idx': pidx // g, 'true_idx': pidx % g, 'ious': _key_scores(pk)})
    return res


def _box_pairs(boxes, order32, gts, k, g, iou_min):
    """launch(cap) -> (pair keys [cap], counts needed: [pairs]) over hdy_match_pairs."""
    dev = boxes.device

    def launch(cap):
        pk = torch.empty(cap, dtype=torch.int64, device=dev)
        pb = torch.empty((cap, 4), dtype=torch.float32, device=dev)
        pc = _Cand.__new__(_Cand)
        pc.bs, pc.cap, pc.keys, pc.boxes, pc.cls = 1, cap, pk, pb, None
        pc.counts = torch.zeros(2, dtype=torch.int32, device=dev)
        kc = torch.tensor([k, g], dtype=torch.int32).to(dev)
        _call("hdy_match_pairs", ptr(boxes), ptr(order32), ptr(kc[0:1]), 1, k, ptr(gts), ptr(kc[1:2]), g,
              float(np.float32(iou_min)), cap, ptr(pk), ptr(pb), ptr(pc.counts), pc.status_ptr, _stream())
        return pk, pc.counts[:1]
    return launch


def _mask_pairs(pm: PackedMasks, gm: PackedMasks, order32, k, g, iou_min):
    """launch(cap) -> (pair keys [cap], counts needed: [pairs, candidates]) over hdy_match_mask_pairs; `cap` bounds
    both lists (every pair is a candidate)."""
    dev = order32.device
    ap, ag = pm.areas(), gm.areas()
    pgeom, ggeom = _aligned16(pm.geom.contiguous()), _aligned16(gm.geom.contiguous())
    pbits, gbits = pm._bits_nonempty(), gm._bits_nonempty()

    def launch(cap):
        cand = torch.empty(cap, dtype=torch.int32, device=dev)
        pk = torch.empty(cap, dtype=torch.int64, device=dev)
        counts = torch.zeros(3, dtype=torch.int32, device=dev)     # pairs, candidates, status
        _call("hdy_match_mask_pairs", ptr(pgeom), ptr(pm.offsets), ptr(pbits), ptr(ap), ptr(order32), k, ptr(ggeom),
              ptr(gm.offsets), ptr(gbits), ptr(ag), g, float(np.float32(iou_min)), cap, ptr(cand), cap, ptr(pk),
              ptr(counts), ptr(counts[2:]), _stream(), launches=2)
        return pk, counts[:2]
    return launch


def _f32_of_orderable(o: int) -> float:
    o &= 0xffffffff
    u = (o & 0x7fffffff) if o & 0x80000000 else (~o & 0xffffffff)
    return float(np.array(u, dtype=np.uint32).view(np.float32))


def _pick_grid(stats):
    """(ox, oy, inv_cell, nx, ny) from hdy_match_bin_stats: cells about one mean ground-truth side across (a nucleus
    covers a few cells), at most 2 * n + 1024 of them (n valid ground truth), larger cells where the extent needs it.
    Any grid gives the same pairs (the cell function clamps: a short last row or column of cells only holds more);
    this one keeps the lists short.  The extent of finite fp32 coordinates is below 2^129, so the cell is below
    2^129 / sqrt(1024) and 1 / cell stays a normal fp32."""
    n = stats[4]
    x0, y0, x1, y1 = (_f32_of_orderable(v) for v in stats[:4])
    w, h = max(x1 - x0, 0.0), max(y1 - y0, 0.0)
    max_cells = min(2 * n + 1024, 1 << 26)
    cell = max(stats[5] / 16.0 / n, 1.0, math.sqrt(w * h / max_cells))
    inv = float(np.float32(1.0 / cell))
    nx = min(int(w * inv) + 1, max_cells)
    ny = min(int(h * inv) + 1, max(max_cells // nx, 1))
    return float(np.float32(x0)), float(np.float32(y0)), inv, nx, ny


def _binned_match(output, target, iou_type, order32, k, g, iou_min, empty):
    """'pred_idx', 'true_idx', 'ious' of match_predictions(binned=True) over csrc/match_binned.cu."""
    dev = order32.device
    i64 = dict(dtype=torch.int64, device=dev)
    i32 = dict(dtype=torch.int32, device=dev)
    thr = float(np.float32(iou_min))
    if iou_type == 'masks':
        pm, gm = _packed(output['masks']), _packed(target['masks'])
        pred = _aligned16(pm.geom.contiguous())
        gb, gg = None, _aligned16(gm.geom.contiguous())
    else:
        pred = _aligned16(output['boxes'].contiguous())
        gb, gg = _aligned16(target['boxes'].contiguous()), None
    # 1. the grid (one read: its statistics), the ground truth's cell entries (one read: their number), sorted by cell
    stats = torch.empty(6, **i64)
    _call("hdy_match_bin_stats", ptr(gb), ptr(gg), g, ptr(stats), _stream(), launches=2)
    stats = stats.tolist()
    if stats[4] == 0:
        return empty                                  # no ground truth can overlap anything
    grid = _pick_grid(stats)
    n_cells = grid[3] * grid[4]
    ent_off = torch.empty(g + 1, **i64)
    _call("hdy_match_bin_entries", ptr(gb), ptr(gg), g, *grid, ptr(ent_off), None, _stream(), launches=3)
    n_ent = int(ent_off[g].item())
    cell_keys = torch.empty(n_ent, **i64)
    _call("hdy_match_bin_entries", ptr(gb), ptr(gg), g, *grid, ptr(ent_off), ptr(cell_keys), _stream())
    from .slide import sort_keys
    sort_keys(cell_keys, first_byte=4, n_bytes=2 if n_cells <= 1 << 16 else 4)
    cell_start = torch.empty(n_cells + 1, **i64)
    _call("hdy_match_bin_cells", ptr(cell_keys), n_ent, n_cells, ptr(cell_start), _stream())
    # 2. the pairs (boxes) or candidates (masks) of every prediction rank, in (rank, j) order (one read: their number)
    off = torch.empty(k + 1, **i64)
    if iou_type == 'masks':
        ap, ag = pm.areas(), gm.areas()
        fn, head = "hdy_match_mask_candidates_binned", (ptr(pred), ptr(ap), ptr(order32), k, ptr(gg), ptr(ag), g)
    else:
        fn, head = "hdy_match_boxes_binned", (ptr(pred), ptr(order32), k, ptr(gb), g)
    tail = (ptr(cell_start), ptr(cell_keys), thr, ptr(off))
    _call(fn, *head, *grid, *tail, *((None,) * (2 if iou_type == 'masks' else 3)), _stream(), launches=4)
    n = int(off[k].item())
    if n >= 2 ** 31:
        raise HdyError(f"{n} {'candidate pairs' if iou_type == 'masks' else 'matching pairs'}: binned matching "
                       "takes fewer than 2^31")
    if n == 0:
        return empty
    rank, j = torch.empty(n, **i32), torch.empty(n, **i32)
    iou = torch.empty(n, dtype=torch.float32, device=dev)
    if iou_type == 'masks':
        _call(fn, *head, *grid, *tail, ptr(rank), ptr(j), _stream())
        # 3. exact intersections of the candidates, the matching ones compacted in order (one read: their number)
        cand_iou = torch.empty(n, dtype=torch.float32, device=dev)
        pr, pj = torch.empty(n, **i32), torch.empty(n, **i32)
        count = torch.zeros(1, **i32)
        blk = torch.empty(4096, **i32)
        _call("hdy_match_mask_exact_list", ptr(pred), ptr(pm.offsets), ptr(pm._bits_nonempty()), ptr(ap),
              ptr(order32), ptr(gg), ptr(gm.offsets), ptr(gm._bits_nonempty()), ptr(ag), ptr(rank), ptr(j), n, thr,
              ptr(cand_iou), ptr(pr), ptr(pj), ptr(iou), ptr(count), ptr(blk), _stream(), launches=4)
        rank, j = pr, pj
        n = int(count.item())
        if n == 0:
            return empty
    else:
        _call(fn, *head, *grid, *tail, ptr(rank), ptr(j), ptr(iou), _stream())
    # 4. IoU-descending order, ties in (rank, j) order: a stable sort of the IoU half of (~orderable(iou), position)
    keys = torch.empty(n, **i64)
    _call("hdy_match_order_keys", ptr(iou), n, ptr(keys), _stream())
    sort_keys(keys, first_byte=4, n_bytes=4)
    pos = keys & 0xffffffff
    return {'pred_idx': rank[pos].to(torch.int64), 'true_idx': j[pos].to(torch.int64), 'ious': _key_scores(keys)}


def _mask_canvas(m, n: int, name: str):
    if isinstance(m, PackedMasks):
        rows, hw = len(m), (m.H, m.W)
        if not (m.geom.is_cuda and m.offsets.is_cuda and m.bits.is_cuda):
            raise HdyError(f"{name} must live on a CUDA device: hd_yolo_b200 has no CPU fallback")
    elif isinstance(m, torch.Tensor):
        if m.dim() not in (3, 4) or (m.dim() == 4 and m.shape[1] != 1):
            raise HdyError(f"{name} must be [n, H, W] or [n, 1, H, W], got {tuple(m.shape)}")
        rows, hw = int(m.shape[0]), tuple(int(s) for s in m.shape[-2:])
    else:
        raise HdyError(f"{name} must be a CUDA tensor or a PackedMasks, got {type(m).__name__}")
    if rows != n:
        raise HdyError(f"{name} has {rows} rows for {n} boxes")
    return hw


def _check_mask_inputs(output, target, k: int, g: int, iou_min: float) -> None:
    if 'masks' not in output or 'masks' not in target:
        raise HdyError("iou_type='masks' needs 'masks' in both output and target")
    if not iou_min > 0:
        raise HdyError(f"mask matching needs iou_min > 0 (pairs of disjoint masks have IoU 0), got {iou_min}")
    cp, cg = _mask_canvas(output['masks'], k, "output['masks']"), _mask_canvas(target['masks'], g, "target['masks']")
    if cp != cg:
        raise HdyError(f"predicted masks lie on a {cp[0]} x {cp[1]} canvas, ground-truth masks on {cg[0]} x {cg[1]}")


def _packed(m) -> PackedMasks:
    if isinstance(m, PackedMasks):
        m.check()                                     # an overflowed plane lacks bits: its IoUs would be wrong
        return m
    return PackedMasks.from_dense(m)


def _key_scores(keys: torch.Tensor) -> torch.Tensor:
    """fp32 value stored in the high word of order keys ((~orderable(v) << 32) | index, csrc/hdy_common.cuh)."""
    o = (~(keys >> 32)) & 0xffffffff                                    # orderable(v)
    bits = torch.where(o >= 0x80000000, o & 0x7fffffff, (~o) & 0xffffffff)
    return torch.where(bits >= 0x80000000, bits - (1 << 32), bits).to(torch.int32).view(torch.float32)


class APMeter(object):
    """APMeter (metrics.py:250-303) with the matching done on the device.  The accumulator fields and their meaning
    are the reference's (n_pred, n_true, n_match, scores, y_pred, y_true, ious, m_pred, m_true: CPU tensors), so
    `ap_per_class` of the reference can be bound to an instance of this class unchanged."""

    def __init__(self, labels_text={}):
        self.reset()
        self.iouv = np.linspace(0.5, 0.95, 10)
        self.labels_text = labels_text

    def reset(self):
        self.n_pred, self.n_true, self.n_match = 0, 0, 0
        self.scores = torch.empty(0, dtype=torch.float32)
        self.y_pred = torch.empty(0, dtype=torch.int64)
        self.y_true = torch.empty(0, dtype=torch.int64)
        self.ious = torch.empty(0, dtype=torch.float32)
        self.m_pred = torch.empty(0, dtype=torch.int64)
        self.m_true = torch.empty(0, dtype=torch.int64)

    def add(self, output, target, iou_type='boxes', binned=False):
        """binned=True: match_predictions(..., binned=True), for region- or slide-scale inputs (same fields)."""
        # the reference's rule: mask IoU when asked for and both sides carry masks, box IoU otherwise
        use_masks = iou_type == 'masks' and ('masks' in output and 'masks' in target)
        m = match_predictions(output, target, float(self.iouv.min()), iou_type='masks' if use_masks else 'boxes',
                              binned=binned)
        n_pred, n_true = int(output['boxes'].shape[0]), int(target['boxes'].shape[0])
        self.m_pred = torch.cat([self.m_pred, (m['pred_idx'] + self.n_pred).cpu()])
        self.m_true = torch.cat([self.m_true, (m['true_idx'] + self.n_true).cpu()])
        self.ious = torch.cat([self.ious, m['ious'].cpu()])
        self.n_match += int(m['ious'].shape[0])
        self.y_true = torch.cat([self.y_true, target['labels'].to(torch.int64).cpu()])
        self.n_true += n_true
        self.y_pred = torch.cat([self.y_pred, m['labels'].to(torch.int64).cpu()])
        self.scores = torch.cat([self.scores, m['scores'].cpu()])
        self.n_pred += n_pred
