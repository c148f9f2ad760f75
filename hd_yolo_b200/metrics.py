"""Prediction <-> ground-truth matching on the device (SURVEY 8f rank 2): host mirror of ``box_iou``
(metayolo/models/utils_general.py:247-265) and of the matching half of ``APMeter.add``
(metayolo/models/metrics.py:270-303), over ``hdy_box_iou`` / ``hdy_match_pairs``.

The reference moves every image's detections to the host and builds a dense k x g IoU matrix there; here the
matching pairs are produced on the device and only they (a few hundred rows per image) are copied back.
``APMeter`` keeps the reference's accumulator fields (CPU tensors), so the reference's own ``ap_per_class`` /
plotting code runs on it unchanged.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from ._lib import HdyError, ptr
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
                      cap: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """The device half of APMeter.add (metrics.py:271-284), box IoU only.

    Returns (all on the device): 'order' (rows of `output` by score, descending, ties by lower row), 'scores' /
    'labels' in that order, and the matching pairs 'pred_idx' (rank in `order`), 'true_idx', 'ious' sorted by IoU
    descending (ties in row-major (pred, true) order).  One D2H read (the pair count)."""
    boxes, scores, gts = output['boxes'], output['scores'], target['boxes']
    _need_cuda(boxes, "output['boxes']")
    _need_cuda(scores, "output['scores']")
    _need_cuda(gts, "target['boxes']")
    dev = boxes.device
    k, g = int(boxes.shape[0]), int(gts.shape[0])
    i64 = dict(dtype=torch.int64, device=dev)
    empty = {'pred_idx': torch.empty(0, **i64), 'true_idx': torch.empty(0, **i64),
             'ious': torch.empty(0, dtype=torch.float32, device=dev)}
    if k == 0:
        return {'order': torch.empty(0, **i64), 'scores': scores.reshape(0), 'labels': output['labels'].reshape(0), **empty}
    boxes = _aligned16(boxes.contiguous())
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
    gts = _aligned16(gts.contiguous())
    # 2. pairs with iou >= iou_min
    cap = int(cap) if cap is not None else max(4 * max(k, g), 1024)
    while True:
        pk = torch.empty(cap, dtype=torch.int64, device=dev)
        pb = torch.empty((cap, 4), dtype=torch.float32, device=dev)
        pc = _Cand.__new__(_Cand)
        pc.bs, pc.cap, pc.keys, pc.boxes, pc.cls = 1, cap, pk, pb, None
        pc.counts = torch.zeros(2, dtype=torch.int32, device=dev)
        kc = torch.tensor([k, g], dtype=torch.int32).to(dev)
        _call("hdy_match_pairs", ptr(boxes), ptr(order32), ptr(kc[0:1]), 1, k, ptr(gts), ptr(kc[1:2]), g,
              float(np.float32(iou_min)), cap, ptr(pk), ptr(pb), ptr(pc.counts), pc.status_ptr, _stream())
        n_match = int(pc.counts[0].item())          # the reference's torch.where synchronises here too
        if n_match <= cap:
            break
        cap = n_match                                 # a crowded image: retry with the size the kernel reported
    if n_match == 0:
        return {**res, **empty}
    # 3. IoU-descending order of the pairs: a key sort (pairs of one prediction share a box -- as an "NMS that only
    #    sorts" they would all land in one spatial-hash cell); index and IoU are read back out of the key
    pk = pk[:n_match].contiguous()
    sort_keys(pk)
    pidx = pk & 0xffffffff
    res.update({'pred_idx': pidx // g, 'true_idx': pidx % g, 'ious': _key_scores(pk)})
    return res


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

    def add(self, output, target, iou_type='boxes'):
        if iou_type == 'masks' and ('masks' in output and 'masks' in target):
            raise HdyError("mask IoU matching is not on the device path; use iou_type='boxes'")
        m = match_predictions(output, target, float(self.iouv.min()))
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
