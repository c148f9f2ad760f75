"""ORACLE -- test infrastructure, not product code.

The iou_type='masks' branch of APMeter.add (metayolo/models/metrics.py:270-303): mask IoU and the matching built on
it, next to the box form in ``oracle/port.py`` (whose ordering, ties and accumulator fields it shares).  No reference
output of this branch exists to pin against, so the definition in ``mask_iou`` is the contract: parity unpinned, pinned
instead on hand-computable cases (tests/test_mask_match_host.py).
"""
from __future__ import annotations

from typing import Dict

import torch

from . import port


def _mask_set(m: torch.Tensor) -> torch.Tensor:
    """Set pixels of [n, H, W] or [n, 1, H, W] masks: > 0.5 for floating point (what `paste_masks_in_image(...) > 0.5`
    holds), nonzero for integer and bool masks."""
    if m.dim() == 4:
        m = m[:, 0]
    if m.dtype == torch.bool:
        return m
    return m > 0.5 if m.dtype.is_floating_point else m != 0


def mask_iou(m1: torch.Tensor, m2: torch.Tensor, chunk: int = 256) -> torch.Tensor:
    """Mask IoU [N, H, W] x [M, H, W] -> fp32 [N, M].  inter = pixels set in both, union = area1 + area2 - inter (exact
    integers), iou = float32(inter) / float32(union), each rounded to nearest; 0/0 = NaN.  inter is an fp32 product of
    the flattened 0/1 masks with TF32 off: every partial sum is an integer <= H * W <= 2^24, so it is exact in any
    summation order, on CPU or CUDA tensors."""
    a, b = _mask_set(m1), _mask_set(m2)
    assert a.shape[1:] == b.shape[1:], "both mask sets must lie on one canvas"
    assert a.shape[1] * a.shape[2] <= 2 ** 24, "fp32 partial sums of more than 2^24 pixels are not exact"
    fa, fb = a.flatten(1), b.flatten(1)
    inter = torch.empty((fa.shape[0], fb.shape[0]), dtype=torch.int64, device=fa.device)
    fbf = fb.float()
    prec = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision('highest')      # no TF32 / bf16 passes: exact integer sums
    try:
        for i in range(0, fa.shape[0], chunk):
            inter[i:i + chunk] = (fa[i:i + chunk].float() @ fbf.T).to(torch.int64)
    finally:
        torch.set_float32_matmul_precision(prec)
    union = fa.sum(1)[:, None] + fb.sum(1)[None, :] - inter        # bool sums: int64
    return inter.float() / union.float()


def apmeter_match(output: Dict[str, torch.Tensor], target: Dict[str, torch.Tensor], iou_min: float = 0.5):
    """port.apmeter_match with mask_iou of output['masks'] / target['masks'] in place of box_iou: predictions by score
    (descending, stable), pairs with iou >= iou_min sorted by IoU (descending, stable).  Returns o_scores, o_labels,
    pred_idx (rank in score order), true_idx, ious."""
    o_scores, order = torch.sort(output['scores'], descending=True, stable=True)
    o_labels = output['labels'][order]
    ious = mask_iou(output['masks'], target['masks'])[order]
    pred_idx, true_idx = torch.where(ious >= iou_min)
    ious, o2 = torch.sort(ious[pred_idx, true_idx], descending=True, stable=True)
    return o_scores, o_labels, pred_idx[o2], true_idx[o2], ious


class APMeterState(port.APMeterState):
    """port.APMeterState with APMeter.add's iou_type: mask IoU when asked for and both sides carry masks, box IoU
    otherwise (the reference's rule)."""

    def add(self, output, target, iou_min: float = 0.5, iou_type: str = 'boxes'):
        if not (iou_type == 'masks' and 'masks' in output and 'masks' in target):
            return super().add(output, target, iou_min)
        s, l, p, t, i = apmeter_match(output, target, iou_min)
        self.m_pred = torch.cat([self.m_pred, p + self.n_pred])
        self.m_true = torch.cat([self.m_true, t + self.n_true])
        self.ious = torch.cat([self.ious, i])
        self.n_match += len(i)
        self.y_true = torch.cat([self.y_true, target['labels']])
        self.n_true += len(target['boxes'])
        self.y_pred = torch.cat([self.y_pred, l])
        self.scores = torch.cat([self.scores, s])
        self.n_pred += len(output['boxes'])
