"""ORACLE -- test infrastructure, not product code.

The sparse form of ``mask_match.apmeter_match`` / ``port.apmeter_match`` (APMeter.add's matching,
metayolo/models/metrics.py:270-303) for region- and slide-scale sizes, where the dense P x G IoU matrix cannot exist.
It finds candidate pairs with a k-d tree over box centres -- a mechanism of its own, independent of the grid the binned
kernels use -- and computes each candidate's IoU exactly: port.box_iou's fp32 expression for boxes, pixel counts of
masks unpacked on the CPU for masks.  Checked against the dense forms in tests/test_match_binned_host.py.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

from .mask_match import _mask_set


def _rects(b: np.ndarray):
    """Boxes [n, 4] (fp32 xyxy) -> (centres, half diagonals, usable): a box with a non-finite coordinate or without
    positive width and height overlaps nothing (its IoU with anything is 0 or NaN)."""
    b64 = b.astype(np.float64)
    ok = np.isfinite(b64).all(1) & (b64[:, 2] > b64[:, 0]) & (b64[:, 3] > b64[:, 1])
    b64 = np.where(ok[:, None], b64, 0.0)
    c = 0.5 * (b64[:, :2] + b64[:, 2:])
    r = 0.5 * np.hypot(b64[:, 2] - b64[:, 0], b64[:, 3] - b64[:, 1])
    return c, r, ok


def _candidates(bp: np.ndarray, bg: np.ndarray):
    """(i, j) of every pair of boxes that may overlap: centre distance <= the sum of the two half diagonals, found with
    a k-d tree over the centres (radius: the largest half diagonals of both sides)."""
    from scipy.spatial import cKDTree
    cp, rp, okp = _rects(bp)
    cg, rg, okg = _rects(bg)
    ip, ig = np.flatnonzero(okp), np.flatnonzero(okg)
    if len(ip) == 0 or len(ig) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    radius = (rp[ip].max() + rg[ig].max()) * (1 + 1e-9) + 1e-6
    lists = cKDTree(cp[ip]).query_ball_tree(cKDTree(cg[ig]), radius)
    n = np.array([len(l) for l in lists], dtype=np.int64)
    i = np.repeat(ip, n)
    j = ig[np.concatenate([np.asarray(l, dtype=np.int64) for l in lists])] if n.sum() else np.zeros(0, np.int64)
    return i, j


def _pixel_sets(m, H: int, W: int):
    """Set pixels of every mask as a CSR matrix [n, H * W] (row = mask, column = y * W + x): from a dense [n, H, W]
    tensor, or from a PackedMasks' windows and bit planes unpacked with numpy."""
    from scipy.sparse import csr_matrix
    if isinstance(m, torch.Tensor):
        s = _mask_set(m.cpu()).flatten(1).numpy()
        r, col = np.nonzero(s)
        n = s.shape[0]
    else:
        geom, off = m.geom.cpu().numpy().astype(np.int64), m.offsets.cpu().numpy()
        bits = m.bits.cpu().numpy().view(np.uint32)
        n = geom.shape[0]
        w, h = np.maximum(geom[:, 2], 0), np.maximum(geom[:, 3], 0)
        w = np.where(h > 0, w, 0)
        wpr = (w + 31) // 32
        nw = wpr * h
        mask = np.repeat(np.arange(n), nw)
        local = np.arange(int(nw.sum())) - np.repeat(np.cumsum(nw) - nw, nw)
        row, wd = local // wpr[mask], local % wpr[mask]
        words = bits[off[:-1][mask] + local]
        b = np.unpackbits(words.astype('<u4').view(np.uint8).reshape(-1, 4), axis=1, bitorder='little')
        k, bit = np.nonzero(b)
        x = wd[k] * 32 + bit
        keep = x < w[mask[k]]
        k, x = k[keep], x[keep]
        r = mask[k]
        col = (geom[r, 1] + row[k]) * W + geom[r, 0] + x
    return csr_matrix((np.ones(len(r), np.int64), (r, col)), shape=(n, H * W))


def apmeter_match_sparse(output: Dict[str, torch.Tensor], target: Dict[str, torch.Tensor], iou_min: float = 0.5,
                         iou_type: str = 'boxes'):
    """apmeter_match (iou_type='masks') / port.apmeter_match (iou_type='boxes') for sizes where the dense P x G matrix
    cannot exist.  Candidate pairs come from a k-d tree over box centres (mask windows for masks), the IoU of each is
    exact: port.box_iou's fp32 expression, or float32(inter) / float32(union) with intersections counted over the
    pixels of the unpacked masks.  iou_min > 0 (pairs that do not overlap never match).  Same sorts and returns as
    apmeter_match."""
    assert iou_min > 0
    thr = np.float32(iou_min)
    o_scores, order = torch.sort(output['scores'].cpu(), descending=True, stable=True)
    o_labels = output['labels'].cpu()[order]
    order = order.numpy()
    if iou_type == 'masks':
        pm, gm = output['masks'], target['masks']
        H, W = (pm.H, pm.W) if not isinstance(pm, torch.Tensor) else tuple(pm.shape[-2:])
        A, B = _pixel_sets(pm, H, W)[order], _pixel_sets(gm, H, W)
        # candidates over the pixel bounding rectangles [x0, x1 + 1) x [y0, y1 + 1) of the set pixels
        def bounds(S):
            n = S.shape[0]
            out = np.full((n, 4), np.nan, np.float32)
            r = np.repeat(np.arange(n), np.diff(S.indptr))
            if len(r):
                y, x = S.indices // W, S.indices % W
                for c, (v, f) in enumerate([(x, np.minimum), (y, np.minimum), (x + 1, np.maximum), (y + 1, np.maximum)]):
                    acc = np.full(n, np.iinfo(np.int64).max if f is np.minimum else -1, np.int64)
                    f.at(acc, r, v)
                    out[:, c] = np.where(np.diff(S.indptr) > 0, acc, np.nan)
            return out
        i, j = _candidates(bounds(A), bounds(B))
        inter = np.asarray(A[i].multiply(B[j]).sum(1)).ravel().astype(np.int64)
        ap, ag = np.diff(A.indptr).astype(np.int64), np.diff(B.indptr).astype(np.int64)
        with np.errstate(invalid='ignore', divide='ignore'):
            ious = inter.astype(np.float32) / (ap[i] + ag[j] - inter).astype(np.float32)
    else:
        bp = output['boxes'].cpu().numpy().astype(np.float32)[order]
        bg = target['boxes'].cpu().numpy().astype(np.float32)
        i, j = _candidates(bp, bg)
        a, b = bp[i], bg[j]
        with np.errstate(invalid='ignore', over='ignore'):
            w = np.maximum(np.minimum(a[:, 2], b[:, 2]) - np.maximum(a[:, 0], b[:, 0]), np.float32(0))
            h = np.maximum(np.minimum(a[:, 3], b[:, 3]) - np.maximum(a[:, 1], b[:, 1]), np.float32(0))
            inter = w * h
            area_a = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1])
            area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
            ious = inter / (area_a + area_b - inter)
    keep = ious >= thr
    i, j, ious = i[keep], j[keep], ious[keep]
    o = np.lexsort((j, i))                                  # torch.where's row-major order ...
    i, j, ious = i[o], j[o], ious[o]
    o2 = np.argsort(-ious, kind='stable')                   # ... then IoU descending, stable
    return (o_scores, o_labels, torch.from_numpy(i[o2].astype(np.int64)), torch.from_numpy(j[o2].astype(np.int64)),
            torch.from_numpy(ious[o2].astype(np.float32)))
