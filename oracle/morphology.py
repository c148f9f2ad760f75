"""ORACLE -- test infrastructure, not product code.

Morphometry of bit-packed masks (the contract of PackedMasks.measure, DESIGN §3.10b), restated without the kernels'
word arithmetic:
  * moments with numpy over np.nonzero of the unpacked window;
  * corner patterns over the 2 x 2 windows of the zero-padded mask;
  * the convex hull by Andrew's monotone chain over all four corners of every set pixel, in Python ints, then rotated to
    start at its least vertex in (y, x) order (Andrew's order is already the exterior rings' rotational sense);
  * the calipers brute force over vertex pairs and (edge, vertex) pairs;
  * convex_perimeter and feret_min with the same fp64 expressions and summation order as the contract, and the derived
    columns with the same expressions as MaskMeasurements.
"""
from __future__ import annotations

import math
from typing import List, Sequence, Tuple

import numpy as np
import torch

FIELDS = ("area", "bbox", "moments", "quads", "hull", "hull_len")


def convex_hull(m: np.ndarray) -> List[Tuple[int, int]]:
    """[(x, y)] vertices of the convex hull of the set pixels' unit squares (window coordinates), collinear points
    dropped, starting at the least vertex in (y, x) order, positive shoelace sum; [] for an empty mask."""
    ys, xs = np.nonzero(np.asarray(m, bool))
    if xs.size == 0:
        return []
    return hull_of_points(np.concatenate([xs, xs + 1, xs, xs + 1]), np.concatenate([ys, ys, ys + 1, ys + 1]))


def hull_of_points(cx, cy) -> List[Tuple[int, int]]:
    """The convex hull of lattice points (x, y), coordinates in [0, 2^20), in the order convex_hull gives."""
    cx, cy = np.asarray(cx, np.int64), np.asarray(cy, np.int64)
    key = np.unique(cx * (1 << 20) + cy)
    pts = [(int(k >> 20), int(k & ((1 << 20) - 1))) for k in key]      # sorted by (x, y)

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    lower, upper = [], []
    for p in pts:
        while len(lower) >= 2 and cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    for p in reversed(pts):
        while len(upper) >= 2 and cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    hull = lower[:-1] + upper[:-1]
    k = min(range(len(hull)), key=lambda j: (hull[j][1], hull[j][0]))
    return hull[k:] + hull[:k]


def quads(m: np.ndarray) -> Tuple[int, int, int, int]:
    """(n1, n2, n3, nD) over the (w+1)(h+1) corners of the window."""
    P = np.zeros((m.shape[0] + 2, m.shape[1] + 2), np.int64)
    P[1:-1, 1:-1] = m
    nw, ne, sw, se = P[:-1, :-1], P[:-1, 1:], P[1:, :-1], P[1:, 1:]
    s = nw + ne + sw + se
    diag = (s == 2) & (nw == se)
    return int((s == 1).sum()), int(((s == 2) & ~diag).sum()), int((s == 3).sum()), int(diag.sum())


def measure_window(x0: int, y0: int, m: np.ndarray) -> dict:
    """The exact fields of one mask [h, w] bool whose window starts at canvas pixel (x0, y0)."""
    m = np.asarray(m, bool)
    ys, xs = np.nonzero(m)
    zero = {"area": 0, "bbox": [0] * 4, "moments": [0] * 5, "quads": [0] * 4, "hull": [0] * 3, "hull_len": [0.0] * 2}
    if xs.size == 0:
        return zero
    xs, ys = xs.astype(np.int64), ys.astype(np.int64)
    hull, hull_len = hull_fields(convex_hull(m))
    return {"area": int(xs.size),
            "bbox": [x0 + int(xs.min()), y0 + int(ys.min()), x0 + int(xs.max()) + 1, y0 + int(ys.max()) + 1],
            "moments": [int(xs.sum()), int(ys.sum()), int((xs * xs).sum()), int((ys * ys).sum()), int((xs * ys).sum())],
            "quads": list(quads(m)), "hull": hull, "hull_len": hull_len}


def hull_fields(hull: List[Tuple[int, int]]):
    """([convex_area2, feret_max2, hull_verts], [convex_perimeter, feret_min]) of a hull in convex_hull's order."""
    n = len(hull)
    H = np.array(hull, np.int64)
    E = np.roll(H, -1, axis=0) - H                                      # edge j: vertex j -> j + 1
    area2 = int((H[:, 0] * np.roll(H[:, 1], -1) - np.roll(H[:, 0], -1) * H[:, 1]).sum())
    D = H[None, :, :] - H[:, None, :]                                   # D[j, v] = vertex v - vertex j
    feret_max2 = int((D ** 2).sum(2).max())
    cr = np.abs(E[:, None, 0] * D[:, :, 1] - E[:, None, 1] * D[:, :, 0]).max(1)
    feret_min = float(np.min(cr.astype(np.float64) / np.sqrt((E ** 2).sum(1).astype(np.float64))))
    perim = 0.0
    for j in range(n):
        perim += math.sqrt(float(int(E[j, 0]) ** 2 + int(E[j, 1]) ** 2))
    return [area2, feret_max2, n], [perim, feret_min]


def measure(windows: Sequence[Tuple[int, int, np.ndarray]]) -> dict:
    """The arrays hdy_mask_measure writes for [(x0, y0, mask)], as CPU tensors: area [K] i32, bbox [K,4] i32, moments
    [K,5] i64, quads [K,4] i32, hull [K,3] i64 (convex_area2, feret_max2, hull_verts), hull_len [K,2] f64
    (convex_perimeter, feret_min)."""
    rows = [measure_window(x0, y0, m) for x0, y0, m in windows]
    dt = {"area": torch.int32, "bbox": torch.int32, "moments": torch.int64, "quads": torch.int32,
          "hull": torch.int64, "hull_len": torch.float64}
    width = {"area": None, "bbox": 4, "moments": 5, "quads": 4, "hull": 3, "hull_len": 2}
    out = {}
    for f in FIELDS:
        t = torch.tensor([r[f] for r in rows], dtype=dt[f])
        out[f] = t if width[f] is None else t.reshape(-1, width[f])
    return out


def columns(fields: dict, geom) -> dict:
    """The derived columns of MaskMeasurements, in numpy fp64 with the same expressions, from the exact fields (as
    returned by measure) and the windows geom [K, 4]."""
    A = np.asarray(fields["area"], np.int64).astype(np.float64)
    m = np.asarray(fields["moments"], np.int64).astype(np.float64)
    g = np.asarray(geom, np.int64).astype(np.float64)
    q = np.asarray(fields["quads"], np.int64)
    n1, n2, n3, nd = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    hull = np.asarray(fields["hull"], np.int64)
    hull_len = np.asarray(fields["hull_len"], np.float64)
    b = np.asarray(fields["bbox"], np.int64)
    with np.errstate(divide="ignore", invalid="ignore"):
        ps = n2.astype(np.float64) + (n1 + n3 + 2 * nd).astype(np.float64) * math.sqrt(0.5)
        convex_area = hull[:, 0].astype(np.float64) / 2
        mx, my = m[:, 0] / A, m[:, 1] / A
        c20, c02, c11 = m[:, 2] / A - mx * mx, m[:, 3] / A - my * my, m[:, 4] / A - mx * my
        d = (c20 - c02) / 2
        half, root = (c20 + c02) / 2, np.sqrt(d * d + c11 * c11)
        l1, l2 = half + root, np.maximum(half - root, 0.0)
        return {"centroid_x": g[:, 0] + m[:, 0] / A + 0.5, "centroid_y": g[:, 1] + m[:, 1] / A + 0.5,
                "area": A, "perimeter": (n1 + n2 + n3 + 2 * nd).astype(np.float64), "perimeter_smooth": ps,
                "euler": (n1 - n3 + 2 * nd) // 4, "convex_area": convex_area, "convex_perimeter": hull_len[:, 0],
                "solidity": A / convex_area,
                "extent": A / ((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])).astype(np.float64),
                "equivalent_diameter": np.sqrt(4 * A / math.pi), "circularity": 4 * math.pi * A / (ps * ps),
                "major_axis": 4 * np.sqrt(l1), "minor_axis": 4 * np.sqrt(l2),
                "eccentricity": np.where(l1 == 0, 0.0, np.sqrt(1 - l2 / l1)),
                "orientation": np.arctan2(2 * c11, c20 - c02) / 2,
                "feret_max": np.sqrt(hull[:, 1].astype(np.float64)), "feret_min": hull_len[:, 1]}
