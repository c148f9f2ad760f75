"""ORACLE -- test infrastructure, not product code.

Boundary polygons of bit-packed masks (the contract of PackedMasks.contours, DESIGN §3.10), restated over the general
edge graph rather than by walking a bit plane:
  * every unit edge between a set and an unset pixel is a graph edge, directed so that the set pixel is on its right
    (y down);
  * at a corner with one incoming and one outgoing edge the successor is that edge; at a saddle corner (two of each)
    the successor of an edge is the outgoing edge a right turn away;
  * the cycles of the successor map are the rings; a ring's vertices are the corners where the heading changes, rotated
    to start at the least one in (y, x) order; a mask's rings are sorted by their start;
  * the 4-connected components come from scipy.ndimage.label; a ring belongs to the component of the pixel on the right
    of any of its edges, and a component's exterior ring is its ring with positive shoelace area.
Also: the even-odd rasteriser, the local vertex count and the hole count the tests check the rings against.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import torch
from scipy import ndimage

# headings 0 = +x, 1 = +y, 2 = -x, 3 = -y; the pixel on the right of an edge leaving corner (x, y) heading d
_RIGHT_PIXEL = np.array([[0, 0], [-1, 0], [-1, -1], [0, -1]])


def _padded(m: np.ndarray) -> np.ndarray:
    P = np.zeros((m.shape[0] + 2, m.shape[1] + 2), bool)
    P[1:-1, 1:-1] = m
    return P


def mask_rings(m: np.ndarray) -> Tuple[List[np.ndarray], List[int]]:
    """One mask [h, w] bool -> (rings, parent): rings [n_i, 2] int64 (x, y) corners in window coordinates, in start
    order; parent[r] = -1 for an exterior ring, else the index of its component's exterior ring."""
    m = np.asarray(m, bool)
    h, w = m.shape
    if not m.any():
        return [], []
    P = _padded(m)
    above, below = P[:-1, 1:-1], P[1:, 1:-1]              # [h+1, w]: pixels (x, y-1) and (x, y) of corner row y
    left, right = P[1:-1, :-1], P[1:-1, 1:]               # [h, w+1]: pixels (x-1, y) and (x, y) of corner column x
    parts = []
    for sel, d, off in ((below & ~above, 0, (0, 0)), (above & ~below, 2, (1, 0)),
                        (left & ~right, 1, (0, 0)), (right & ~left, 3, (0, 1))):
        y, x = np.nonzero(sel)
        parts.append(np.stack([x + off[0], y + off[1], np.full_like(x, d)], 1))
    e = np.concatenate(parts)                              # start x, start y, heading
    step = np.array([[1, 0], [0, 1], [-1, 0], [0, -1]])
    end = e[:, :2] + step[e[:, 2]]
    W1 = w + 1
    out = np.full(((h + 1) * W1, 4), -1, np.int64)
    out[e[:, 1] * W1 + e[:, 0], e[:, 2]] = np.arange(len(e))
    at_end = out[end[:, 1] * W1 + end[:, 0]]
    n_out = (at_end >= 0).sum(1)
    assert ((n_out == 1) | (n_out == 2)).all(), "every corner on a boundary has one or two outgoing edges"
    succ = np.where(n_out == 1, at_end.max(1), at_end[np.arange(len(e)), (e[:, 2] + 1) % 4])
    assert (succ >= 0).all() and len(np.unique(succ)) == len(e), "the successor map is a permutation"
    labels, _ = ndimage.label(m)
    seen = np.zeros(len(e), bool)
    rings, comp, area2 = [], [], []
    for s in range(len(e)):
        if seen[s]:
            continue
        cyc = [s]
        seen[s] = True
        nxt = succ[s]
        while nxt != s:
            cyc.append(nxt)
            seen[nxt] = True
            nxt = succ[nxt]
        c = e[np.array(cyc)]
        turn = c[:, 2] != np.roll(c[:, 2], 1)
        v = c[turn][:, :2]
        k = np.lexsort((v[:, 0], v[:, 1]))[0]
        v = np.roll(v, -k, axis=0)
        x, y = v[:, 0], v[:, 1]
        area2.append(int((x * np.roll(y, -1) - np.roll(x, -1) * y).sum()))
        px, py = c[0, :2] + _RIGHT_PIXEL[c[0, 2]]
        comp.append(int(labels[py, px]))
        rings.append(v.astype(np.int64))
    order = sorted(range(len(rings)), key=lambda r: (int(rings[r][0, 1]), int(rings[r][0, 0])))
    rings = [rings[r] for r in order]
    comp = [comp[r] for r in order]
    area2 = [area2[r] for r in order]
    ext = {}
    for r, (c, a) in enumerate(zip(comp, area2)):
        if a > 0:
            assert c not in ext, "one exterior ring per component"
            ext[c] = r
    return rings, [-1 if a > 0 else ext[c] for c, a in zip(comp, area2)]


def unpack_windows(geom, offsets, bits) -> List[Tuple[int, int, np.ndarray]]:
    """Cropped bit planes (CPU or CUDA tensors) -> [(x0, y0, [h, w] bool)] per mask; padding bits are ignored."""
    geom = geom.cpu().numpy()
    offsets = offsets.cpu().numpy()
    bits = bits.cpu().numpy().view('<u4')
    out = []
    for i, (x0, y0, w, h) in enumerate(geom.tolist()):
        if w <= 0 or h <= 0:
            out.append((int(x0), int(y0), np.zeros((0, 0), bool)))
            continue
        wpr = (w + 31) // 32
        o = int(offsets[i])
        rows = np.unpackbits(bits[o:o + wpr * h].view(np.uint8), bitorder='little').reshape(h, wpr * 32)[:, :w]
        out.append((int(x0), int(y0), rows.astype(bool)))
    return out


def contours(windows: Sequence[Tuple[int, int, np.ndarray]]) -> dict:
    """The arrays of PackedMasks.contours() for [(x0, y0, mask)]: mask_rings [K+1], ring_verts [R+1] int64, xy [V, 2]
    int32 in canvas pixels, parent [R] int32 global ring indices."""
    starts, ring_verts, xy, parent = [0], [0], [], []
    for x0, y0, m in windows:
        rings, par = mask_rings(m) if m.size else ([], [])
        base = starts[-1]
        for v, p in zip(rings, par):
            xy.append(v + np.array([x0, y0]))
            ring_verts.append(ring_verts[-1] + len(v))
            parent.append(-1 if p < 0 else base + p)
        starts.append(base + len(rings))
    xy = np.concatenate(xy).astype(np.int32) if xy else np.zeros((0, 2), np.int32)
    return {'mask_rings': torch.tensor(starts, dtype=torch.int64),
            'ring_verts': torch.tensor(ring_verts, dtype=torch.int64),
            'xy': torch.from_numpy(xy.reshape(-1, 2)), 'parent': torch.tensor(parent, dtype=torch.int32)}


def signed_area(v: np.ndarray) -> float:
    x, y = v[:, 0].astype(np.int64), v[:, 1].astype(np.int64)
    return 0.5 * float((x * np.roll(y, -1) - np.roll(x, -1) * y).sum())


def rasterize_even_odd(rings: Sequence[np.ndarray], h: int, w: int) -> np.ndarray:
    """Even-odd fill of rectilinear rings (window coordinates) -> [h, w] bool: pixel (x, y) is inside iff a ray from
    its centre toward +x crosses an odd number of vertical edges."""
    cross = np.zeros((h, w + 2), np.int64)
    for v in rings:
        a, b = v, np.roll(v, -1, axis=0)
        vert = a[:, 0] == b[:, 0]
        for (xa, ya), (_, yb) in zip(a[vert], b[vert]):
            lo, hi = min(ya, yb), max(ya, yb)
            cross[lo:hi, xa] += 1
    suffix = np.cumsum(cross[:, ::-1], axis=1)[:, ::-1]    # suffix[:, c] = crossings at columns >= c
    return (suffix[:, 1:w + 1] % 2).astype(bool)


def local_vertex_count(m: np.ndarray) -> int:
    """Corners whose four pixels hold an odd number of set pixels, plus two per saddle corner."""
    P = _padded(np.asarray(m, bool)).astype(np.int64)
    nw, ne, sw, se = P[:-1, :-1], P[:-1, 1:], P[1:, :-1], P[1:, 1:]
    odd = (nw + ne + sw + se) % 2
    saddle = (nw == se) & (ne == sw) & (nw != ne)
    return int(odd.sum() + 2 * saddle.sum())


def hole_count(m: np.ndarray) -> int:
    """Bounded 8-connected background components."""
    _, n = ndimage.label(~_padded(np.asarray(m, bool)), structure=np.ones((3, 3), bool))
    return n - 1


def component_count(m: np.ndarray) -> int:
    return int(ndimage.label(np.asarray(m, bool))[1])
