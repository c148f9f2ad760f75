"""Synthetic head-output generator (seeded).  Shared by bench.py, the tests and the golden generator
bench.py so that oracle and kernels always see identical bytes (SURVEY.md section 8d)."""
import math
from typing import List, Sequence, Tuple

import torch

# anchors of the reference's nuclei configs (metayolo/hub/yolov5l6-mask.yaml:7-11 uses 4 levels;
# the 3-level variant below is the P3-P5 subset named by BASELINE.json configs[1..2])
ANCHORS_3 = [[10, 13, 16, 30, 33, 23], [30, 61, 62, 45, 59, 119], [116, 90, 156, 198, 373, 326]]
ANCHORS_4 = [[19, 27, 44, 40, 38, 94], [96, 68, 86, 152, 180, 137], [140, 301, 303, 264, 238, 542],
             [436, 615, 739, 380, 925, 792]]
STRIDES_3 = [8, 16, 32]
STRIDES_4 = [8, 16, 32, 64]


def level_shapes(tile: int, strides: Sequence[int]) -> List[Tuple[int, int]]:
    return [(tile // s, tile // s) for s in strides]


def nuclei_logits(bs: int, tile: int, nc: int, n_cand: int, seed: int, anchors=ANCHORS_3, strides=STRIDES_3,
                  extra: int = 0, conf: float = 0.25, size_range=(12.0, 36.0), generator_device="cpu"):
    """Raw head logits [bs,na,ny,nx,5+nc+extra] per level such that ~n_cand rows per tile pass
    sigmoid(obj) > conf and decode to nuclei-sized boxes (SURVEY 8d, cfg 2/3).
    Objectness logits are N(mu,1) with mu chosen so the expected pass count is n_cand; the wh logits
    of every row are set so the decoded box has a side drawn from size_range."""
    g = torch.Generator(device=generator_device).manual_seed(seed)
    na = len(anchors[0]) // 2
    shapes = level_shapes(tile, strides)
    N = sum(na * ny * nx for ny, nx in shapes)
    frac = min(max(n_cand / N, 1e-6), 0.999)
    # P(N(mu,1) > logit(conf)) = frac
    z = math.sqrt(2.0) * torch.erfinv(torch.tensor(1.0 - 2.0 * frac, dtype=torch.float64)).item()  # Phi^-1(1-frac)
    mu = math.log(conf / (1.0 - conf)) - z
    dets = []
    for l, (ny, nx) in enumerate(shapes):
        no = 5 + nc + extra
        d = torch.randn((bs, na, ny, nx, no), generator=g, device=generator_device)
        d[..., 4] += mu
        a = torch.tensor(anchors[l], dtype=torch.float32, device=generator_device).view(na, 2)
        side = torch.rand((bs, na, ny, nx, 2), generator=g, device=generator_device) * (size_range[1] - size_range[0]) + size_range[0]
        # (2*sig)^2 * anchor = side  ->  sig = sqrt(side/anchor)/2, clamped into (0,1)
        sig = (side / a.view(1, na, 1, 1, 2)).sqrt().mul(0.5).clamp(0.02, 0.98)
        d[..., 2:4] = torch.log(sig / (1 - sig))
        dets.append(d.contiguous())
    return dets


# ------------------------------------------------------------------------------------------------ whole slide
def _tile_seed(seed: int, tile_index: int) -> int:
    return (int(seed) * 1000003 + int(tile_index) * 7919 + 12345) & 0x7fffffffffff


def _field_uniform(h: torch.Tensor, k: int) -> torch.Tensor:
    """Uniform k in [0, 1) of the global nuclei field at grid hash h: a pure function of (h, k)."""
    v = (h * (2 * k + 1) + 0x9E3779B9 * (k + 1)) & 0x7fffffff
    v = (v * 1103515245 + 12345) & 0x7fffffff
    return (v >> 7).to(torch.float32) / float(1 << 24)


def _field_nuclei(I: torch.Tensor, J: torch.Tensor, pitch: float, size_range):
    """Centre, box side and score of the field's nucleus at grid index (I, J) (int64 tensors)."""
    h = (I * 73856093) ^ (J * 19349663)
    cx = (I.float() + 0.15 + 0.7 * _field_uniform(h, 0)) * pitch
    cy = (J.float() + 0.15 + 0.7 * _field_uniform(h, 1)) * pitch
    side = size_range[0] + (size_range[1] - size_range[0]) * _field_uniform(h, 2)
    score = 0.3 + 0.65 * _field_uniform(h, 3)
    return cx, cy, side, score


def slide_tile_logits(rois: torch.Tensor, tile: int, nc: int, seed: int, pitch: float = 18.7, extra: int = 0,
                      conf: float = 0.25, size_range=(12.0, 30.0), strides=STRIDES_3, anchors=ANCHORS_3,
                      device="cuda", background_mu: float = -6.0, first_tile: int = 0, dtype=torch.float32):
    """Raw head logits for a batch of slide tiles (rois [bs,4] = x0,y0,x1,y1 from sliding_window_scanner) cut from
    ONE global nuclei field (SURVEY 8d, cfg 4): nuclei sit on a jittered grid of `pitch` px over the whole slide
    (~3 000 per 1024^2 tile); a nucleus is a pure function of its grid index, so the tiles that share an overlap band
    report the same nucleus with the same box (up to fp32 rounding of the tile-local decode) and a tile-dependent
    score jitter -- consistent duplicates for the merge NMS.  Every nucleus is written into the stride-8 level at the
    cell holding its centre, anchor chosen by size; all other rows are background (objectness logit ~ N(mu,1), far
    below the threshold).  Edge tiles (clipped windows) simply contain fewer nuclei.

    DETERMINISTIC AND RANK-INDEPENDENT: tile b of the batch is global tile `first_tile + b`, and everything random about
    it (background noise, score jitter, the `extra` coefficient channels) comes from a generator seeded with
    (seed, global tile index) alone -- however the tiles are batched or sharded over ranks, a tile's logits are the
    same bytes.  Two nuclei landing in the same (anchor, cell) are resolved by a fixed rule (the first in grid order
    wins), never by the order in which a scatter happens to commit duplicates.
    Returns the level tensors [bs,na,ny,nx,5+nc+extra] (`dtype`: float32, or float16 = what a half() model emits)."""
    bs = rois.shape[0]
    dev = torch.device(device)
    g = torch.Generator(device=dev)
    na = len(anchors[0]) // 2
    no = 5 + nc + extra
    shapes = level_shapes(tile, strides)
    dets = [torch.empty((bs, na, ny, nx, no), dtype=torch.float32, device=dev) for (ny, nx) in shapes]
    rois = rois.to(dev, torch.float32)
    rois_h = rois.cpu().tolist()
    s0 = float(strides[0])
    a0 = torch.tensor(anchors[0], dtype=torch.float32, device=dev).view(na, 2)
    ncell = int(math.ceil(tile / pitch)) + 1
    ny0, nx0 = shapes[0]
    for b in range(bs):
        g.manual_seed(_tile_seed(seed, first_tile + b))
        for d in dets:
            d[b] = torch.randn(tuple(d.shape[1:]), generator=g, device=dev)
            d[b, ..., 4] += background_mu
        x0, y0, x1, y1 = rois_h[b]
        i0, j0 = int(math.floor(x0 / pitch)), int(math.floor(y0 / pitch))
        ii = torch.arange(i0, i0 + ncell, device=dev, dtype=torch.int64)
        jj = torch.arange(j0, j0 + ncell, device=dev, dtype=torch.int64)
        J, I = torch.meshgrid(jj, ii, indexing='ij')
        cx, cy, side, score = _field_nuclei(I, J, pitch, size_range)
        inside = (cx >= x0) & (cx < x1) & (cy >= y0) & (cy < y1)
        cx, cy, side, score = cx[inside] - x0, cy[inside] - y0, side[inside], score[inside]
        jitter = torch.rand((ncell * ncell,), generator=g, device=dev)[:score.numel()]   # fixed draw count per tile
        if cx.numel() == 0:
            continue
        gx = torch.clamp((cx / s0).floor().long(), 0, nx0 - 1)
        gy = torch.clamp((cy / s0).floor().long(), 0, ny0 - 1)
        a = torch.where(side < 14.0, 0, torch.where(side < 23.0, 1, 2)).long()
        sx = ((cx / s0 - gx.float()) + 0.5) / 2.0
        sy = ((cy / s0 - gy.float()) + 0.5) / 2.0
        sw = (side / a0[a, 0]).sqrt() / 2.0
        sh = (side / a0[a, 1]).sqrt() / 2.0
        sc = (score + 0.04 * (jitter - 0.5)).clamp(conf + 0.02, 0.99)
        sig = torch.stack([sx, sy, sw, sh, sc], 1).clamp(0.02, 0.98)
        # one nucleus per (anchor, cell): the first in grid order wins (stable sort + first of every run)
        lin = (a * ny0 + gy) * nx0 + gx
        order = torch.argsort(lin, stable=True)
        ls = lin[order]
        first = torch.ones_like(ls, dtype=torch.bool)
        first[1:] = ls[1:] != ls[:-1]
        win = order[first]
        dets[0][b, a[win], gy[win], gx[win], :5] = torch.log(sig[win] / (1 - sig[win]))
    if dtype != torch.float32:
        dets = [d.to(dtype) for d in dets]
    return [d.contiguous() for d in dets]


def slide_tile_protos(n: int, tile: int, seed: int, first_tile: int = 0, nm: int = 32, device="cuda",
                      dtype=torch.float32) -> torch.Tensor:
    """Prototype maps [n, nm, tile/4, tile/4] of the global tiles [first_tile, first_tile + n): N(0,1), seeded per
    global tile index like slide_tile_logits (the same bytes however the tiles are batched or sharded)."""
    dev = torch.device(device)
    g = torch.Generator(device=dev)
    mh = tile // 4
    out = torch.empty((n, nm, mh, mh), dtype=dtype, device=dev)
    for b in range(n):
        g.manual_seed(_tile_seed(seed + 77, first_tile + b))
        out[b] = torch.randn((nm, mh, mh), generator=g, device=dev).to(dtype)
    return out


def ellipse_masks(centres: torch.Tensor, radii: torch.Tensor, H: int, W: int, chunk: int = 256) -> torch.Tensor:
    """Filled axis-aligned ellipses: centres / radii [n, 2] (x, y) in pixels -> [n, H, W] bool on their device."""
    dev = centres.device
    n = int(centres.shape[0])
    out = torch.empty((n, H, W), dtype=torch.bool, device=dev)
    y = torch.arange(H, dtype=torch.float32, device=dev)[None, :, None] + 0.5
    x = torch.arange(W, dtype=torch.float32, device=dev)[None, None, :] + 0.5
    for i in range(0, n, chunk):
        c, r = centres[i:i + chunk, :, None, None], radii[i:i + chunk, :, None, None]
        out[i:i + chunk] = ((x - c[:, 0]) / r[:, 0]) ** 2 + ((y - c[:, 1]) / r[:, 1]) ** 2 <= 1.0
    return out


def nuclei_match_case(k: int, g: int, size: int, seed: int, device="cuda"):
    """Seeded inputs of mask matching on a size x size canvas: g ground-truth nuclei (filled ellipses 12-36 px across),
    min(k, g) predictions that are jittered copies of them plus k - min(k, g) false positives, in random order; scores
    quantised to 1/256 (ties).  Returns (output, target) dicts of 'boxes' (the ellipses' boxes), 'scores', 'labels',
    'masks' ([n, size, size] bool) on `device`."""
    gen = torch.Generator().manual_seed(seed)
    cg = torch.rand((g, 2), generator=gen) * size
    rg = 6.0 + 12.0 * torch.rand((g, 2), generator=gen)
    m = min(k, g)
    cp = torch.cat([cg[:m] + torch.randn((m, 2), generator=gen) * 1.5, torch.rand((k - m, 2), generator=gen) * size])
    rp = torch.cat([rg[:m] * (1.0 + 0.08 * torch.randn((m, 2), generator=gen)),
                    6.0 + 12.0 * torch.rand((k - m, 2), generator=gen)]).clamp_min(1.0)
    perm = torch.randperm(k, generator=gen)
    cp, rp = cp[perm], rp[perm]
    scores = (torch.rand(k, generator=gen) * 256).round() / 256
    labels_p, labels_g = torch.randint(-1, 5, (k,), generator=gen), torch.randint(1, 5, (g,), generator=gen)

    def side(c, r, scores_labels):
        c, r = c.to(device), r.to(device)
        d = {'boxes': torch.cat([c - r, c + r], 1).clamp(0, size).contiguous(),
             'masks': ellipse_masks(c, r, size, size)}
        d.update({key: v.to(device) for key, v in scores_labels.items()})
        return d

    return side(cp, rp, {'scores': scores, 'labels': labels_p}), side(cg, rg, {'labels': labels_g})


def slide_nuclei(region, canvas=None, pitch: float = 18.7, size_range=(12.0, 30.0), nc: int = 4, seed: int = 0,
                 jitter: float = 0.0, device="cuda", rows_per_band: int = 256, masks_per_chunk: int = 1 << 20):
    """The nuclei of slide_tile_logits' global field (same `pitch` / `size_range`) whose centres lie in the slide region
    (x0, y0, x1, y1), as ground truth: 'boxes' [n, 4] (clipped to the canvas), 'labels' [n] int64 in 1..nc, 'scores'
    (the field's), and 'masks', filled ellipses (x radius side / 2, y radius 0.7-1.0 of it) built straight into a
    PackedMasks -- each one in a small patch of its own, never a canvas as large as the slide.  Coordinates are slide
    pixels on the (H, W) `canvas` (default: (y1, x1)).  Rows in grid order (row-major over the field's grid).
    jitter > 0: every nucleus moves by up to `jitter` px and its radii by up to jitter / 10 relative, seeded by (seed,
    grid index) -- a second, prediction-like set over the same field."""
    from .masks import PackedMasks
    dev = torch.device(device)
    x0, y0, x1, y1 = (float(v) for v in region)
    H, W = (int(y1), int(x1)) if canvas is None else (int(canvas[0]), int(canvas[1]))
    i0, i1 = int(math.floor(x0 / pitch)) - 1, int(math.ceil(x1 / pitch)) + 1
    j0, j1 = int(math.floor(y0 / pitch)) - 1, int(math.ceil(y1 / pitch)) + 1
    rmax = 0.5 * size_range[1] * (1.0 + jitter / 10.0)
    S = int(math.ceil(2.0 * rmax)) + 2                   # patch side: holds every ellipse
    boxes, labels, scores, cs, rs = [], [], [], [], []
    ii = torch.arange(i0, i1 + 1, device=dev, dtype=torch.int64)
    for jb in range(j0, j1 + 1, rows_per_band):
        jj = torch.arange(jb, min(jb + rows_per_band, j1 + 1), device=dev, dtype=torch.int64)
        J, I = torch.meshgrid(jj, ii, indexing='ij')
        I, J = I.reshape(-1), J.reshape(-1)
        cx, cy, side, score = _field_nuclei(I, J, pitch, size_range)
        keep = (cx >= x0) & (cx < x1) & (cy >= y0) & (cy < y1)
        I, J, cx, cy, side, score = I[keep], J[keep], cx[keep], cy[keep], side[keep], score[keep]
        h = (I * 73856093) ^ (J * 19349663)
        rx = 0.5 * side
        ry = rx * (0.7 + 0.3 * _field_uniform(h, 5))
        if jitter > 0:
            hs = h ^ (int(seed) * 83492791 + 1)
            cx = cx + jitter * (2.0 * _field_uniform(hs, 6) - 1.0)
            cy = cy + jitter * (2.0 * _field_uniform(hs, 7) - 1.0)
            rx = rx * (1.0 + jitter / 10.0 * (2.0 * _field_uniform(hs, 8) - 1.0))
            ry = ry * (1.0 + jitter / 10.0 * (2.0 * _field_uniform(hs, 9) - 1.0))
        labels.append(1 + torch.clamp((_field_uniform(h, 4) * nc).long(), max=nc - 1))
        scores.append(score)
        boxes.append(torch.stack([cx - rx, cy - ry, cx + rx, cy + ry], 1))
        cs.append(torch.stack([cx, cy], 1))
        rs.append(torch.stack([rx, ry], 1))
    boxes, c, r = torch.cat(boxes), torch.cat(cs), torch.cat(rs)
    boxes[:, 0::2] = boxes[:, 0::2].clamp(0, W)
    boxes[:, 1::2] = boxes[:, 1::2].clamp(0, H)
    # masks: patch S x S at (floor(cx - rx), floor(cy - ry)); pixel centres tested as ellipse_masks does
    n = int(c.shape[0])
    geoms, offs, bits, base = [], [], [], 0
    k = torch.arange(S, device=dev, dtype=torch.float32)
    for a in range(0, n, masks_per_chunk):
        cc, rr = c[a:a + masks_per_chunk], r[a:a + masks_per_chunk]
        org = torch.floor(cc - rr)
        px = org[:, 0, None] + k[None, :]                 # [m, S] pixel x
        py = org[:, 1, None] + k[None, :]
        fx = ((px + 0.5 - cc[:, 0, None]) / rr[:, 0, None]) ** 2
        fy = ((py + 0.5 - cc[:, 1, None]) / rr[:, 1, None]) ** 2
        inside = (fy[:, :, None] + fx[:, None, :] <= 1.0)
        inside &= ((py >= 0) & (py < H))[:, :, None] & ((px >= 0) & (px < W))[:, None, :]
        pm = PackedMasks.from_dense(inside)
        g = pm.geom.clone()
        live = (g[:, 2] > 0) & (g[:, 3] > 0)
        g[:, 0] += torch.where(live, org[:, 0].to(torch.int32), 0)
        g[:, 1] += torch.where(live, org[:, 1].to(torch.int32), 0)
        geoms.append(g)
        offs.append(pm.offsets[:-1] + base)
        bits.append(pm.bits)
        base += int(pm.bits.numel())
    if n == 0:
        geoms, offs = [torch.zeros((0, 4), dtype=torch.int32, device=dev)], [torch.zeros(0, dtype=torch.int64, device=dev)]
    masks = PackedMasks(torch.cat(geoms).contiguous(),
                        torch.cat(offs + [torch.tensor([base], dtype=torch.int64, device=dev)]),
                        torch.cat(bits) if bits else torch.zeros(0, dtype=torch.int32, device=dev), H, W,
                        torch.zeros(1, dtype=torch.int32, device=dev))
    return {'boxes': boxes.contiguous(), 'labels': torch.cat(labels), 'scores': torch.cat(scores), 'masks': masks}
