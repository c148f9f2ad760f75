"""GPU tests of PackedMasks.measure() (csrc/measure.cu): every exact field bit-identical to oracle/morphology.py on
hand-made, random, packed-by-the-library and slide-scale planes, on both kernel paths (windows up to 64 x 64 one warp
per mask, larger ones one CTA per mask); the derived columns against the oracle's; identities with areas() and
contours() on every mask at slide scale; a slide result measured and exported."""
import json
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import synth
from hd_yolo_b200.masks import PackedMasks
from oracle import contours as oc
from oracle import morphology as om
from test_gpu_contours import _local_vertex_counts, _pack, _shapes

pytestmark = pytest.mark.gpu


def _exact(m):
    return {"area": m.area, "bbox": m.bbox, "moments": m.moments, "quads": m.quads,
            "hull": torch.stack([m.convex_area2, m.feret_max2, m.hull_verts.long()], 1),
            "hull_len": torch.stack([m.convex_perimeter, m.feret_min], 1)}


def _check_oracle(pm, columns=True):
    m = pm.measure()
    want = om.measure(oc.unpack_windows(pm.geom, pm.offsets, pm.bits))
    got = _exact(m)
    for f in om.FIELDS:
        assert torch.equal(got[f].cpu(), want[f]), f
    if columns:
        ref = om.columns(want, pm.geom.cpu())
        for k, v in m.columns().items():
            assert np.allclose(v.double().cpu().numpy(), ref[k], rtol=1e-12, atol=1e-12 if k == "orientation" else 0,
                               equal_nan=True), k
    return m


@pytest.mark.parametrize("poison", [None, 5])
def test_measure_equal_oracle(cuda_device, poison):
    items = _shapes(np.random.default_rng(1))
    pm = _pack(items, 200, 200, cuda_device, poison_seed=poison)
    m = _check_oracle(pm)
    assert int((m.hull_verts > 8).sum()) > 50 and int((m.euler < 1).sum()) > 10          # real hulls and holes
    _check_oracle(pm.select(torch.tensor([5, 3, 3, 0, 200, 41, 7])))
    _check_oracle(pm.select([]))
    other = _pack(items[:50], 200, 200, cuda_device, poison_seed=9)
    _check_oracle(PackedMasks.cat([pm, other], [(0, 0), (250, 40)], (300, 500)))


def test_measure_of_empty_sets(cuda_device):
    pm = _pack([(0, 0, np.zeros((0, 0), bool)), (3, 3, np.zeros((4, 4), bool))], 10, 10, cuda_device)
    m = _check_oracle(pm)
    assert m.area.tolist() == [0, 0] and bool(torch.isnan(m.centroid).all())
    assert len(_check_oracle(pm.select([]))) == 0


def test_measure_of_large_windows(cuda_device):
    """Windows beyond 64 px on a side: one CTA per mask."""
    rng = np.random.default_rng(2)
    yy, xx = np.mgrid[:1024, :1024]
    blob = np.hypot(yy - 512, xx - 512) < 500
    for c in rng.integers(40, 980, (60, 2)):
        blob[c[0] - 6:c[0] + 6, c[1] - 9:c[1] + 9] = False
    items = [(0, 0, blob), (10, 20, rng.random((300, 300)) < 0.5), (5, 5, rng.random((65, 3)) < 0.5),
             (5, 5, rng.random((2, 200)) < 0.5), (3, 3, np.ones((1, 1), bool)), (0, 0, rng.random((2, 5000)) < 0.3),
             (0, 0, rng.random((5000, 2)) < 0.3), (7, 9, np.hypot(yy[:700, :900] - 300, xx[:700, :900] - 400) < 290)]
    pm = _pack(items, 5100, 5100, cuda_device, poison_seed=4)
    m = _check_oracle(pm)
    assert int(m.hull_verts[0]) > 100 and int(m.hull_verts[-1]) > 100


def test_measure_window_side_limit(cuda_device):
    rng = np.random.default_rng(3)
    row = rng.random((1, 32768)) < 0.5
    m = _check_oracle(_pack([(0, 0, row), (1, 1, np.ones((2, 2), bool))], 2, 32770, cuda_device, poison_seed=1))
    assert int(m.area[0]) == int(row.sum())
    too = _pack([(0, 0, np.ones((1, 3), bool)), (0, 0, np.ones((1, 32769), bool))], 2, 32770, cuda_device)
    with pytest.raises(hdy.HdyError, match="32768"):
        too.measure()


def _long_chain_xl(w, h):
    """Left pixel extremes of up to h rows whose left hull chain takes as many distinct edge directions (a, b) as fit
    sum(b) <= h and x within [0, w - 1] on both of its sides: the longest chains the large path must hold."""
    vs = sorted(((a, b) for b in range(1, 200) for a in range(-200, 201) if math.gcd(abs(a), b) == 1),
                key=lambda v: (abs(v[0]) + 2 * v[1], v[1]))
    sb = sneg = spos = 0
    pick = []
    for a, b in vs:
        if sb + b > h or (a < 0 and sneg - a > w - 1) or (a > 0 and spos + a > w - 1):
            continue
        pick.append((a, b))
        sb, sneg, spos = sb + b, sneg + max(-a, 0), spos + max(a, 0)
    pick.sort(key=lambda v: Fraction(v[0], v[1]))
    ys, xs = np.cumsum([0] + [b for _, b in pick]), np.cumsum([sneg] + [a for a, _ in pick])
    cx = np.ceil(np.interp(np.arange(sb + 1), ys, xs) - 1e-9).astype(np.int64)   # the chain's x at each corner row
    return np.maximum(cx[:-1], cx[1:])          # every corner on or right of the chain, its vertices exactly on it


def _pack_rows(items, H, W, dev):
    """[(x0, y0, w, xl [h], xr [h])]: windows whose row y holds the pixels xl[y] .. xr[y] -> PackedMasks."""
    geom, offs, words = [], [0], []
    for x0, y0, w, xl, xr in items:
        wpr = (w + 31) // 32
        k = 32 * torch.arange(wpr, device=dev, dtype=torch.int64)
        lo = (torch.as_tensor(xl, device=dev)[:, None] - k).clamp(0, 32)
        hi = (torch.as_tensor(xr, device=dev)[:, None] + 1 - k).clamp(0, 32)
        v = ((1 << hi) - 1) - ((1 << lo) - 1)
        words.append((v - (v >= 2 ** 31).long() * 2 ** 32).to(torch.int32).reshape(-1))
        geom.append([x0, y0, w, len(xl)])
        offs.append(offs[-1] + wpr * len(xl))
    return PackedMasks(torch.tensor(geom, dtype=torch.int32, device=dev), torch.tensor(offs, dtype=torch.int64, device=dev),
                       torch.cat(words), H, W, torch.zeros(1, dtype=torch.int32, device=dev))


def test_measure_of_longest_hull_chains(cuda_device):
    """A 32 765-wide window of 32 762 rows whose left hull chain has 2 273 points, and its mirror image, whose right
    chain has them: more than a chain had room for when its bound counted the chain's x travel once."""
    w = 32765
    xl = _long_chain_xl(w, 32762)
    h = len(xl)
    sides = [(xl, np.full(h, w - 1)), (np.zeros(h, np.int64), w - 1 - xl)]
    pm = _pack_rows([(1, 2, w, a, b) for a, b in sides], 32770, 32770, cuda_device)
    m = pm.measure()
    r = np.arange(h, dtype=np.int64)
    for i, (a, b) in enumerate(sides):
        hull = om.hull_of_points(np.concatenate([a, a, b + 1, b + 1]), np.concatenate([r, r + 1, r, r + 1]))
        (area2, fmax2, nv), (perim, fmin) = om.hull_fields(hull)
        assert nv > 2273 and int(m.hull_verts[i]) == nv
        assert int(m.convex_area2[i]) == area2 and int(m.feret_max2[i]) == fmax2
        assert float(m.convex_perimeter[i]) == perim and float(m.feret_min[i]) == fmin
        n = b - a + 1
        sx = (a + b) * n // 2
        sxx = (b * (b + 1) * (2 * b + 1) - (a - 1) * a * (2 * a - 1)) // 6
        assert int(m.area[i]) == int(n.sum())
        assert m.bbox[i].tolist() == [1 + int(a.min()), 2, 2 + int(b.max()), 2 + h]
        assert m.moments[i].tolist() == [int(sx.sum()), int((r * n).sum()), int(sxx.sum()), int((r * r * n).sum()),
                                         int((r * sx).sum())]
        overlap = np.maximum(0, np.minimum(b[1:], b[:-1]) - np.maximum(a[1:], a[:-1]) + 1)
        assert float(m.perimeter[i]) == 2 * h + n[0] + n[-1] + int((n[1:] + n[:-1] - 2 * overlap).sum())
        assert int(m.euler[i]) == 1


def test_measure_of_packed_library_output(cuda_device):
    out, _ = synth.nuclei_match_case(3000, 3000, 1024, seed=3, device=cuda_device)
    pm = PackedMasks.from_dense(out['masks'])
    m = _check_oracle(pm)
    again = pm.measure()
    for f, t in _exact(m).items():
        assert torch.equal(t, _exact(again)[f])
    g = torch.Generator().manual_seed(7)
    bs, md = 2, 300
    protos = torch.randn((bs, 32, 80, 80), generator=g).to(cuda_device)
    coef = (torch.randn((bs, md, 32), generator=g) * 0.5).to(cuda_device)
    xy0 = torch.rand((bs, md, 2), generator=g) * 280
    boxes = torch.cat([xy0, xy0 + 6 + torch.rand((bs, md, 2), generator=g) * 60], 2).clamp(0, 320).to(cuda_device)
    counts = torch.tensor([md, md - 40], dtype=torch.int32, device=cuda_device)
    pp = hdy.process_mask_packed(protos, coef, boxes, counts, (320, 320), upsample=True)
    m = _check_oracle(pp)
    assert int((m.area > 0).sum()) > md


def _ring_lengths(c, K):
    """Per mask: the summed length of its contours() rings."""
    xy = c.xy.long()
    nxt = torch.arange(len(xy), device=xy.device) + 1
    nxt[c.ring_verts[1:] - 1] = c.ring_verts[:-1]
    seg = (xy[nxt] - xy).abs().sum(1)
    nv = c.ring_verts[1:] - c.ring_verts[:-1]
    ring_len = torch.zeros(len(nv), dtype=torch.int64, device=xy.device).index_add_(
        0, torch.repeat_interleave(torch.arange(len(nv), device=xy.device), nv), seg)
    nr = c.mask_rings[1:] - c.mask_rings[:-1]
    mask_of = torch.repeat_interleave(torch.arange(K, device=xy.device), nr)
    ext = torch.zeros(K, dtype=torch.int64, device=xy.device).index_add_(0, mask_of, (c.parent < 0).long())
    holes = torch.zeros(K, dtype=torch.int64, device=xy.device).index_add_(0, mask_of, (c.parent >= 0).long())
    return torch.zeros(K, dtype=torch.int64, device=xy.device).index_add_(0, mask_of, ring_len), ext - holes


def test_measure_at_slide_scale(cuda_device):
    """~10^6 nuclei of the synthetic slide field: identities on every mask, the oracle on 10^4 random rows."""
    pm = synth.slide_nuclei((0, 0, 18700, 18700), device=cuda_device)['masks']
    K = len(pm)
    assert K > 900_000
    m = pm.measure()
    assert torch.equal(m.area, pm.areas())
    c = pm.contours()
    length, euler = _ring_lengths(c, K)
    q = m.quads.long()
    assert torch.equal(m.perimeter, length.double())
    assert torch.equal(m.euler, euler)
    assert torch.equal(q[:, 0] + q[:, 2] + 2 * q[:, 3], _local_vertex_counts(pm))
    assert torch.equal(q[:, 0] + q[:, 2] + 2 * q[:, 3], c.ring_verts[c.mask_rings[1:]] - c.ring_verts[c.mask_rings[:-1]])
    w, h = pm.geom[:, 2].long(), pm.geom[:, 3].long()
    b = m.bbox.long()
    assert torch.equal(b[:, 2] - b[:, 0], w) and torch.equal(b[:, 3] - b[:, 1], h)          # tight windows
    a = m.area.long()
    assert bool(((2 * a <= m.convex_area2) & (m.convex_area2 <= 2 * w * h)).all())
    assert bool(((torch.maximum(w, h) ** 2 <= m.feret_max2) & (m.feret_max2 <= w * w + h * h)).all())
    assert bool((m.feret_min <= torch.minimum(w, h).double()).all())
    rows = torch.randperm(K, generator=torch.Generator().manual_seed(3))[:10_000].sort().values.to(cuda_device)
    sel = _check_oracle(pm.select(rows))
    for f, t in _exact(sel).items():
        assert torch.equal(t, _exact(m)[f][rows]), f
    again = pm.measure()
    for f, t in _exact(m).items():
        assert torch.equal(t, _exact(again)[f]), f


def test_measure_of_slide_result(cuda_device, tmp_path):
    dev = cuda_device
    size, tile, overlap, md, nm = (700, 900), 512, 64, 1200, 32
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=9 + nm)
    post = hdy.SlidePostprocessor(spec, size, (tile, tile), overlap, 0.25, 0.45, md, cap=2048, batch=4, device=dev)
    rois = post.rois
    prov = lambda a, b: synth.slide_tile_logits(rois[a:b], tile, 4, seed=9, first_tile=a, device=dev, pitch=30.0,
                                                extra=nm)
    protos = lambda a, b: synth.slide_tile_protos(b - a, tile, seed=9, first_tile=a, nm=nm, device=dev)
    res = post.run(prov, ordered=True, proto_provider=protos)
    kept = res['masks'].select(res['index'] - res['base'])
    assert len(kept) > 300
    m = _check_oracle(kept)
    c = kept.contours()
    path = str(tmp_path / "slide.geojson")
    n = hdy.save_geojson(path, res, c, measurements=m)
    feats = json.load(open(path))["features"]
    assert n == len(feats) == int((m.area > 0).sum())
    cols = {k: v.cpu() for k, v in m.columns().items()}
    index = res['index'].cpu().tolist()
    for f in feats[:50]:
        i = index.index(f["properties"]["index"])
        for k, v in f["properties"]["measurements"].items():
            want = cols[k][i].item()
            assert (v is None and not math.isfinite(want)) or v == want, k
    det = str(tmp_path / "slide.det")
    res_k = {k: v for k, v in res.items() if isinstance(v, torch.Tensor) and v.dim() >= 1 and v.shape[0] == len(kept)}
    hdy.save_detections(det, {**res_k, **m.columns()}, kept)
    back, masks, _ = hdy.load_detections(det)
    for k, v in m.columns().items():
        assert torch.equal(back[k], v.cpu()), k
    assert torch.equal(masks.geom, kept.geom.cpu())
