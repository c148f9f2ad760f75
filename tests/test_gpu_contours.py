"""GPU tests of PackedMasks.contours() (csrc/contours.cu): every array equal to oracle/contours.py on hand-made,
random, packed-by-the-library and slide-scale planes, both kernel paths (windows up to 64 x 64 one thread per mask,
larger ones one CTA per mask), and the area and local vertex-count identities on every mask at slide scale."""
import numpy as np
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import synth
from hd_yolo_b200.masks import PackedMasks
from oracle import contours as oc

pytestmark = pytest.mark.gpu

FIELDS = ('mask_rings', 'ring_verts', 'xy', 'parent')


def _pack(items, H, W, dev, poison_seed=None):
    """[(x0, y0, [h, w] bool)] -> PackedMasks with those windows; poison_seed: random padding bits."""
    rng = np.random.default_rng(poison_seed)
    geom, offs, words = [], [0], []
    for x0, y0, m in items:
        h, w = m.shape
        if m.size == 0:
            geom.append([x0, y0, 0, 0])
            offs.append(offs[-1])
            continue
        wpr = (w + 31) // 32
        win = np.zeros((h, wpr * 32), bool)
        win[:, :w] = m
        if poison_seed is not None:
            win[:, w:] = rng.random((h, wpr * 32 - w)) < 0.5
        words.append(np.packbits(win.reshape(h, wpr, 32), axis=2, bitorder='little').reshape(-1).view('<u4'))
        geom.append([x0, y0, w, h])
        offs.append(offs[-1] + wpr * h)
    bits = np.concatenate(words).view(np.int32) if words else np.zeros(0, np.int32)
    return PackedMasks(torch.tensor(geom, dtype=torch.int32, device=dev).reshape(-1, 4),
                       torch.tensor(offs, dtype=torch.int64, device=dev), torch.from_numpy(bits.copy()).to(dev), H, W,
                       torch.zeros(1, dtype=torch.int32, device=dev))


def _check_oracle(pm):
    got = pm.contours()
    want = oc.contours(oc.unpack_windows(pm.geom, pm.offsets, pm.bits))
    for f in FIELDS:
        assert torch.equal(getattr(got, f).cpu(), want[f]), f
    return got


def _shapes(rng):
    cb = (np.add.outer(np.arange(15), np.arange(13)) % 2).astype(bool)           # all saddles
    yy, xx = np.mgrid[:41, :41]
    r = np.hypot(yy - 20, xx - 20)
    target = (r < 19) & ~((r > 8) & (r < 14)) & ~(r < 3)                           # hole with an island inside
    frame = np.ones((9, 9), bool)
    frame[1:-1, 1:-1] = False
    frame[4, 4] = True
    items = [(0, 0, cb), (3, 2, target), (50, 60, frame), (7, 7, np.ones((1, 1), bool)),
             (0, 0, np.ones((17, 40), bool)), (10, 10, np.zeros((0, 0), bool)), (4, 4, np.zeros((6, 35), bool))]
    edge = rng.random((20, 33)) < 0.6
    edge[0] = edge[-1] = edge[:, 0] = edge[:, -1] = True                         # touches every window edge
    items.append((1, 1, edge))
    for w in (31, 32, 33, 63, 64, 65):
        for h in (1, 2, 64, 65):
            items.append((int(rng.integers(0, 50)), int(rng.integers(0, 50)), rng.random((h, w)) < rng.random()))
    for _ in range(300):
        h, w = (int(v) for v in rng.integers(1, 71, 2))
        items.append((int(rng.integers(0, 120)), int(rng.integers(0, 120)), rng.random((h, w)) < rng.random()))
    return items


@pytest.mark.parametrize("poison", [None, 5])
def test_contours_equal_oracle(cuda_device, poison):
    items = _shapes(np.random.default_rng(1))
    pm = _pack(items, 200, 200, cuda_device, poison_seed=poison)
    got = _check_oracle(pm)
    assert int((got.parent >= 0).sum()) > 100                                     # holes were traced
    rows = torch.tensor([5, 3, 3, 0, 200, 41, 7])
    _check_oracle(pm.select(rows))
    _check_oracle(pm.select([]))
    other = _pack(items[:50], 200, 200, cuda_device, poison_seed=9)
    _check_oracle(PackedMasks.cat([pm, other], [(0, 0), (250, 40)], (300, 500)))


def test_contours_of_empty_sets(cuda_device):
    pm = _pack([(0, 0, np.zeros((0, 0), bool)), (3, 3, np.zeros((4, 4), bool))], 10, 10, cuda_device)
    got = _check_oracle(pm)
    assert got.xy.shape == (0, 2) and got.parent.shape == (0,) and got.ring_verts.tolist() == [0]
    got = _check_oracle(pm.select([]))
    assert got.mask_rings.tolist() == [0]


def test_contours_of_large_windows(cuda_device):
    """Windows beyond 64 px on a side: one CTA per mask."""
    rng = np.random.default_rng(2)
    yy, xx = np.mgrid[:1024, :1024]
    blob = np.hypot(yy - 512, xx - 512) < 500
    for c in rng.integers(40, 980, (60, 2)):
        blob[c[0] - 6:c[0] + 6, c[1] - 9:c[1] + 9] = False
        blob[c[0] - 1:c[0] + 1, c[1] - 2:c[1] + 3] = True                          # islands inside some holes
    items = [(0, 0, blob), (10, 20, rng.random((300, 300)) < 0.5), (5, 5, rng.random((65, 3)) < 0.5),
             (5, 5, rng.random((2, 200)) < 0.5), (3, 3, np.ones((1, 1), bool))]
    pm = _pack(items, 1100, 1100, cuda_device, poison_seed=4)
    got = _check_oracle(pm)
    assert int((got.parent[got.mask_rings[0]:got.mask_rings[1]] >= 0).sum()) >= 40


def test_contours_of_packed_library_output(cuda_device):
    out, _ = synth.nuclei_match_case(3000, 3000, 1024, seed=3, device=cuda_device)
    pm = PackedMasks.from_dense(out['masks'])
    got = _check_oracle(pm)
    again = pm.contours()                                                         # run to run: identical
    for f in FIELDS:
        assert torch.equal(getattr(got, f), getattr(again, f))
    # process_mask's box windows (not tight), upsampled to the image
    g = torch.Generator().manual_seed(7)
    bs, md = 2, 300
    protos = torch.randn((bs, 32, 80, 80), generator=g).to(cuda_device)
    coef = (torch.randn((bs, md, 32), generator=g) * 0.5).to(cuda_device)
    xy0 = torch.rand((bs, md, 2), generator=g) * 280
    boxes = torch.cat([xy0, xy0 + 6 + torch.rand((bs, md, 2), generator=g) * 60], 2).clamp(0, 320).to(cuda_device)
    counts = torch.tensor([md, md - 40], dtype=torch.int32, device=cuda_device)
    pp = hdy.process_mask_packed(protos, coef, boxes, counts, (320, 320), upsample=True)
    got = _check_oracle(pp)
    assert int(got.mask_rings[-1]) > md


def _rows_u64(pm):
    """Each row of each mask as one int64 of its w (<= 62) pixels -> (values, mask of each row, row in its mask,
    rows per mask)."""
    g = pm.geom.long()
    w, h = g[:, 2].clamp_min(0), g[:, 3].clamp_min(0)
    live = (w > 0) & (h > 0)
    h = torch.where(live, h, torch.zeros_like(h))
    assert int(w.max()) <= 62
    wpr = (w + 31) // 32
    mask_of = torch.repeat_interleave(torch.arange(len(pm), device=g.device), h)
    first = torch.cumsum(h, 0) - h
    r = torch.arange(int(h.sum()), device=g.device) - first[mask_of]
    word = pm.offsets[:-1][mask_of] + r * wpr[mask_of]
    bits = pm.bits.long() & 0xffffffff
    lo = bits[word]
    hi = torch.where(wpr[mask_of] == 2, bits[(word + 1).clamp_max(bits.numel() - 1)], torch.zeros_like(lo))
    v = (lo | (hi << 32)) & ((torch.ones_like(lo) << w[mask_of]) - 1)
    return v, mask_of, r, h


def _popcount(x):
    x = x - ((x >> 1) & 0x5555555555555555)
    x = (x & 0x3333333333333333) + ((x >> 2) & 0x3333333333333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F0F0F0F0F
    return x.contiguous().view(torch.uint8).view(-1, 8).sum(1, dtype=torch.int64)


def _local_vertex_counts(pm):
    """Per mask: corners with an odd number of set pixels among their four, plus two per saddle (row words on the
    device, independent of the kernels)."""
    v, mask_of, r, h = _rows_u64(pm)
    above = torch.where(r > 0, torch.roll(v, 1), torch.zeros_like(v))

    def corners(A, B):
        a, b = A ^ (A << 1), B ^ (B << 1)
        return _popcount(a ^ b) + 2 * _popcount(a & b & (A ^ B))

    last = r == h[mask_of] - 1
    per_row = corners(above, v) + torch.where(last, corners(v, torch.zeros_like(v)), torch.zeros_like(v))
    out = torch.zeros(len(pm), dtype=torch.int64, device=v.device)
    return out.index_add_(0, mask_of, per_row)


def _check_identities(pm, c):
    """Signed ring areas add up to the mask's pixel count; vertex counts are the local count."""
    K = len(pm)
    nv = c.ring_verts[1:] - c.ring_verts[:-1]
    ring_of = torch.repeat_interleave(torch.arange(len(nv), device=nv.device), nv)
    xy = c.xy.long()
    nxt = torch.arange(len(xy), device=xy.device) + 1
    ends = c.ring_verts[1:] - 1
    nxt[ends] = c.ring_verts[:-1]
    cross = xy[:, 0] * xy[nxt, 1] - xy[nxt, 0] * xy[:, 1]
    ring_area2 = torch.zeros(len(nv), dtype=torch.int64, device=xy.device).index_add_(0, ring_of, cross)
    nr = c.mask_rings[1:] - c.mask_rings[:-1]
    mask_of = torch.repeat_interleave(torch.arange(K, device=nr.device), nr)
    area2 = torch.zeros(K, dtype=torch.int64, device=xy.device).index_add_(0, mask_of, ring_area2)
    assert torch.equal(area2, 2 * pm.areas().long())
    assert bool(((ring_area2 > 0) == (c.parent < 0)).all())
    verts = c.ring_verts[c.mask_rings[1:]] - c.ring_verts[c.mask_rings[:-1]]
    assert torch.equal(verts, _local_vertex_counts(pm))


def test_contours_at_slide_scale(cuda_device):
    """~10^6 nuclei of the synthetic slide field: identities on every mask, the oracle on 10^4 random rows."""
    pm = synth.slide_nuclei((0, 0, 18700, 18700), device=cuda_device)['masks']
    assert len(pm) > 900_000
    c = pm.contours()
    _check_identities(pm, c)
    rows = torch.randperm(len(pm), generator=torch.Generator().manual_seed(3))[:10_000].sort().values
    sel = _check_oracle(pm.select(rows.to(cuda_device)))
    # the rows of the whole call are the rows of the selection
    for i in (0, 17, 9999):
        r = int(rows[i])
        a, b = int(c.mask_rings[r]), int(c.mask_rings[r + 1])
        sa, sb = int(sel.mask_rings[i]), int(sel.mask_rings[i + 1])
        assert torch.equal(c.xy[c.ring_verts[a]:c.ring_verts[b]], sel.xy[sel.ring_verts[sa]:sel.ring_verts[sb]])
    again = pm.contours()
    for f in FIELDS:
        assert torch.equal(getattr(c, f), getattr(again, f))


def test_contours_of_slide_result(cuda_device, tmp_path):
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
    c = _check_oracle(kept)
    if int(kept.geom[:, 2].max()) <= 62:
        _check_identities(kept, c)
    n = hdy.save_geojson(str(tmp_path / "slide.geojson"), res, c)
    assert n == int(((c.mask_rings[1:] - c.mask_rings[:-1]) > 0).sum())
