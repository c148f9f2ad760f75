"""GPU tests of matching by mask IoU (APMeter.add(..., iou_type='masks')) over bit-packed masks: the dense -> packed
conversion with tight windows, areas that ignore padding bits, the bit alignment of the pair counts, and parity of
match_predictions / APMeter with oracle/mask_match.py's mask_iou at full sizes (the oracle runs on the device there: its
fp32 overlap product is exact in any summation order)."""
import pytest
import torch
import torchvision

import hd_yolo_b200 as hdy
from hd_yolo_b200 import synth
from hd_yolo_b200.masks import PackedMasks
from oracle import mask_match

pytestmark = pytest.mark.gpu


def _set(x):
    return (x > 0.5) if x.dtype.is_floating_point else (x != 0)


def _assert_same(got, ref):
    s, l, p, t, i = ref
    assert torch.equal(got['scores'].cpu(), s.cpu()) and torch.equal(got['labels'].cpu(), l.cpu())
    assert torch.equal(got['ious'].cpu(), i.cpu())
    assert torch.equal(got['pred_idx'].cpu(), p.cpu()) and torch.equal(got['true_idx'].cpu(), t.cpu())


def _same_result(a, b):
    return all(torch.equal(a[f], b[f]) for f in ('order', 'scores', 'labels', 'pred_idx', 'true_idx', 'ious'))


def _shapes_case(H, W, dev):
    """Masks that exercise the window bounds: empty, single pixels, every canvas edge, widths 1/31/32/33/64/65,
    thresholds exactly at 0.5, random noise."""
    g = torch.Generator().manual_seed(H * 1000 + W)
    vals = []

    def mask(ys, xs, v=1.0):
        m = torch.zeros((H, W))
        m[ys, xs] = v
        vals.append(m)
    mask(slice(0, 0), slice(0, 0))                    # empty
    mask(0, 0)                                        # single pixel, top-left corner
    mask(H - 1, W - 1, 0.75)                          # single pixel, bottom-right corner
    mask(slice(3, 9), 0)                              # left edge
    mask(5, slice(W - 3, W))                          # right edge
    mask(0, slice(7, 20))                             # top edge
    mask(H - 1, slice(2, 5))                          # bottom edge
    mask(slice(0, H), slice(0, W), 0.5)               # exactly 0.5 is not set: empty
    for w in (1, 31, 32, 33, 64, 65):
        if w <= W - 2:
            mask(slice(2, 2 + min(H - 2, 9)), slice(1, 1 + w))
            mask(slice(1, 4), slice(W - w, W), torch.rand((3, w), generator=g) + 0.3)
    for _ in range(6):                                # noise in a random rectangle
        y0, x0 = int(torch.randint(0, H - 1, (1,), generator=g)), int(torch.randint(0, W - 1, (1,), generator=g))
        mask(slice(y0, H), slice(x0, W), torch.rand((H - y0, W - x0), generator=g))
    return torch.stack(vals).to(dev)


@pytest.mark.parametrize("H,W", [(70, 131), (96, 160), (33, 65)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.uint8, torch.bool])
def test_from_dense_round_trip(cuda_device, H, W, dtype):
    x = _shapes_case(H, W, cuda_device)
    if dtype == torch.uint8:
        x = (x * 3).to(torch.uint8)            # 0 < v < 1/3 rounds to 0: set iff nonzero
    elif dtype == torch.bool:
        x = x > 0.5
    else:
        x = x.to(dtype)
    ref = _set(x)
    pm = PackedMasks.from_dense(x)
    pm.check()
    assert torch.equal(pm.to_dense(), ref.to(torch.uint8))
    assert torch.equal(PackedMasks.from_dense(x[:, None]).to_dense(), ref.to(torch.uint8))   # [K, 1, H, W]
    geom = pm.geom.cpu()
    nonempty = ref.flatten(1).any(1).cpu()
    b = torchvision.ops.masks_to_boxes(ref[nonempty.to(ref.device)]).cpu().to(torch.int32)
    want = torch.stack([b[:, 0], b[:, 1], b[:, 2] - b[:, 0] + 1, b[:, 3] - b[:, 1] + 1], 1)
    assert torch.equal(geom[nonempty], want)
    assert int(geom[~nonempty].abs().sum()) == 0                  # empty masks: w = h = 0
    assert torch.equal(pm.areas().cpu(), ref.flatten(1).sum(1).to(torch.int32).cpu())
    # padding bits beyond w in the last word of every row are zero
    wpr = (geom[:, 2] + 31) // 32
    off = pm.offsets.cpu()
    assert torch.equal(off[1:] - off[:-1], (wpr * geom[:, 3]).to(torch.int64))
    bits = pm.bits.cpu()
    for i in range(len(pm)):
        w, h = int(geom[i, 2]), int(geom[i, 3])
        if h and w % 32:
            last = bits[int(off[i]) + torch.arange(h) * int(wpr[i]) + int(wpr[i]) - 1].to(torch.int64) & 0xffffffff
            assert bool((last >> (w % 32) == 0).all()), i


def _poison_padding(pm: PackedMasks) -> PackedMasks:
    """The same masks with every padding bit (beyond w in each row's last word) set."""
    geom, off = pm.geom.cpu(), pm.offsets.cpu()
    bits = pm.bits.cpu().to(torch.int64) & 0xffffffff
    for i in range(len(pm)):
        w, h = int(geom[i, 2]), int(geom[i, 3])
        if h and w % 32:
            wpr = (w + 31) // 32
            idx = int(off[i]) + torch.arange(h) * wpr + wpr - 1
            bits[idx] |= (0xffffffff << (w % 32)) & 0xffffffff
    bits = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32)
    return PackedMasks(pm.geom, pm.offsets, bits.to(pm.bits.device), pm.H, pm.W, pm.status)


def test_areas_and_matches_ignore_padding_bits(cuda_device):
    out, tgt = synth.nuclei_match_case(300, 260, 256, seed=7, device=cuda_device)
    pp, pg = PackedMasks.from_dense(out['masks']), PackedMasks.from_dense(tgt['masks'])
    qp, qg = _poison_padding(pp), _poison_padding(pg)
    assert not torch.equal(qp.bits, pp.bits)
    assert torch.equal(qp.areas(), pp.areas()) and torch.equal(qg.areas(), pg.areas())
    assert torch.equal(pp.areas(), out['masks'].flatten(1).sum(1).to(torch.int32))
    clean = hdy.match_predictions({**out, 'masks': pp}, {**tgt, 'masks': pg}, 0.5, iou_type='masks')
    dirty = hdy.match_predictions({**out, 'masks': qp}, {**tgt, 'masks': qg}, 0.5, iou_type='masks')
    assert len(clean['ious']) > 100 and _same_result(clean, dirty)


def test_bit_alignment_every_shift(cuda_device):
    """Prediction windows start at every x offset 0..31 from the ground truth's, and several words left and right of
    it, on different rows: the funnel-shifted pair counts equal the oracle's."""
    H, W = 64, 512
    g = torch.Generator().manual_seed(3)
    gts = torch.zeros((3, H, W))
    gts[0, 10:30, 150:220] = torch.rand((20, 70), generator=g)   # 70 wide: 3 words
    gts[1, 20:40, 200:205] = torch.rand((20, 5), generator=g)    # 5 wide: 1 word
    gts[2, 5:60, 100:400] = torch.rand((55, 300), generator=g)   # 300 wide: 10 words
    preds = []
    for dx in list(range(-40, 41)) + [-97, -64, -33, 63, 64, 65, 96, 130]:
        for dy in (0, 3):
            m = torch.zeros((H, W))
            m[12 + dy:28 + dy, 150 + dx:230 + dx] = torch.rand((16, 80), generator=g)
            preds.append(m)
    preds = torch.stack(preds)
    k = len(preds)
    boxes = torch.zeros((k, 4))
    out = {'boxes': boxes, 'scores': torch.rand(k, generator=g), 'labels': torch.ones(k, dtype=torch.int64),
           'masks': preds}
    tgt = {'boxes': torch.zeros((3, 4)), 'labels': torch.ones(3, dtype=torch.int64), 'masks': gts}
    iou_min = 1e-6                                     # every pair with one common pixel matches
    got = hdy.match_predictions({a: b.to(cuda_device) for a, b in out.items()},
                                {a: b.to(cuda_device) for a, b in tgt.items()}, iou_min, iou_type='masks')
    ref = mask_match.apmeter_match(out, tgt, iou_min)
    assert len(ref[4]) > k
    _assert_same(got, ref)


@pytest.mark.parametrize("k,g,seed", [(1500, 1400, 1), (40, 4500, 2), (3000, 3000, 3)])
def test_match_predictions_masks_parity(cuda_device, k, g, seed):
    out, tgt = synth.nuclei_match_case(k, g, 1024, seed=seed, device=cuda_device)
    ref = mask_match.apmeter_match(out, tgt, 0.5)           # on the device: exact integer products
    assert len(ref[4]) > min(k, g) // 2
    assert len(torch.unique(out['scores'])) < k                 # score ties
    dense = hdy.match_predictions(out, tgt, 0.5, iou_type='masks')
    _assert_same(dense, ref)
    pp, pg = PackedMasks.from_dense(out['masks']), PackedMasks.from_dense(tgt['masks'])
    packed = hdy.match_predictions({**out, 'masks': pp}, {**tgt, 'masks': pg}, 0.5, iou_type='masks')
    mixed = hdy.match_predictions({**out, 'masks': pp}, {**tgt, 'masks': tgt['masks'].to(torch.uint8)[:, None]}, 0.5,
                                  iou_type='masks')
    mixed2 = hdy.match_predictions({**out, 'masks': out['masks'].float()}, {**tgt, 'masks': pg}, 0.5, iou_type='masks')
    assert _same_result(dense, packed) and _same_result(dense, mixed) and _same_result(dense, mixed2)


def test_match_predictions_masks_ties_and_capacity(cuda_device):
    # every prediction is the same mask as every ground truth: k*g pairs of iou 1, more than the capacity
    m = synth.ellipse_masks(torch.tensor([[40.0, 30.0]]), torch.tensor([[9.0, 7.0]]), 64, 96)
    k, n_gt = 70, 60
    out = {'boxes': torch.zeros((k, 4)), 'scores': torch.linspace(0.9, 0.1, k), 'labels': torch.ones(k, dtype=torch.int64),
           'masks': m.repeat(k, 1, 1)}
    tgt = {'boxes': torch.zeros((n_gt, 4)), 'labels': torch.ones(n_gt, dtype=torch.int64), 'masks': m.repeat(n_gt, 1, 1)}
    got = hdy.match_predictions({a: b.to(cuda_device) for a, b in out.items()},
                                {a: b.to(cuda_device) for a, b in tgt.items()}, 0.5, cap=64, iou_type='masks')
    assert len(got['ious']) == k * n_gt and bool((got['ious'] == 1.0).all())
    idx = torch.arange(k * n_gt)
    assert torch.equal(got['pred_idx'].cpu(), idx // n_gt) and torch.equal(got['true_idx'].cpu(), idx % n_gt)


def test_match_predictions_masks_edge_cases(cuda_device):
    dev = cuda_device
    out, tgt = synth.nuclei_match_case(60, 50, 128, seed=5, device=dev)
    out['masks'][::7] = False                          # empty predictions
    tgt['masks'][::5] = False                          # empty ground truth: empty x empty is 0/0 = NaN, never a match
    got = hdy.match_predictions(out, tgt, 0.5, iou_type='masks')
    ref = mask_match.apmeter_match(out, tgt, 0.5)
    assert bool(torch.isnan(mask_match.mask_iou(out['masks'][:1], tgt['masks'][:1])).all())
    _assert_same(got, ref)
    assert not bool(torch.isin(got['true_idx'], torch.arange(0, 50, 5, device=dev)).any())
    # windows without a set pixel (producers other than from_dense leave such windows): no pair matches
    def zeroed(m):
        pm = PackedMasks.from_dense(m)
        return PackedMasks(pm.geom, pm.offsets, torch.zeros_like(pm.bits), pm.H, pm.W, pm.status)
    none = hdy.match_predictions({**out, 'masks': zeroed(out['masks'])}, {**tgt, 'masks': zeroed(tgt['masks'])}, 0.5,
                                 iou_type='masks')
    assert len(none['ious']) == 0 and len(none['scores']) == 60
    # k = 0, g = 0
    k0 = hdy.match_predictions({a: v[:0] for a, v in out.items()}, tgt, 0.5, iou_type='masks')
    assert len(k0['order']) == 0 and len(k0['ious']) == 0
    g0 = hdy.match_predictions(out, {a: v[:0] for a, v in tgt.items()}, 0.5, iou_type='masks')
    assert len(g0['ious']) == 0 and torch.equal(g0['scores'].cpu(), ref[0].cpu())
    # iou_min <= 0, canvas mismatch, row mismatch, missing masks
    for bad in (0.0, -0.5, float('nan')):
        with pytest.raises(hdy.HdyError):
            hdy.match_predictions(out, tgt, bad, iou_type='masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, {**tgt, 'masks': tgt['masks'][:, :, :127]}, 0.5, iou_type='masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, {**tgt, 'masks': PackedMasks.from_dense(tgt['masks'][:, :100])}, 0.5,
                              iou_type='masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, {**tgt, 'masks': tgt['masks'][:10]}, 0.5, iou_type='masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, {a: v for a, v in tgt.items() if a != 'masks'}, 0.5, iou_type='masks')


def test_apmeter_add_masks_matches_oracle(cuda_device):
    dev = cuda_device
    cases = [synth.nuclei_match_case(k, g, 192, seed=20 + i, device=dev)
             for i, (k, g) in enumerate([(80, 70), (0, 30), (40, 0), (120, 90)])]
    meter, oracle = hdy.APMeter(), mask_match.APMeterState()
    box_meter, box_oracle = hdy.APMeter(), hdy.APMeter()
    for i, (out, tgt) in enumerate(cases):
        pm = PackedMasks.from_dense(out['masks']) if i % 2 else out['masks']    # dense and packed inputs
        meter.add({**out, 'masks': pm}, tgt, iou_type='masks')
        oracle.add({a: v.cpu() for a, v in out.items()}, {a: v.cpu() for a, v in tgt.items()}, 0.5, iou_type='masks')
        strip = lambda d: {a: v for a, v in d.items() if a != 'masks'}
        box_meter.add(strip(out), strip(tgt), iou_type='masks')   # no masks: box IoU, as the reference does
        box_oracle.add(strip(out), strip(tgt))
    assert meter.n_match > 100
    assert [meter.n_pred, meter.n_true, meter.n_match] == [oracle.n_pred, oracle.n_true, oracle.n_match]
    for f in ("scores", "y_pred", "y_true", "ious", "m_pred", "m_true"):
        assert torch.equal(getattr(meter, f), getattr(oracle, f)), f
        assert torch.equal(getattr(box_meter, f), getattr(box_oracle, f)), f
    assert not torch.equal(meter.ious, box_meter.ious)


def test_slide_form_packed_masks(cuda_device):
    """process_mask_packed's planes (box windows, slots past a tile's count empty) match exactly like their own
    to_dense()."""
    dev = cuda_device
    g = torch.Generator().manual_seed(9)
    bs, md, ih, iw = 2, 150, 320, 320
    protos = torch.randn((bs, 32, 80, 80), generator=g)
    coef = torch.randn((bs, md, 32), generator=g) * 0.5
    c = torch.rand((bs, md, 2), generator=g) * ih
    r = 6 + 12 * torch.rand((bs, md, 2), generator=g)
    boxes = torch.cat([c - r, c + r], 2)
    counts = torch.tensor([md - 20, md - 45], dtype=torch.int32, device=dev)
    pm = hdy.process_mask_packed(protos.to(dev), coef.to(dev), boxes.to(dev), counts, (ih, iw), upsample=True)
    pm.check()
    dense = pm.to_dense()
    k = bs * md
    assert int((pm.geom[:, 2] * pm.geom[:, 3] == 0).sum()) >= 65
    gt_masks = torch.roll(dense[::2], shifts=(1, 2), dims=(1, 2))
    n_gt = gt_masks.shape[0]
    out = {'boxes': boxes.view(k, 4).to(dev), 'scores': torch.rand(k, generator=g).to(dev),
           'labels': torch.ones(k, dtype=torch.int64, device=dev)}
    tgt = {'boxes': torch.zeros((n_gt, 4), device=dev), 'labels': torch.ones(n_gt, dtype=torch.int64, device=dev),
           'masks': gt_masks}
    a = hdy.match_predictions({**out, 'masks': pm}, tgt, 0.5, iou_type='masks')
    b = hdy.match_predictions({**out, 'masks': dense}, tgt, 0.5, iou_type='masks')
    assert len(a['ious']) >= 40 and _same_result(a, b)
    _assert_same(a, mask_match.apmeter_match({**out, 'masks': dense}, tgt, 0.5))
