"""GPU tests of binned matching (match_predictions(..., binned=True), APMeter.add(..., binned=True)): bit-identical to
the all-pairs path wherever that one runs, equal to oracle/sparse_match.py beyond 2^32 (prediction, ground truth)
pairs, deterministic from run to run, and end to end on a slide result's kept masks."""
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import synth
from hd_yolo_b200.masks import PackedMasks
from oracle import sparse_match

pytestmark = pytest.mark.gpu

FIELDS = ('order', 'scores', 'labels', 'pred_idx', 'true_idx', 'ious')


def _assert_equal(a, b):
    for f in FIELDS:
        assert torch.equal(a[f], b[f]), f


def _assert_oracle(got, ref):
    s, l, p, t, i = ref
    assert torch.equal(got['scores'].cpu(), s) and torch.equal(got['labels'].cpu(), l)
    assert torch.equal(got['pred_idx'].cpu(), p) and torch.equal(got['true_idx'].cpu(), t)
    assert torch.equal(got['ious'].cpu(), i)


def _both(out, tgt, iou_min, iou_type):
    a = hdy.match_predictions(out, tgt, iou_min, iou_type=iou_type)
    b = hdy.match_predictions(out, tgt, iou_min, iou_type=iou_type, binned=True)
    _assert_equal(b, a)
    return b


@pytest.mark.parametrize("iou_type", ['boxes', 'masks'])
@pytest.mark.parametrize("k,g,seed", [(1500, 1400, 1), (40, 4500, 2), (3000, 3000, 3)])
def test_binned_equals_all_pairs(cuda_device, k, g, seed, iou_type):
    out, tgt = synth.nuclei_match_case(k, g, 1024, seed=seed, device=cuda_device)
    for iou_min in (0.5, 0.95, 1e-6):
        got = _both(out, tgt, iou_min, iou_type)
        if iou_min == 0.5:
            assert len(got['ious']) > min(k, g) // 2


def _edge_boxes(dev):
    """Lattice boxes (shared edges, corners on cell boundaries), duplicates, a box over the whole canvas, and boxes
    that match nothing: zero area, NaN, inf, negative extent, off the canvas."""
    g = torch.Generator().manual_seed(11)
    x = torch.randint(0, 60, (400, 2), generator=g).float() * 16
    s = torch.randint(1, 4, (400, 2), generator=g).float() * 16
    lattice = torch.cat([x, x + s], 1)
    odd = torch.tensor([[0., 0., 1024., 1024.], [100., 100., 100., 140.], [50., 50., 80., 50.],
                        [float('nan'), 0., 10., 10.], [0., float('nan'), 10., 10.], [0., 0., float('inf'), 10.],
                        [float('-inf'), 0., 10., 10.], [float('inf'), float('inf'), float('inf'), float('inf')],
                        [300., 300., 280., 320.], [-500., -500., -400., -400.], [2000., 2000., 2100., 2060.],
                        [-50., 1000., 40., 1100.]])
    huge = torch.tensor([[1e30, 1e30, 3e38, 3e38], [-3e38, -3e38, 3e38, 3e38]])   # areas overflow to inf
    preds = torch.cat([lattice, lattice[:100] + 4, odd, odd, huge])
    gts = torch.cat([lattice[50:350], lattice[60:90], odd, lattice[::7] + 8])     # duplicates: lattice[60:90]
    return preds.to(dev), gts.to(dev), huge.to(dev)


@pytest.mark.parametrize("huge_gt", [False, True])
def test_binned_boxes_edge_cases(cuda_device, huge_gt):
    """huge_gt: the overflowing boxes on the ground-truth side too, so the grid spans the whole fp32 range."""
    pb, gb, huge = _edge_boxes(cuda_device)
    if huge_gt:
        gb = torch.cat([gb, huge])
    k, n = len(pb), len(gb)
    gen = torch.Generator().manual_seed(5)
    out = {'boxes': pb, 'scores': ((torch.rand(k, generator=gen) * 8).round() / 8).to(cuda_device),
           'labels': torch.ones(k, dtype=torch.int64, device=cuda_device)}
    tgt = {'boxes': gb, 'labels': torch.ones(n, dtype=torch.int64, device=cuda_device)}
    for iou_min in (0.5, 0.95, 1e-6, 1.0):
        got = _both(out, tgt, iou_min, 'boxes')
        if iou_min == 1e-6:
            assert len(got['ious']) > 1000 and len(torch.unique(got['ious'])) < len(got['ious'])   # IoU ties
            _assert_oracle(got, sparse_match.apmeter_match_sparse(out, tgt, iou_min))
    # empty sides, and ground truth of which nothing can overlap anything
    _both(out, {a: v[:0] for a, v in tgt.items()}, 0.5, 'boxes')
    _both({a: v[:0] for a, v in out.items()}, tgt, 0.5, 'boxes')
    bad = {'boxes': torch.tensor([[5., 5., 5., 9.], [float('nan')] * 4], device=cuda_device),
           'labels': torch.ones(2, dtype=torch.int64, device=cuda_device)}
    assert len(_both(out, bad, 1e-6, 'boxes')['ious']) == 0
    for iou_min in (0.0, -0.5, float('nan'), 1e-50):
        with pytest.raises(hdy.HdyError):
            hdy.match_predictions(out, tgt, iou_min, binned=True)


def test_binned_masks_edge_cases(cuda_device):
    dev = cuda_device
    out, tgt = synth.nuclei_match_case(300, 260, 256, seed=8, device=dev)
    out['masks'][::9] = False                                   # empty predictions
    tgt['masks'][::7] = False                                   # empty ground truth
    tgt['masks'][1] = True                                      # one mask over the whole canvas
    out['masks'][2] = True
    tgt['masks'][10:20] = tgt['masks'][20:30]                   # duplicates: IoU ties
    for iou_min in (0.5, 0.95, 1e-6):
        got = _both(out, tgt, iou_min, 'masks')
    assert len(got['ious']) > 300
    pp, pg = PackedMasks.from_dense(out['masks']), PackedMasks.from_dense(tgt['masks'])
    _assert_equal(hdy.match_predictions({**out, 'masks': pp}, {**tgt, 'masks': pg}, 1e-6, iou_type='masks',
                                        binned=True), got)
    _assert_oracle(got, sparse_match.apmeter_match_sparse({**out, 'masks': pp}, {**tgt, 'masks': pg}, 1e-6, 'masks'))
    none = {**tgt, 'masks': torch.zeros_like(tgt['masks'])}
    assert len(_both(out, none, 0.5, 'masks')['ious']) == 0
    _both(out, {a: v[:0] for a, v in tgt.items()}, 0.5, 'masks')
    _both({a: v[:0] for a, v in out.items()}, tgt, 0.5, 'masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, {**tgt, 'masks': tgt['masks'][:, :, :200]}, 0.5, iou_type='masks', binned=True)
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, tgt, 0.0, iou_type='masks', binned=True)


def _large_case(dev):
    """~90 k predictions against ~80 k ground truth on a 16 384^2 canvas: P * G ~ 7e9 > 2^32."""
    region = (0, 0, 16384, 16384)
    gt = synth.slide_nuclei(region, pitch=58.0, device=dev)
    near = synth.slide_nuclei(region, pitch=58.0, jitter=3.0, seed=1, device=dev)
    extra = synth.slide_nuclei(region, pitch=160.0, jitter=5.0, seed=2, device=dev)
    out = {'boxes': torch.cat([near['boxes'], extra['boxes']]),
           'scores': (torch.cat([near['scores'], extra['scores'] * 0.9]) * 512).round() / 512,
           'labels': torch.cat([near['labels'], extra['labels']]),
           'masks': PackedMasks.cat([near['masks'], extra['masks']], [(0, 0), (0, 0)], (16384, 16384))}
    return out, gt


def test_binned_beyond_32_bit_pair_index(cuda_device):
    out, gt = _large_case(cuda_device)
    k, g = len(out['boxes']), len(gt['boxes'])
    assert k * g >= 2 ** 32 and k > 85000 and g > 75000
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, gt, 0.5)
    for iou_type in ('boxes', 'masks'):
        got = hdy.match_predictions(out, gt, 0.5, iou_type=iou_type, binned=True)
        assert len(got['ious']) > g // 2
        _assert_oracle(got, sparse_match.apmeter_match_sparse(out, gt, 0.5, iou_type))
        again = hdy.match_predictions(out, gt, 0.5, iou_type=iou_type, binned=True)       # run to run
        _assert_equal(again, got)


def test_apmeter_binned_equals_all_pairs(cuda_device):
    cases = [synth.nuclei_match_case(k, g, 320, seed=40 + i, device=cuda_device)
             for i, (k, g) in enumerate([(200, 180), (0, 30), (40, 0), (350, 300)])]
    for iou_type in ('boxes', 'masks'):
        a, b = hdy.APMeter(), hdy.APMeter()
        for out, tgt in cases:
            a.add(out, tgt, iou_type=iou_type)
            b.add(out, tgt, iou_type=iou_type, binned=True)
        assert a.n_match > 100
        assert [a.n_pred, a.n_true, a.n_match] == [b.n_pred, b.n_true, b.n_match]
        for f in ("scores", "y_pred", "y_true", "ious", "m_pred", "m_true"):
            assert torch.equal(getattr(a, f), getattr(b, f)), f


def test_slide_result_against_field_ground_truth(cuda_device):
    """A slide result's kept rows (select) matched against the synthetic field's ground truth: equal to the sparse
    oracle, and to the all-pairs path (small enough to run here)."""
    dev = cuda_device
    size, tile, overlap, md, nm = (700, 900), 512, 64, 1200, 32
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=9 + nm)
    post = hdy.SlidePostprocessor(spec, size, (tile, tile), overlap, 0.25, 0.45, md, cap=2048, batch=4, device=dev)
    rois = post.rois
    prov = lambda a, b: synth.slide_tile_logits(rois[a:b], tile, 4, seed=9, first_tile=a, device=dev, pitch=30.0,
                                                extra=nm)
    protos = lambda a, b: synth.slide_tile_protos(b - a, tile, seed=9, first_tile=a, nm=nm, device=dev)
    res = post.run(prov, ordered=True, proto_provider=protos)
    res['masks'].check()
    kept = res['masks'].select(res['index'] - res['base'])
    assert len(kept) == len(res['boxes']) > 300
    out = {'boxes': res['boxes'], 'scores': res['scores'], 'labels': res['labels'], 'masks': kept}
    gt = synth.slide_nuclei((0, 0, size[1], size[0]), canvas=(kept.H, kept.W), pitch=30.0, device=dev)
    for iou_type, iou_min in (('boxes', 0.5), ('masks', 0.5), ('masks', 0.1)):
        got = hdy.match_predictions(out, gt, iou_min, iou_type=iou_type, binned=True)
        assert len(got['ious']) > (50 if iou_type == 'boxes' else 0)
        _assert_oracle(got, sparse_match.apmeter_match_sparse(out, gt, iou_min, iou_type))
        _assert_equal(got, hdy.match_predictions(out, gt, iou_min, iou_type=iou_type))
