"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C-ABI
(hd_yolo_b200/libhdyolo_b200.so) and is compared with the oracle / the committed reference goldens.

Bars (BASELINE.json north_star): kept-index lists and labels bit-exact; boxes and scores within
1e-5 relative (they are bit-exact whenever no transcendental is involved); NMS decisions in fp32 in
torchvision's operation order.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, unpack_list
import hd_yolo_b200 as hdy
from oracle import nms_c, port
from hd_yolo_b200 import synth

pytestmark = pytest.mark.gpu

REL = 1e-5  # tolerance for values that pass through sigmoid (expf differs by ulps between libraries)
ATOL_PX = 1e-4  # pixel coordinates: cx - w/2 or (2s - 0.5 + g)*stride cancel near 0, so a purely relative
                # bound is meaningless there; 1e-4 px is 1e-5 of a 10 px nucleus


def _dets(g):
    i, dets, preds = 0, [], []
    while f"det{i}" in g:
        dets.append(torch.from_numpy(g[f"det{i}"]))
        preds.append(torch.from_numpy(g[f"pred{i}"]))
        i += 1
    return dets, preds


def _spec(g, extra=0):
    nc = int(g["nc"])
    return hdy.HeadSpec(g["anchors"].tolist(), g["strides"].tolist(), nc=nc, no=5 + nc + extra)


def _close(a, b, rel=REL, atol=1e-12):
    a, b = a.double(), b.double()
    return bool(((a - b).abs() <= rel * b.abs() + atol).all())


# ------------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("name", ["detect_640_l3", "detect_320_l4"])
def test_compute_proposals_vs_reference_golden(cuda_device, name):
    g = load_golden(name)
    dets, preds = _dets(g)
    out = hdy.compute_proposals([d.to(cuda_device) for d in dets], _spec(g))
    for o, p in zip(out, preds):
        assert o.shape == p.shape
        assert _close(o.cpu()[..., :4], p[..., :4], atol=ATOL_PX)
        assert _close(o.cpu()[..., 4:], p[..., 4:])


@pytest.mark.parametrize("name", ["detect_640_l3", "detect_320_l4"])
def test_decode_concat_layouts(cuda_device, name):
    g = load_golden(name)
    dets, preds = _dets(g)
    spec = _spec(g)
    cat_ref = port.concat_levels(preds)
    cat0 = hdy.decode_concat([d.to(cuda_device) for d in dets], spec, layout=0)
    assert _close(cat0.cpu()[..., :4], cat_ref[..., :4], atol=ATOL_PX)
    assert _close(cat0.cpu()[..., 4:], cat_ref[..., 4:])
    assert torch.equal(cat0.cpu()[..., -1], cat_ref[..., -1])  # level ids exact
    # planar layout [bs, na*no, ny, nx] (the conv's native output) gives the same bits
    planar = [d.permute(0, 1, 4, 2, 3).reshape(d.shape[0], -1, d.shape[2], d.shape[3]).contiguous().to(cuda_device)
              for d in dets]
    cat1 = hdy.decode_concat(planar, spec, layout=1)
    assert torch.equal(cat0, cat1)
    # compute_proposals and decode_concat agree bit for bit
    out = hdy.compute_proposals([d.to(cuda_device) for d in dets], spec)
    cat2 = torch.cat([o.view(o.shape[0], -1, spec.no) for o in out], 1)
    assert torch.equal(cat2, cat0[..., :-1])


def test_decode_odd_shapes_misaligned(cuda_device):
    # odd grid sizes / odd `no` make tile bases 4-byte aligned only: exercises the scalar head/tail path
    torch.manual_seed(5)
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=2)
    dets = [torch.randn(3, 3, ny, nx, 7) for ny, nx in [(9, 7), (5, 3), (1, 1)]]
    ref = port.concat_levels(port.compute_proposals(dets, synth.ANCHORS_3, synth.STRIDES_3))
    out = hdy.decode_concat([d.to(cuda_device) for d in dets], spec)
    assert _close(out.cpu()[..., :4], ref[..., :4], atol=ATOL_PX) and _close(out.cpu()[..., 4:], ref[..., 4:])


# ------------------------------------------------------------------------------- nms_per_image (N1)
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_nms_per_image_vs_reference_golden(cuda_device, tag):
    g = load_golden("nms_rows")
    preds = torch.from_numpy(g["preds"]).to(cuda_device)
    conf, iou, md = g[f"npi_{tag}_params"].tolist()
    out = hdy.nms_per_image(preds, int(g["nc"]), conf, iou, int(md))
    ref = unpack_list(g, f"npi_{tag}", ["boxes", "scores", "extra"])
    assert len(out) == len(ref)
    for a, b in zip(out, ref):
        for k in ("boxes", "scores", "extra"):
            assert a[k].shape == b[k].shape, (k, a[k].shape, b[k].shape)
            assert torch.equal(a[k].cpu(), b[k]), k   # no transcendental on this path: bit-exact


YOLO_KW = {"a": dict(conf_thres=0.25, iou_thres=0.45, max_det=300),
           "b": dict(conf_thres=0.1, iou_thres=0.45, multi_label=True, max_det=1000),
           "c": dict(conf_thres=0.25, iou_thres=0.5, agnostic=True, max_det=300),
           "d": dict(conf_thres=0.2, iou_thres=0.45, classes=[1, 3], max_det=300)}


@pytest.mark.parametrize("tag", list(YOLO_KW))
def test_non_max_suppression_vs_reference_golden(cuda_device, tag):
    g = load_golden("nms_rows")
    nc = int(g["nc"])
    pred = torch.from_numpy(g["preds"])[..., :5 + nc].contiguous().to(cuda_device)
    out = hdy.non_max_suppression(pred, **YOLO_KW[tag])
    sizes = g[f"yolo_{tag}_sizes"].tolist()
    assert [len(o) for o in out] == sizes
    assert torch.equal(torch.cat(out).cpu(), torch.from_numpy(g[f"yolo_{tag}_out"]))


def test_non_max_suppression_apriori_labels(cuda_device):
    g = load_golden("nms_rows")
    nc = int(g["nc"])
    pred = torch.from_numpy(g["preds"])[:2, :400, :5 + nc].contiguous()
    labels = [torch.tensor([[1, 50., 60., 20., 22.], [3, 200., 100., 30., 18.]]), torch.zeros((0, 5))]
    ref = port.non_max_suppression(pred.clone(), 0.25, 0.45, labels=labels)
    out = hdy.non_max_suppression(pred.to(cuda_device), 0.25, 0.45, labels=[l.to(cuda_device) for l in labels])
    for a, b in zip(out, ref):
        assert torch.equal(a.cpu(), b)


# ------------------------------------------------------------------------------------- plain nms
def _rand_boxes(g, n, span, lo, hi):
    c = torch.rand((n, 2), generator=g) * span
    wh = torch.rand((n, 2), generator=g) * (hi - lo) + lo
    return torch.cat([c - wh / 2, c + wh / 2], 1)


@pytest.mark.parametrize("n,span,lo,hi,thr", [
    (1, 10, 2, 5, 0.5), (2, 10, 8, 9, 0.1), (37, 40, 4, 20, 0.45), (1000, 640, 12, 36, 0.45),
    (3000, 1024, 12, 36, 0.45), (4096, 1024, 12, 36, 0.45), (4097, 1024, 12, 36, 0.45),
    (3000, 300, 10, 200, 0.3), (9000, 1024, 12, 36, 0.5), (20000, 640, 2, 400, 0.45),
    (2500, 100, 20, 30, 0.6), (2000, 50000, 12, 36, 0.45)])
def test_nms_vs_oracle_random(cuda_device, n, span, lo, hi, thr):
    g = torch.Generator().manual_seed(n + int(span))
    b = _rand_boxes(g, n, span, lo, hi)
    s = (torch.rand(n, generator=g) * 200).round() / 200  # plenty of exact ties
    ref = nms_c.nms(b.numpy(), s.numpy(), thr)
    out = hdy.nms(b.to(cuda_device), s.to(cuda_device), thr)
    assert out.dtype == torch.int64
    assert np.array_equal(out.cpu().numpy(), ref)


def test_nms_known_answers(cuda_device):
    def run(boxes, scores, thr):
        return hdy.nms(torch.tensor(boxes, dtype=torch.float32, device=cuda_device),
                       torch.tensor(scores, dtype=torch.float32, device=cuda_device), thr).tolist()
    assert run([[0, 0, 10, 10]] * 3, [.5, .5, .5], 0.5) == [0]
    assert run([[0, 0, 10, 10], [0, 0, 10, 5]], [.9, .8], 0.5) == [0, 1]     # iou == thr is kept (strict >)
    assert run([[0, 0, 10, 10], [0, 0, 10, 5]], [.9, .8], 0.4999) == [0]
    assert run([[5, 5, 5, 5], [5, 5, 5, 5]], [.9, .8], 0.1) == [0, 1]        # zero area: 0/0 never suppresses
    assert run([[0, 0, 4, 4], [10, 10, 14, 14], [0, 0, 4, 4]], [.1, .9, .5], 0.5) == [1, 2]
    assert run([[3, 3, 1, 1], [0, 0, 4, 4]], [.9, .8], 0.0) == [0, 1]        # inverted box never intersects
    assert hdy.nms(torch.zeros((0, 4), device=cuda_device), torch.zeros(0, device=cuda_device), 0.5).numel() == 0
    # chain a>b>c: a kills b, so c (overlapping only b) survives
    assert run([[0, 0, 10, 10], [4, 0, 14, 10], [8, 0, 18, 10]], [.9, .8, .7], 0.3) == [0, 2]


def test_nms_threshold_compare_modes(cuda_device):
    # iou exactly float32(0.3): torchvision CPU (float > double) suppresses, torchvision CUDA (fp32) keeps
    a = [0.0, 0.0, 10.0, 10.0]
    # find a box whose fp32 IoU with `a` equals float32(0.3) exactly: w*10 / (100 + w*10 - w*10) -> w = 3 gives 0.3
    b = [0.0, 0.0, 3.0, 10.0]
    iou = np.float32(30.0) / np.float32(100.0)
    assert iou == np.float32(0.3)
    boxes = torch.tensor([a, b], device=cuda_device)
    scores = torch.tensor([.9, .8], device=cuda_device)
    assert port.nms(boxes.cpu(), scores.cpu(), 0.3).tolist() == [0]
    hdy.set_iou_compare("cpu")
    assert hdy.nms(boxes, scores, 0.3).tolist() == [0]
    hdy.set_iou_compare("cuda")
    assert hdy.nms(boxes, scores, 0.3).tolist() == [0, 1]
    hdy.set_iou_compare("cpu")


def test_batched_nms_coordinate_trick(cuda_device):
    import torchvision
    g = torch.Generator().manual_seed(3)
    b = _rand_boxes(g, 900, 200, 10, 60)
    s = torch.rand(900, generator=g)
    idx = torch.randint(0, 5, (900,), generator=g)
    ref = torchvision.ops.batched_nms(b, s, idx, 0.5)
    out = hdy.batched_nms(b.to(cuda_device), s.to(cuda_device), idx.to(cuda_device), 0.5)
    assert torch.equal(out.cpu(), ref)


# ------------------------------------------------------------------------------- fused head path
def _oracle_on_device_decode(cat_gpu, nc, conf, iou, max_det):
    """Oracle NMS + score select applied to the rows the DEVICE decoded: isolates the decision logic
    from last-ulp differences between CUDA's and the CPU's expf."""
    cat = cat_gpu.cpu()
    outs = port.nms_per_image(cat, nc, conf, iou, max_det)
    res = []
    for o in outs:
        s, l = port.select_scores(o['scores'].clone(), conf, port.default_descendants(nc))
        res.append({'boxes': o['boxes'], 'scores': s, 'labels': l, 'levels': o['extra'][:, 0]})
    return res


@pytest.mark.parametrize("name,layout", [("detect_640_l3", 0), ("detect_640_l3", 1), ("detect_320_l4", 0)])
def test_detect_postprocess_bit_exact_on_device_rows(cuda_device, name, layout):
    g = load_golden(name)
    dets, _ = _dets(g)
    spec = _spec(g)
    conf, iou, md = float(g["conf_thres"]), float(g["iou_thres"]), int(g["max_det"])
    d0 = [d.to(cuda_device) for d in dets]
    cat = hdy.decode_concat(d0, spec)
    ref = _oracle_on_device_decode(cat, spec.nc, conf, iou, md)
    if layout == 1:
        d0 = [d.permute(0, 1, 4, 2, 3).reshape(d.shape[0], -1, d.shape[2], d.shape[3]).contiguous() for d in d0]
    out = hdy.detect_postprocess(d0, spec, conf, iou, md, layout=layout)
    lst = out.to_list()
    for i, (a, b) in enumerate(zip(lst, ref)):
        k = len(b['boxes'])
        assert k > 0 and len(a['boxes']) == k
        assert torch.equal(a['boxes'].cpu(), b['boxes'])
        assert torch.equal(a['scores'].cpu(), b['scores'])
        assert torch.equal(a['labels'].cpu(), b['labels'])
        assert torch.equal(out.levels[i, :k].cpu(), b['levels'])


@pytest.mark.parametrize("name", ["detect_640_l3", "detect_320_l4"])
def test_detect_postprocess_vs_reference_golden(cuda_device, name):
    """End to end against what the reference itself returned (CPU sigmoid): same detections, labels
    identical, boxes/scores within 1e-5 relative."""
    g = load_golden(name)
    dets, _ = _dets(g)
    spec = _spec(g)
    conf, iou, md = float(g["conf_thres"]), float(g["iou_thres"]), int(g["max_det"])
    out = hdy.detect_postprocess([d.to(cuda_device) for d in dets], spec, conf, iou, md).to_list()
    ref = unpack_list(g, "out", ["boxes", "scores", "labels"])
    for a, b in zip(out, ref):
        assert len(a['boxes']) == len(b['boxes'])
        assert torch.equal(a['labels'].cpu(), b['labels'])
        assert _close(a['boxes'].cpu(), b['boxes'], atol=ATOL_PX)
        assert _close(a['scores'].cpu(), b['scores'])


def test_nms_per_image_pipeline_equals_fused(cuda_device):
    """decode_concat -> nms_per_image (the reference's two-step call sequence) == fused path."""
    dets = synth.nuclei_logits(3, 320, 4, 400, seed=21, conf=0.25)
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    d0 = [d.to(cuda_device) for d in dets]
    two = hdy.nms_per_image(hdy.decode_concat(d0, spec), 4, 0.25, 0.45, 1000)
    one = hdy.detect_postprocess(d0, spec, 0.25, 0.45, 1000)
    for i, t in enumerate(two):
        k = int(one.counts[i])
        assert k == len(t['boxes']) and k > 100
        assert torch.equal(one.boxes[i, :k], t['boxes'])
        assert torch.equal(one.levels[i, :k], t['extra'][:, 0])


def test_extra_channels_are_carried(cuda_device):
    dets = synth.nuclei_logits(2, 160, 4, 120, seed=8, conf=0.25, extra=32)
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=41)
    out = hdy.detect_postprocess([d.to(cuda_device) for d in dets], spec, 0.25, 0.45, 500)
    cat = torch.cat([d.view(d.shape[0], -1, 41) for d in dets], 1)
    for i in range(2):
        k = int(out.counts[i])
        rows = out.rows[i, :k].cpu().long()
        assert torch.equal(out.extra[i, :k].cpu(), cat[i, rows, 9:])


@pytest.mark.parametrize("kernel", ["tma", "planar", "generic"])
@pytest.mark.parametrize("tile,bs,n_cand,conf", [(320, 3, 500, 0.25), (640, 2, 1000, 0.15), (160, 5, 60, 0.5)])
def test_wide_rows_filters_equal_two_step_path(cuda_device, tile, bs, n_cand, conf, kernel):
    """no = 41 (32 mask coefficients behind the scores), through the TMA streamer (layout 0), the planar filter
    (conv-native layout 1) and the one-row-per-thread filter (layout 1 with level tensors 4 bytes off a 16-byte
    boundary): same survivors, boxes, scores, labels and rows as decode_concat -> nms_per_image on the same logits, and
    as the oracle on the device-decoded rows; ragged last chunks (160-px tiles: 1200 + 300 + 75 rows) and a level that
    contributes nothing included."""
    layout = 0 if kernel == "tma" else 1                          # conv-native [bs, na*no, ny, nx]: same logits
    dets = synth.nuclei_logits(bs, tile, 4, n_cand, seed=tile + bs, conf=conf, extra=32)
    dets[0][bs - 1, ..., 4] = -20.0                                # last tile: level 0 contributes nothing
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=41)
    d0 = [d.to(cuda_device) for d in dets]
    raw = torch.cat([d.view(d.shape[0], -1, 41) for d in dets], 1)
    src = d0 if layout == 0 else [d.permute(0, 1, 4, 2, 3).reshape(d.shape[0], -1, d.shape[2], d.shape[3]).contiguous()
                                  for d in d0]
    if kernel == "generic":
        src = [torch.empty(d.numel() + 1, device=cuda_device)[1:].view(d.shape).copy_(d) for d in src]
        assert all(d.data_ptr() % 16 == 4 for d in src)
    one = hdy.detect_postprocess(src, spec, conf, 0.45, 2000, layout=layout)
    cat = hdy.decode_concat(d0, spec)
    two = hdy.nms_per_image(cat, 4, conf, 0.45, 2000)
    ref = port.nms_per_image(cat.cpu(), 4, conf, 0.45, 2000)
    total = 0
    for i, (t, r) in enumerate(zip(two, ref)):
        k = int(one.counts[i])
        total += k
        assert k == len(t['boxes']) == len(r['boxes'])
        assert torch.equal(one.boxes[i, :k], t['boxes']) and torch.equal(one.boxes[i, :k].cpu(), r['boxes'])
        s, l = port.select_scores(r['scores'].clone(), conf, port.default_descendants(4))
        assert torch.equal(one.scores[i, :k].cpu(), s) and torch.equal(one.labels[i, :k].cpu(), l)
        assert torch.equal(one.levels[i, :k].cpu(), r['extra'][:, -1])      # the level-id column (yolo_head.py:311)
        rows = one.rows[i, :k].cpu().long()
        assert torch.equal(one.extra[i, :k].cpu(), raw[i, rows, 9:])        # raw coefficients ride along
    assert total > bs * n_cand // 3


def test_empty_and_overflow(cuda_device):
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    dets = synth.nuclei_logits(2, 160, 4, 100, seed=9, conf=0.25)
    dets = [d.to(cuda_device) for d in dets]
    for d in dets:
        d[1, ..., 4] = -20.0  # tile 1: nothing passes
    out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, 300)
    lst = out.to_list()
    assert len(lst[0]['boxes']) > 20 and lst[1]['boxes'].shape == (0, 4) and lst[1]['labels'].shape == (0,)
    small = hdy.detect_postprocess(dets, spec, 0.25, 0.45, 300, cap=16)
    with pytest.raises(hdy.HdyError, match="overflow"):
        small.to_list()
    # bs = 0 / N = 0 in the reference-signature wrappers
    assert hdy.nms_per_image(torch.zeros((0, 10, 9), device=cuda_device), 4) == []
    r = hdy.nms_per_image(torch.zeros((2, 0, 10), device=cuda_device), 4)
    assert r[0]['boxes'].shape == (0, 4) and r[0]['scores'].shape == (0, 5) and r[0]['extra'].shape == (0, 1)


def test_hier_tree_select(cuda_device):
    g = load_golden("hier_tree")
    from hd_yolo_b200 import _lib
    from hd_yolo_b200.ops import _stream
    import ctypes as C
    x = torch.from_numpy(g["scores_in"]).to(cuda_device).clone()[None].contiguous()  # [1, k, 1+nc]
    k, ns = x.shape[1], x.shape[2]
    ops = list(zip(g["ops_dst"].tolist(), g["ops_src"].tolist()))
    flat = (C.c_int32 * (2 * len(ops)))(*[v for p in ops for v in p])
    counts = torch.tensor([k], dtype=torch.int32, device=cuda_device)
    score = torch.empty((1, k), device=cuda_device)
    label = torch.empty((1, k), dtype=torch.int64, device=cuda_device)
    _lib.check(_lib.load().hdy_select_scores(_lib.ptr(x), _lib.ptr(counts), 1, k, ns - 1, flat, len(ops), 0.2,
                                             _lib.ptr(score), _lib.ptr(label), _stream()))
    assert torch.equal(x[0].cpu(), torch.from_numpy(g["scores_out"]))
    desc = {}
    for kk, v in zip(g["ops_src"].tolist(), g["ops_dst"].tolist()):
        desc.setdefault(kk, []).append(v)
    s_ref, l_ref = port.select_scores(torch.from_numpy(g["scores_in"]).clone(), 0.2, desc)
    assert torch.equal(score[0].cpu(), s_ref) and torch.equal(label[0].cpu(), l_ref)


# ------------------------------------------------------------- full-size, size-independent properties
@pytest.mark.parametrize("tile,bs,n_cand,md", [(640, 64, 1000, 1000), (1024, 32, 3000, 3000)])
def test_full_size_properties(cuda_device, tile, bs, n_cand, md):
    """BASELINE.json configs[1]/[2] shapes.  Checked without the (slow) oracle: score order,
    idempotence (NMS of the survivors keeps all of them), pairwise IoU of survivors <= thr on a
    sample, candidate counts near the target; one tile is checked against the oracle outright."""
    dets = synth.nuclei_logits(bs, tile, 4, n_cand, seed=tile, conf=0.25, generator_device="cuda")
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, md)
    torch.cuda.synchronize()
    cand = out.cand_counts[:bs].float()
    assert abs(float(cand.mean()) - n_cand) < 0.1 * n_cand and int(out.cand_counts[bs]) == 0
    counts = out.counts.cpu().tolist()
    for i in range(0, bs, max(1, bs // 8)):
        k = counts[i]
        assert 0 < k <= md
        obj = out.scores_full[i, :k, 0]
        cls_best = out.scores_full[i, :k, 1:].max(1).values
        # survivors are listed by descending objectness (hierarchical products leave column 0 alone)
        assert bool((obj[:-1] >= obj[1:]).all())
        assert bool((cls_best <= obj).all())
        b = out.boxes[i, :k]
        again = hdy.nms(b, obj, 0.45)
        assert again.numel() == k and torch.equal(again, torch.arange(k, device=b.device))
    # one tile outright against the oracle on device-decoded rows
    cat = hdy.decode_concat([d[:1].contiguous() for d in dets], spec)
    ref = _oracle_on_device_decode(cat, 4, 0.25, 0.45, md)[0]
    k = counts[0]
    assert k == len(ref['boxes'])
    assert torch.equal(out.boxes[0, :k].cpu(), ref['boxes'])
    assert torch.equal(out.labels[0, :k].cpu(), ref['labels'])
    assert torch.equal(out.scores[0, :k].cpu(), ref['scores'])


@pytest.mark.parametrize("n_small,n_large,seed", [(2500, 40, 0), (3500, 6, 1), (800, 200, 2)])
def test_nms_small_nuclei_with_large_boxes(cuda_device, n_small, n_large, seed):
    """Nuclei-sized boxes plus clusters of near-identical LARGE boxes (the "large" bucket of the per-tile kernel, which
    the whole CTA scans; clusters of > 4 make their dominator lists overflow) vs torchvision.ops.nms."""
    import torchvision
    g = torch.Generator().manual_seed(seed)
    c = torch.rand((n_small, 2), generator=g) * 1000
    s = 12 + 24 * torch.rand((n_small, 2), generator=g)
    small = torch.cat([c - s / 2, c + s / 2], 1)
    centers = torch.rand((max(n_large // 8, 1), 2), generator=g) * 600 + 200
    which = torch.randint(0, len(centers), (n_large,), generator=g)
    lc = centers[which] + 6 * torch.rand((n_large, 2), generator=g)
    ls = 250 + 30 * torch.rand((n_large, 2), generator=g)
    large = torch.cat([lc - ls / 2, lc + ls / 2], 1)
    boxes = torch.cat([small, large])
    scores = torch.rand((len(boxes),), generator=g)
    perm = torch.randperm(len(boxes), generator=g)
    boxes, scores = boxes[perm].contiguous(), scores[perm].contiguous()
    for thr in (0.45, 0.7):
        ref = torchvision.ops.nms(boxes, scores, thr)
        got = hdy.nms(boxes.to(cuda_device), scores.to(cuda_device), thr).cpu()
        assert torch.equal(got, ref)


@pytest.mark.parametrize("nc,extra,layout", [(40, 0, 0), (40, 3, 1), (31, 5, 0), (4, 32, 1)])
def test_detect_postprocess_many_classes_and_extras(cuda_device, nc, extra, layout):
    """1 + nc > 32 takes hdy_gather_logits + hdy_select_scores, otherwise the fused warp-per-survivor kernel; both
    must give what the oracle gives on the device-decoded rows, and carry the raw extra channels."""
    dets = synth.nuclei_logits(2, 160, nc, 150, seed=nc + extra, extra=extra, conf=0.25)
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=nc, no=5 + nc + extra)
    d0 = [d.to(cuda_device) for d in dets]
    cat = hdy.decode_concat(d0, spec)
    ref = _oracle_on_device_decode(cat, nc, 0.25, 0.45, 300)
    src = d0
    if layout == 1:
        src = [d.permute(0, 1, 4, 2, 3).reshape(d.shape[0], -1, d.shape[2], d.shape[3]).contiguous() for d in d0]
    out = hdy.detect_postprocess(src, spec, 0.25, 0.45, 300, layout=layout)
    lst = out.to_list()
    rawcat = torch.cat([d.reshape(2, -1, spec.no) for d in dets], 1)
    for i, (a, b) in enumerate(zip(lst, ref)):
        k = len(b['boxes'])
        assert k > 0 and len(a['boxes']) == k
        assert torch.equal(a['boxes'].cpu(), b['boxes'])
        assert torch.equal(a['scores'].cpu(), b['scores'])
        assert torch.equal(a['labels'].cpu(), b['labels'])
        if extra:
            rows = out.rows[i, :k].cpu().long()
            assert torch.equal(out.extra[i, :k].cpu(), rawcat[i, rows, 5 + nc:])


# ------------------------------------------------------------------------------------------ fp16 ingestion
@pytest.mark.parametrize("tile,bs,n_cand,extra", [(320, 3, 400, 0), (640, 4, 1000, 32), (1024, 2, 3000, 0)])
def test_fp16_logits_equal_fp32_path_on_rounded_inputs(cuda_device, tile, bs, n_cand, extra):
    """val_nuclei.py:115-116: on CUDA the reference runs a half() model, so the head hands over fp16 logits.  They are
    widened on load (exact), all arithmetic stays fp32: every output must be BIT-identical to the fp32 path fed the
    fp16-rounded numbers -- and the oracle, fed those numbers as fp32, keeps the same rows."""
    dets = synth.nuclei_logits(bs, tile, 4, n_cand, seed=tile + extra, conf=0.25, extra=extra,
                               generator_device="cuda")
    d16 = [d.half() for d in dets]
    d32 = [d.float() for d in d16]
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=9 + extra)
    a = hdy.detect_postprocess(d16, spec, 0.25, 0.45, 3000, cap=4096)
    b = hdy.detect_postprocess(d32, spec, 0.25, 0.45, 3000, cap=4096)
    assert torch.equal(a.counts, b.counts) and torch.equal(a.cand_counts, b.cand_counts)
    kc = a.counts.cpu().tolist()
    assert min(kc) > 0.5 * n_cand
    for i, k in enumerate(kc):
        for f in ("boxes", "scores_full", "scores", "labels", "levels", "rows") + (("extra",) if extra else ()):
            assert torch.equal(getattr(a, f)[i, :k], getattr(b, f)[i, :k]), f
    assert torch.equal(hdy.decode_concat(d16, spec), hdy.decode_concat(d32, spec))
    ref = _oracle_on_device_decode(hdy.decode_concat(d32, spec)[:1], 4, 0.25, 0.45, 3000)[0]
    assert torch.equal(a.boxes[0, :kc[0]].cpu(), ref['boxes']) and torch.equal(a.labels[0, :kc[0]].cpu(), ref['labels'])


def test_fp16_logits_golden_rows_and_unaligned_levels(cuda_device):
    """Reference golden logits rounded to fp16: same kept rows as the oracle on the rounded numbers; a level tensor that
    is not 16-byte aligned (a view at an odd offset) is refused loudly -- there is no slow fp16 path to fall into."""
    g = load_golden("detect_640_l3")
    dets, _ = _dets(g)
    spec = _spec(g)
    conf, iou, md = float(g["conf_thres"]), float(g["iou_thres"]), int(g["max_det"])
    d16 = [d.to(cuda_device).half() for d in dets]
    out = hdy.detect_postprocess(d16, spec, conf, iou, md).to_list()
    ref = _oracle_on_device_decode(hdy.decode_concat([d.float() for d in d16], spec), spec.nc, conf, iou, md)
    for a, b in zip(out, ref):
        assert torch.equal(a['boxes'].cpu(), b['boxes']) and torch.equal(a['labels'].cpu(), b['labels'])
    flat = torch.zeros((d16[0].numel() + 8,), dtype=torch.float16, device=cuda_device)
    odd = flat[1:1 + d16[0].numel()].view(d16[0].shape)
    odd.copy_(d16[0])
    with pytest.raises(hdy.HdyError):
        hdy.detect_postprocess([odd] + d16[1:], spec, conf, iou, md)


# ------------------------------------------------------------------------------------------ every tile, full size
@pytest.mark.parametrize("tile,bs,n_cand,md", [(640, 64, 1000, 1000), (1024, 128, 3000, 3000)])
def test_full_size_every_tile_against_the_oracle(cuda_device, tile, bs, n_cand, md):
    """BASELINE.json configs[1] (64 tiles of 640 px) and configs[2] (128 tiles of 1024 px) at their FULL sizes: every
    tile's kept boxes / scores / labels against the oracle (nms_per_image + score select on the device-decoded rows)."""
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    dets = synth.nuclei_logits(bs, tile, 4, n_cand, seed=7 * tile, conf=0.25, generator_device="cuda")
    out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, md, cap=4096)
    counts = out.counts.cpu().tolist()
    assert int(out.cand_counts[bs]) == 0
    boxes, scores, labels = out.boxes.cpu(), out.scores.cpu(), out.labels.cpu()
    for t0 in range(0, bs, 16):
        cat = hdy.decode_concat([d[t0:t0 + 16].contiguous() for d in dets], spec)
        ref = _oracle_on_device_decode(cat, 4, 0.25, 0.45, md)
        for j, r in enumerate(ref):
            i, k = t0 + j, counts[t0 + j]
            assert k == len(r['boxes']), f"tile {i}"
            assert torch.equal(boxes[i, :k], r['boxes']) and torch.equal(scores[i, :k], r['scores']) and \
                torch.equal(labels[i, :k], r['labels']), f"tile {i}"


# ------------------------------------------------------------------------------------------ the library GPU path
def test_kept_indices_from_raw_logits_match_torch_cuda_reference(cuda_device):
    """The north star's own wording: kept-detection index lists bit-exact against the reference's PyTorch/torchvision
    path -- here run on the SAME B200 (oracle/port.py on CUDA tensors: ATen's CUDA sigmoid, torchvision's CUDA nms,
    `set_iou_compare("cuda")`), from RAW logits, on >= 1 000 tiles.  Row lists and labels must be identical on every
    tile; a tile where they are not is reported with the margin of the row that flipped."""
    import torchvision  # noqa: F401
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    hdy.set_iou_compare("cuda")
    try:
        n_tiles, bad = 0, []
        for rep in range(8):
            bs = 128
            dets = synth.nuclei_logits(bs, 320, 4, 350, seed=9000 + rep, conf=0.25, generator_device="cuda")
            out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, 1000)
            counts = out.counts.cpu().tolist()
            preds = port.compute_proposals(dets, synth.ANCHORS_3, synth.STRIDES_3)      # ATen CUDA kernels
            cat = port.concat_levels(preds)
            ref = port.nms_per_image(cat, 4, 0.25, 0.45, 1000)                          # torchvision CUDA nms
            for i, r in enumerate(ref):
                k = counts[i]
                s, l = port.select_scores(r['scores'].clone(), 0.25, port.default_descendants(4))
                if k != len(r['boxes']) or not torch.equal(out.labels[i, :k], l):
                    bad.append((rep, i, k, len(r['boxes'])))
                    continue
                b = out.boxes[i, :k]
                if not bool(((b - r['boxes']).abs() <= 1e-5 * r['boxes'].abs() + 1e-4).all()):
                    bad.append((rep, i, "boxes"))
                if not bool(((out.scores[i, :k] - s).abs() <= 1e-5 * s.abs()).all()):
                    bad.append((rep, i, "scores"))
            n_tiles += bs
        assert n_tiles >= 1000
        assert not bad, f"{len(bad)} of {n_tiles} tiles differ from the torch/torchvision CUDA path: {bad[:5]}"
    finally:
        hdy.set_iou_compare("cpu")


def test_nms_instances_agree(cuda_device):
    """hdy_nms_tiles has two shared-memory instances, chosen by cap (<= 3072 candidates: 126 KB, shares an SM with a
    filter CTA; 4096: 168 KB).  The same candidate lists through both give identical survivors, and what the oracle
    keeps."""
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4)
    dets = synth.nuclei_logits(6, 1024, 4, 2900, seed=31, conf=0.25, generator_device="cuda")
    ref = None
    for cap in (3072, 4096):                                       # every list has <= 3072 candidates: the same lists
        out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, 3072, cap=cap)
        assert int(out.cand_counts[-1]) == 0 and int(out.cand_counts[:-1].max()) > 2900
        assert int(out.cand_counts.max()) <= 3072
        got = (out.counts.clone(), out.rows.clone(), out.boxes.clone(), out.scores.clone())
        kc = got[0].cpu().tolist()
        if ref is None:
            ref = got
            o = _oracle_on_device_decode(hdy.decode_concat([d[:1].contiguous() for d in dets], spec), 4, 0.25, 0.45,
                                         3072)[0]
            assert torch.equal(out.boxes[0, :kc[0]].cpu(), o['boxes'])
        else:
            assert torch.equal(got[0], ref[0])
            for i, k in enumerate(kc):
                assert torch.equal(got[1][i, :k], ref[1][i, :k]) and torch.equal(got[2][i, :k], ref[2][i, :k])
