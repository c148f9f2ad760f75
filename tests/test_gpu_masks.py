"""GPU parity tests of the mask stage (pytest -m gpu), through the C-ABI, against the reference golden
(paste_masks_in_image) and the oracle port.

Bars (BASELINE.json north_star): binary masks agree on >= 99.99 % of pixels; dense fp32 canvases within 2e-6
absolute of the reference (values are probabilities in [0,1]; ATen's CPU bilinear kernel contracts some products
into FMAs, the device code rounds every product, so the last bit can differ)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
import hd_yolo_b200 as hdy
from hd_yolo_b200 import masks as hm
from oracle import port

pytestmark = pytest.mark.gpu

AGREE = 0.9999
ATOL = 2e-6


def _agreement(a, b):
    return float((a == b).double().mean())


def _rand_boxes(g, k, H, W, lo, hi):
    c = torch.rand((k, 2), generator=g) * torch.tensor([W, H], dtype=torch.float32)
    s = torch.rand((k, 2), generator=g) * (hi - lo) + lo
    return torch.cat([c - s / 2, c + s / 2], 1)


# ------------------------------------------------------------------------------------------------ M1
def test_mask_select_vs_oracle(cuda_device):
    g = torch.Generator().manual_seed(1)
    K, C, M, nc = 37, 3, 28, 4
    logits = torch.randn((K, C, M, M), generator=g) * 3
    labels = torch.randint(-1, nc + 1, (K,), generator=g)
    labels[labels < 0] = -100                                   # the reference's "no class" label
    mask_indices = torch.tensor([0, 0, 1, -1, 2])               # class 3 has no mask head
    ref = port.mask_select(logits, labels, mask_indices)
    out = hm.mask_select(logits.to(cuda_device), labels.to(cuda_device), mask_indices.to(cuda_device))
    assert out.shape == ref.shape == (K, 1, M, M)
    assert float((out.cpu() - ref).abs().max()) < ATOL
    zero = mask_indices[labels.clamp(min=0)] < 0
    assert zero.any() and bool((out.cpu()[zero] == 0).all())


# ------------------------------------------------------------------------------------------------ M2
def test_paste_masks_vs_reference_golden(cuda_device):
    g = load_golden("paste_masks")
    H, W = g["shape"].tolist()
    masks, boxes, ref = torch.from_numpy(g["masks"]), torch.from_numpy(g["boxes"]), torch.from_numpy(g["out"])
    out = hm.paste_masks_in_image(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=1)
    assert out.shape == ref.shape and out.dtype == torch.float32
    assert float((out.cpu() - ref).abs().max()) < ATOL
    assert bool(((out.cpu() == 0) == (ref == 0)).all())        # identical paste windows
    packed = hm.paste_masks_packed(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=1)
    packed.check()
    dense = packed.to_dense().cpu()
    assert _agreement(dense, (ref[:, 0] > 0.5).to(torch.uint8)) >= AGREE
    assert torch.equal(dense, (out[:, 0] > 0.5).to(torch.uint8).cpu())   # packed == dense path, bit for bit


@pytest.mark.parametrize("k,H,W,lo,hi,pad", [(300, 640, 640, 8, 48, 1), (64, 200, 333, 1, 150, 1), (50, 128, 128, 4, 40, 0),
                                              (40, 100, 90, 2, 30, 2)])
def test_paste_masks_vs_oracle_random(cuda_device, k, H, W, lo, hi, pad):
    g = torch.Generator().manual_seed(k + H)
    masks = torch.rand((k, 1, 28, 28), generator=g)
    boxes = _rand_boxes(g, k, H, W, lo, hi)
    ref = port.paste_masks_in_image(masks, boxes, (H, W), padding=pad)
    out = hm.paste_masks_in_image(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=pad).cpu()
    assert float((out - ref).abs().max()) < ATOL
    packed = hm.paste_masks_packed(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=pad)
    assert _agreement(packed.to_dense().cpu(), (ref[:, 0] > 0.5).to(torch.uint8)) >= AGREE
    # geometry: window == bounding box of the reference's non-zero paste region (masks are > 0 everywhere inside)
    geom = packed.geom.cpu()
    for i in range(0, k, max(1, k // 16)):
        nz = ref[i, 0].nonzero()
        x0, y0, w, h = geom[i].tolist()
        if len(nz) == 0:
            continue
        assert y0 <= int(nz[:, 0].min()) and int(nz[:, 0].max()) < y0 + h
        assert x0 <= int(nz[:, 1].min()) and int(nz[:, 1].max()) < x0 + w


def test_paste_fused_sigmoid_channel(cuda_device):
    """M1 + M2 + M3 in one kernel == mask_select -> paste -> > 0.5 done separately."""
    g = torch.Generator().manual_seed(9)
    K, C, M, H, W = 80, 2, 28, 320, 320
    logits = torch.randn((K, C, M, M), generator=g) * 2
    labels = torch.randint(0, 5, (K,), generator=g)
    mask_indices = torch.tensor([0, 0, 1, -1, 1])
    boxes = _rand_boxes(g, K, H, W, 10, 40)
    ch = mask_indices[labels.clamp(min=0)].to(torch.int32)
    sel = hm.mask_select(logits.to(cuda_device), labels.to(cuda_device), mask_indices.to(cuda_device))
    two = hm.paste_masks_packed(sel, boxes.to(cuda_device), (H, W)).to_dense()
    one = hm.paste_masks_packed(logits.to(cuda_device), boxes.to(cuda_device), (H, W), channel=ch.to(cuda_device),
                                apply_sigmoid=True).to_dense()
    assert torch.equal(one, two)
    ref = port.paste_masks_in_image(port.mask_select(logits, labels, mask_indices), boxes, (H, W))
    assert _agreement(one.cpu(), (ref[:, 0] > 0.5).to(torch.uint8)) >= AGREE


def test_paste_empty_and_capacity(cuda_device):
    z = hm.paste_masks_in_image(torch.zeros((0, 1, 28, 28), device=cuda_device), torch.zeros((0, 4), device=cuda_device),
                                (32, 48))
    assert z.shape == (0, 1, 32, 48)
    p = hm.paste_masks_packed(torch.zeros((0, 1, 28, 28), device=cuda_device), torch.zeros((0, 4), device=cuda_device),
                              (32, 48))
    assert len(p) == 0 and p.to_dense().shape == (0, 32, 48)
    g = torch.Generator().manual_seed(2)
    masks = torch.rand((10, 1, 28, 28), generator=g).to(cuda_device)
    boxes = _rand_boxes(g, 10, 64, 64, 10, 30).to(cuda_device)
    small = hm.paste_masks_packed(masks, boxes, (64, 64), capacity_words=8)
    with pytest.raises(hdy.HdyError, match="overflow"):
        small.check()
    with pytest.raises(hdy.HdyError):
        hm.paste_masks_in_image(torch.zeros((1, 1, 28, 28)), torch.zeros((1, 4)), (8, 8))   # CPU tensors


# ------------------------------------------------------------------------------- process_mask (variant B)
@pytest.mark.parametrize("upsample", [False, True])
@pytest.mark.parametrize("n,mh,mw,ih,iw", [(120, 160, 160, 640, 640), (33, 40, 56, 160, 224), (7, 24, 24, 90, 100)])
def test_process_mask_vs_oracle(cuda_device, upsample, n, mh, mw, ih, iw):
    g = torch.Generator().manual_seed(n)
    protos = torch.randn((32, mh, mw), generator=g)
    coef = torch.randn((n, 32), generator=g) * 0.5
    boxes = _rand_boxes(g, n, ih, iw, 6, 60)
    boxes[0] = torch.tensor([-5.0, -3.0, 20.5, 17.25])          # clipped
    boxes[1] = torch.tensor([iw - 9.5, ih - 12.0, iw + 8.0, ih + 3.0])
    ref = port.process_mask(protos, coef, boxes.clone(), (ih, iw), upsample=upsample)
    out = hm.process_mask(protos.to(cuda_device), coef.to(cuda_device), boxes.to(cuda_device), (ih, iw), upsample=upsample)
    assert out.shape == ref.shape
    assert set(out.unique().tolist()) <= {0.0, 1.0}
    assert _agreement(out.cpu(), ref) >= AGREE
    assert float(ref.sum()) > 0
    # bit-packed variant == dense variant, exactly
    counts = torch.tensor([n], dtype=torch.int32, device=cuda_device)
    packed = hm.process_mask_packed(protos.to(cuda_device)[None], coef.to(cuda_device)[None], boxes.to(cuda_device)[None],
                                    counts, (ih, iw), upsample=upsample)
    packed.check()
    assert torch.equal(packed.to_dense(), out.to(torch.uint8))


def test_process_mask_batch_counts(cuda_device):
    g = torch.Generator().manual_seed(4)
    bs, md, mh, mw, ih, iw = 3, 20, 40, 40, 160, 160
    protos = torch.randn((bs, 32, mh, mw), generator=g)
    coef = torch.randn((bs, md, 32), generator=g)
    boxes = torch.stack([_rand_boxes(g, md, ih, iw, 8, 50) for _ in range(bs)])
    counts = torch.tensor([20, 0, 7], dtype=torch.int32)
    out = hm.process_mask_batch(protos.to(cuda_device), coef.to(cuda_device), boxes.to(cuda_device), counts.to(cuda_device),
                                (ih, iw), upsample=True).cpu()
    for i, k in enumerate(counts.tolist()):
        assert float(out[i, k:].abs().sum()) == 0
        if k:
            ref = port.process_mask(protos[i], coef[i, :k], boxes[i, :k].clone(), (ih, iw), upsample=True)
            assert _agreement(out[i, :k], ref) >= AGREE
    assert hm.process_mask(protos[0].to(cuda_device), coef[0, :0].to(cuda_device), boxes[0, :0].to(cuda_device), (ih, iw)).shape == (0, mh, mw)


@pytest.mark.parametrize("upsample", [False, True])
def test_process_mask_mixed_small_and_large_boxes(cuda_device, upsample):
    """Boxes up to 64 px go through the two-phase path (TMA-staged regions -> patches -> upsample/pack), larger ones
    through the per-detection kernel; both write into the same bit planes."""
    g = torch.Generator().manual_seed(11)
    n, mh, mw, ih, iw = 90, 96, 128, 384, 512
    protos = torch.randn((32, mh, mw), generator=g)
    coef = torch.randn((n, 32), generator=g) * 0.5
    boxes = torch.cat([_rand_boxes(g, 60, ih, iw, 6, 60), _rand_boxes(g, 30, ih, iw, 70, 300)])
    ref = port.process_mask(protos, coef, boxes.clone(), (ih, iw), upsample=upsample)
    dev = cuda_device
    out = hm.process_mask(protos.to(dev), coef.to(dev), boxes.to(dev), (ih, iw), upsample=upsample)
    assert _agreement(out.cpu(), ref) >= AGREE
    counts = torch.tensor([n], dtype=torch.int32, device=dev)
    packed = hm.process_mask_packed(protos.to(dev)[None], coef.to(dev)[None], boxes.to(dev)[None], counts, (ih, iw),
                                    upsample=upsample)
    packed.check()
    assert torch.equal(packed.to_dense(), out.to(torch.uint8))
    # a second call re-uses the bit planes' storage pattern: stale words must not leak (nothing is memset)
    packed2 = hm.process_mask_packed(protos.to(dev)[None], coef.to(dev)[None], boxes.to(dev)[None], counts, (ih, iw),
                                     upsample=upsample)
    assert torch.equal(packed2.to_dense(), out.to(torch.uint8))


def test_process_mask_other_prototype_counts(cuda_device):
    """nm != 32 takes the per-detection kernel."""
    g = torch.Generator().manual_seed(12)
    n, nm, mh, mw, ih, iw = 25, 16, 40, 40, 160, 160
    protos = torch.randn((nm, mh, mw), generator=g)
    coef = torch.randn((n, nm), generator=g) * 0.7
    boxes = _rand_boxes(g, n, ih, iw, 8, 80)
    ref = port.process_mask(protos, coef, boxes.clone(), (ih, iw), upsample=True)
    out = hm.process_mask(protos.to(cuda_device), coef.to(cuda_device), boxes.to(cuda_device), (ih, iw), upsample=True)
    assert _agreement(out.cpu(), ref) >= AGREE


def test_process_mask_crowded_region_and_empty_regions(cuda_device):
    """More than 254 detections in one 24x24 proto region (the region's list fills up and the binning hands the rest
    to the per-detection body, some of them already listed in another region) while most regions of the plane are
    touched by nobody (they load nothing)."""
    g = torch.Generator().manual_seed(21)
    n, mh, mw, ih, iw = 600, 128, 128, 512, 512
    protos = torch.randn((32, mh, mw), generator=g)
    coef = torch.randn((n, 32), generator=g) * 0.5
    c = torch.cat([200.0 + 40.0 * torch.rand((500, 2), generator=g),          # 500 boxes inside ~2 regions
                   torch.rand((100, 2), generator=g) * 500.0])
    wh = 10.0 + 30.0 * torch.rand((n, 2), generator=g)
    boxes = torch.cat([c - wh / 2, c + wh / 2], 1)
    dev = cuda_device
    for upsample in (False, True):
        ref = port.process_mask(protos, coef, boxes.clone(), (ih, iw), upsample=upsample)
        out = hm.process_mask(protos.to(dev), coef.to(dev), boxes.to(dev), (ih, iw), upsample=upsample)
        assert _agreement(out.cpu(), ref) >= AGREE
        counts = torch.tensor([n], dtype=torch.int32, device=dev)
        packed = hm.process_mask_packed(protos.to(dev)[None], coef.to(dev)[None], boxes.to(dev)[None], counts,
                                        (ih, iw), upsample=upsample)
        packed.check()
        assert torch.equal(packed.to_dense(), out.to(torch.uint8))


@pytest.mark.parametrize("M", [14, 56])
def test_paste_other_mask_sizes(cuda_device, M):
    """Mask sides other than the reference's 28 (the padded mask is staged in dynamic shared memory)."""
    g = torch.Generator().manual_seed(M)
    k, H, W = 40, 300, 260
    masks = torch.rand((k, 1, M, M), generator=g)
    boxes = _rand_boxes(g, k, H, W, 5, 120)
    ref = port.paste_masks_in_image(masks, boxes, (H, W), padding=1)
    out = hm.paste_masks_in_image(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=1).cpu()
    assert float((out - ref).abs().max()) < ATOL
    packed = hm.paste_masks_packed(masks.to(cuda_device), boxes.to(cuda_device), (H, W), padding=1)
    assert _agreement(packed.to_dense().cpu(), (ref[:, 0] > 0.5).to(torch.uint8)) >= AGREE


@pytest.mark.parametrize("ih,iw,mh,mw,seed", [(640, 640, 160, 160, 0), (320, 480, 80, 120, 1), (300, 500, 100, 125, 2)])
def test_process_mask_window_holds_every_set_pixel(cuda_device, ih, iw, mh, mw, seed):
    """The packed window is trimmed to the pixels that can exceed 0.5 (mask_common.cuh pm_trim): no pixel the oracle
    sets may fall outside it, including saturated masks (sigmoid == 1), boxes on the image border and non-integer
    scales, and the bits inside must be the oracle's."""
    g = torch.Generator().manual_seed(seed)
    k = 240
    protos = torch.randn((32, mh, mw), generator=g) * 3.0
    protos[0] += 40.0                                              # with coef[:, 0] = 1: saturated everywhere
    coef = torch.randn((k, 32), generator=g) * 0.5
    coef[::3, 0] = 1.0
    c = torch.rand((k, 2), generator=g) * torch.tensor([iw, ih])
    s = torch.rand((k, 2), generator=g) * 50 + 6
    boxes = torch.cat([c - s / 2, c + s / 2], 1)
    boxes[:8] = torch.tensor([[-5., -5., 20., 20.], [iw - 20., ih - 20., iw + 9., ih + 9.], [0., 0., 33., 17.],
                              [iw - 31., 0., iw, 12.], [0., ih - 9., 40., ih], [100.5, 60.25, 131.75, 91.0],
                              [10., 10., 14., 14.], [200., 100., 203., 260.]])
    ref = port.process_mask(protos, coef, boxes.clone(), (ih, iw), upsample=True)        # [k, ih, iw] 0/1
    counts = torch.tensor([k], dtype=torch.int32)
    pm = hm.process_mask_packed(protos[None].to(cuda_device), coef[None].to(cuda_device), boxes[None].to(cuda_device),
                                counts.to(cuda_device), (ih, iw), upsample=True)
    pm.check()
    geom = pm.geom.cpu()
    dense = pm.to_dense().cpu()
    assert _agreement(dense, ref.to(torch.uint8)) >= AGREE
    n_two_words = 0
    for i in range(k):
        x0, y0, w, h = geom[i].tolist()
        nz = torch.nonzero(ref[i])
        if len(nz):
            assert y0 <= int(nz[:, 0].min()) and int(nz[:, 0].max()) < y0 + h, (i, geom[i].tolist())
            assert x0 <= int(nz[:, 1].min()) and int(nz[:, 1].max()) < x0 + w, (i, geom[i].tolist())
        n_two_words += w > 32
    # saturated masks fill their window up to the trimmed edge: the trim is tight, not just safe
    sat = [i for i in range(9, k, 3) if geom[i, 2] > 0 and boxes[i, 0] > 8 and boxes[i, 2] < iw - 8]
    tight = sum(int(ref[i, :, geom[i, 0]].any()) + int(ref[i, :, geom[i, 0] + geom[i, 2] - 1].any()) for i in sat)
    assert tight >= 1.6 * len(sat)


# ------------------------------------------------------------------------------- fp16 prototypes / full-size masks
@pytest.mark.parametrize("upsample", [False, True])
def test_process_mask_fp16_prototypes_equal_fp32_path_on_rounded_inputs(cuda_device, upsample):
    """A half() model hands over fp16 prototypes (val_nuclei.py:115-116).  They are widened on load and every fp16
    value is an fp32 value, so the result must be BIT-identical to the fp32 path fed the rounded numbers."""
    g = torch.Generator().manual_seed(21)
    bs, md, mh, mw, ih, iw = 2, 150, 96, 120, 384, 480
    protos = torch.randn((bs, 32, mh, mw), generator=g).half()
    coef = (torch.randn((bs, md, 32), generator=g) * 0.5).to(cuda_device)
    boxes = torch.stack([_rand_boxes(g, md, ih, iw, 6, 90) for _ in range(bs)]).to(cuda_device)
    counts = torch.tensor([150, 97], dtype=torch.int32, device=cuda_device)
    a = hm.process_mask_packed(protos.to(cuda_device), coef, boxes, counts, (ih, iw), upsample=upsample)
    b = hm.process_mask_packed(protos.float().to(cuda_device), coef, boxes, counts, (ih, iw), upsample=upsample)
    a.check()
    assert torch.equal(a.geom, b.geom) and torch.equal(a.offsets, b.offsets) and torch.equal(a.bits, b.bits)
    assert int(a.offsets[-1]) > 0
    d16 = hm.process_mask_batch(protos.to(cuda_device), coef, boxes, counts, (ih, iw), upsample=upsample)
    d32 = hm.process_mask_batch(protos.float().to(cuda_device), coef, boxes, counts, (ih, iw), upsample=upsample)
    assert torch.equal(d16, d32)
    # and against the oracle on the rounded prototypes
    ref = port.process_mask(protos[1].float(), coef[1, :97].cpu(), boxes[1, :97].cpu().clone(), (ih, iw),
                            upsample=upsample)
    assert _agreement(d16[1, :97].cpu(), ref) >= AGREE


def test_process_mask_full_size_config2(cuda_device):
    """BASELINE configs[2] scale: 256 x 256 prototypes x ~2 650 nuclei-sized detections of a 1024-px tile (two tiles,
    one of them crowded into a corner), bit planes vs the oracle's process_mask(upsample) > 0.5."""
    g = torch.Generator().manual_seed(33)
    bs, md, mh, ih = 2, 2650, 256, 1024
    protos = torch.randn((bs, 32, mh, mh), generator=g)
    coef = torch.randn((bs, md, 32), generator=g) * 0.4
    boxes = torch.stack([_rand_boxes(g, md, ih, ih, 12, 36), _rand_boxes(g, md, 300, 300, 12, 36)])
    counts = torch.tensor([md, md - 650], dtype=torch.int32)
    pk = hm.process_mask_packed(protos.to(cuda_device), coef.to(cuda_device), boxes.to(cuda_device),
                                counts.to(cuda_device), (ih, ih), upsample=True)
    pk.check()
    geom, offs, bits = pk.geom.cpu(), pk.offsets.cpu(), pk.bits.cpu()
    agree = total = 0
    for t in range(bs):
        k = int(counts[t])
        for c0 in range(0, k, 250):                      # the oracle's dense canvases: 250 x 4 MB at a time
            c1 = min(c0 + 250, k)
            ref = port.process_mask(protos[t], coef[t, c0:c1], boxes[t, c0:c1].clone(), (ih, ih), upsample=True)
            sub = hm.PackedMasks(pk.geom[t * md + c0:t * md + c1], pk.offsets[t * md + c0:t * md + c1 + 1], pk.bits,
                                 ih, ih, pk.status)
            got = sub.to_dense().cpu()
            agree += int((got.float() == ref).sum())
            total += ref.numel()
        assert int((geom[t * md + k:(t + 1) * md, 2:] != 0).sum()) == 0      # slots beyond counts are empty
    assert agree / total >= AGREE, f"agreement {agree / total}"
    assert int(offs[-1]) <= bits.numel() and int(offs[-1]) > 30 * 2000


@pytest.mark.parametrize("form", ["packed_upsampled", "packed", "dense_upsampled", "dense"])
@pytest.mark.parametrize("mh,mw,ih,iw,md,lo,hi,half", [(160, 160, 640, 640, 900, 12, 36, False),
                                                       (256, 256, 1024, 1024, 2650, 12, 36, False),
                                                       (64, 80, 250, 333, 300, 4, 120, False),
                                                       (128, 128, 512, 512, 700, 10, 70, True)])
def test_packed_mask_kernel_paths_agree_bit_for_bit(cuda_device, mh, mw, ih, iw, md, lo, hi, half, form):
    """Every form runs regions -> patches -> upsample / pack, with the detections the patch path leaves out riding in
    the region launch.  The per-detection kernel must give the same output: for the bit-packed forms reached by
    hdy_process_mask_packed without a workspace (a) or without the windows (b), on the same geometry and offsets; for
    the dense forms by hdy_process_mask without a workspace -- including boxes too large for the patch path, crowded
    regions whose lists overflow, empty tiles and non-integer scales."""
    from hd_yolo_b200 import _lib, ops
    upsample = form.endswith("upsampled")
    g = torch.Generator().manual_seed(mh + md)
    bs = 3
    protos = torch.randn((bs, 32, mh, mw), generator=g)
    if half:
        protos = protos.half()
    coef = torch.randn((bs, md, 32), generator=g) * 0.5
    boxes = torch.stack([_rand_boxes(g, md, ih, iw, lo, hi),
                         _rand_boxes(g, md, ih // 6, iw // 6, lo, min(hi, 30)),        # > 254 boxes in one region
                         _rand_boxes(g, md, ih, iw, lo, hi)])
    boxes[0, 3] = torch.tensor([5.0, 7.0, iw - 20.0, ih * 0.6])                       # huge: per-detection kernel
    counts = torch.tensor([md, md - 7, 0], dtype=torch.int32)
    protos, coef, boxes, counts = (t.to(cuda_device) for t in (protos, coef, boxes, counts))
    lib = _lib.load()
    ws_bytes = lib.hdy_process_mask_workspace_bytes(bs, md)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=cuda_device)
    dtype = _lib.HDY_F16 if half else _lib.HDY_F32
    if form.startswith("dense"):
        oh, ow = (ih, iw) if upsample else (mh, mw)
        outs = []
        for workspace, nbytes in ((ws, ws_bytes), (None, 0)):
            out = torch.full((bs, md, oh, ow), -1.0, dtype=torch.float32, device=cuda_device)
            _lib.check(lib.hdy_process_mask(_lib.ptr(protos), dtype, _lib.ptr(coef), _lib.ptr(boxes), _lib.ptr(counts),
                                            bs, md, 32, mh, mw, ih, iw, int(upsample), _lib.ptr(out),
                                            _lib.ptr(workspace), nbytes, ops._stream()))
            outs.append(out)
        a, b = outs
        assert torch.equal(a, b), f"dense outputs differ in {int((a != b).sum())} pixels"
        assert float(a[0].sum()) > (50 if upsample else 3) * md
        return
    pk = hm.process_mask_packed(protos, coef, boxes, counts, (ih, iw), upsample=upsample)
    pk.check()
    words = int(pk.offsets[-1])
    for what, geom, workspace, nbytes in (("no workspace", pk.geom, None, 0), ("no geom", None, ws, ws_bytes)):
        bits = torch.full((max(words, 1),), -1, dtype=torch.int32, device=cuda_device)
        status = torch.zeros((1,), dtype=torch.int32, device=cuda_device)
        _lib.check(lib.hdy_process_mask_packed(_lib.ptr(protos), dtype, _lib.ptr(coef), _lib.ptr(boxes),
                                               _lib.ptr(counts), _lib.ptr(geom), _lib.ptr(pk.offsets), bs, md, 32, mh,
                                               mw, ih, iw, int(upsample), _lib.ptr(bits), words, _lib.ptr(status),
                                               _lib.ptr(workspace), nbytes, ops._stream()))
        assert int(status.item()) == 0, f"{what}: status {int(status.item())}"
        d = bits[:words]
        assert torch.equal(pk.bits, d), f"{what}: bits differ ({int((pk.bits != d).sum())} of {words} words)"
    assert words > (20 if upsample else 2) * (md - 7)


def test_mask_agreement_is_tight_inside_the_windows(cuda_device):
    """The 99.99 % bar of the north star is over whole canvases, where a nucleus covers < 1 % of the pixels.  The
    stricter statement: mismatching pixels are fewer than 1e-4 of the pixels the oracle SETS (differences can only
    come from values within an ulp of 0.5)."""
    g = torch.Generator().manual_seed(77)
    n, mh, ih = 600, 160, 640
    protos = torch.randn((32, mh, mh), generator=g)
    coef = torch.randn((n, 32), generator=g) * 0.5
    boxes = _rand_boxes(g, n, ih, ih, 10, 50)
    ref = port.process_mask(protos, coef, boxes.clone(), (ih, ih), upsample=True)
    out = hm.process_mask(protos.to(cuda_device), coef.to(cuda_device), boxes.to(cuda_device), (ih, ih), upsample=True).cpu()
    diff = int((out != ref).sum())
    assert float(ref.sum()) > 1e5 and diff <= 1e-4 * float(ref.sum()), f"{diff} of {int(ref.sum())} set pixels differ"
