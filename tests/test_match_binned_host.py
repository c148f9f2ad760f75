"""CPU tests of binned matching's host side: argument checks before any launch, PackedMasks.select / cat on CPU
tensors, and oracle/sparse_match.py against the dense oracles."""
import numpy as np
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import _lib, synth
from hd_yolo_b200.masks import PackedMasks
from oracle import mask_match, port, sparse_match


def _pack(dense: torch.Tensor) -> PackedMasks:
    """[K, H, W] 0/1 -> PackedMasks with tight windows, in numpy (the layout of include/hd_yolo_b200.h)."""
    K, H, W = dense.shape
    geom, offs, words = [], [0], []
    for m in dense.numpy().astype(bool):
        ys, xs = np.nonzero(m)
        if len(ys) == 0:
            geom.append([0, 0, 0, 0])
            offs.append(offs[-1])
            continue
        x0, y0, w, h = xs.min(), ys.min(), xs.max() - xs.min() + 1, ys.max() - ys.min() + 1
        wpr = (w + 31) // 32
        win = np.zeros((h, wpr * 32), bool)
        win[:, :w] = m[y0:y0 + h, x0:x0 + w]
        words.append(np.packbits(win.reshape(h, wpr, 32), axis=2, bitorder='little').reshape(-1).view('<u4'))
        geom.append([x0, y0, w, h])
        offs.append(offs[-1] + wpr * h)
    bits = np.concatenate(words).view(np.int32) if words else np.zeros(0, np.int32)
    return PackedMasks(torch.tensor(geom, dtype=torch.int32).reshape(-1, 4), torch.tensor(offs, dtype=torch.int64),
                       torch.from_numpy(bits.copy()), H, W, torch.zeros(1, dtype=torch.int32))


def _unpack(pm: PackedMasks) -> torch.Tensor:
    out = np.zeros((len(pm), pm.H, pm.W), np.uint8)
    bits = pm.bits.numpy().view('<u4')
    for i, (x0, y0, w, h) in enumerate(pm.geom.tolist()):
        if w <= 0 or h <= 0:
            continue
        wpr = (w + 31) // 32
        o = int(pm.offsets[i])
        rows = np.unpackbits(bits[o:o + wpr * h].view(np.uint8), bitorder='little').reshape(h, wpr * 32)[:, :w]
        out[i, y0:y0 + h, x0:x0 + w] = rows
    return torch.from_numpy(out)


def _ellipses(n, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.rand((n, 2), generator=g) * torch.tensor([W, H])
    r = 2.0 + 9.0 * torch.rand((n, 2), generator=g)
    return synth.ellipse_masks(c, r, H, W).to(torch.uint8), c, r


def test_binned_argument_checks():
    out = {'boxes': torch.zeros(2, 4), 'scores': torch.zeros(2), 'labels': torch.zeros(2)}
    tgt = {'boxes': torch.zeros(2, 4), 'labels': torch.zeros(2)}
    for bad in (0.0, -1.0, float('nan'), 1e-60):                   # 1e-60 is 0 in fp32
        with pytest.raises(hdy.HdyError, match="iou_min > 0"):
            hdy.match_predictions(out, tgt, bad, binned=True)
        with pytest.raises(hdy.HdyError, match="iou_min > 0"):
            hdy.match_predictions(out, tgt, bad, iou_type='masks', binned=True)
    with pytest.raises(hdy.HdyError, match="CUDA"):                 # CPU tensors: no fallback
        hdy.match_predictions(out, tgt, 0.5, binned=True)
    lib = _lib.load()
    args = (None, None, 1, None, 1, 0.0, 0.0, 1.0, 4, 4, None, None)
    assert lib.hdy_match_boxes_binned(*args, 0.0, None, None, None, None, None) == -1
    assert b"iou_min" in lib.hdy_last_error()
    assert lib.hdy_match_boxes_binned(None, None, 1, None, 1, 0.0, 0.0, 0.0, 4, 4, None, None, 0.5, None, None, None,
                                      None, None) == -1
    assert lib.hdy_match_bin_stats(None, None, 4, None, None) == -1
    assert lib.hdy_match_bin_cells(None, 0, 0, None, None) == -1
    assert lib.hdy_match_mask_exact_list(*([None] * 11), 1, 0.0, *([None] * 7)) == -1


def test_select_and_cat_round_trip():
    dense, _, _ = _ellipses(40, 60, 90, seed=1)
    dense[5] = 0                                                   # an empty mask
    pm = _pack(dense)
    assert torch.equal(_unpack(pm), dense)
    rows = torch.tensor([7, 3, 5, 3, 39, 0])
    sel = pm.select(rows)
    assert sel.bits is pm.bits and len(sel) == len(rows) and int(sel.offsets[-1]) == int(pm.offsets[-1])
    assert torch.equal(_unpack(sel), dense[rows])
    assert len(pm.select([])) == 0
    # two region canvases placed on one slide canvas
    other, _, _ = _ellipses(25, 50, 70, seed=2)
    po = _pack(other)
    cat = PackedMasks.cat([pm, po], [(10, 4), (100, 30)], (90, 200))
    assert (cat.H, cat.W) == (90, 200) and len(cat) == 65
    want = torch.zeros((65, 90, 200), dtype=torch.uint8)
    want[:40, 4:64, 10:100] = dense
    want[40:, 30:80, 100:170] = other
    assert torch.equal(_unpack(cat), want)
    assert torch.equal(cat.geom[5], torch.zeros(4, dtype=torch.int32))            # empty stays empty
    assert torch.equal(_unpack(cat.select(torch.arange(40, 65))), want[40:])
    with pytest.raises(hdy.HdyError):
        PackedMasks.cat([pm, po], [(10, 4), (140, 30)], (90, 200))                 # does not fit the canvas
    with pytest.raises(hdy.HdyError):
        PackedMasks.cat([pm], [(0, 0), (1, 1)], (90, 200))


def _box_case(k, g, seed, size=300):
    gen = torch.Generator().manual_seed(seed)
    c = torch.rand((g, 2), generator=gen) * size
    r = 3 + 12 * torch.rand((g, 2), generator=gen)
    gt = torch.cat([c - r, c + r], 1)
    m = min(k, g)
    pc = torch.cat([gt[:m] + torch.randn((m, 4), generator=gen), gt[:k - m] * 0.7 + 20])
    pc[3] = float('nan')
    pc[4, 2] = float('inf')
    pc[6] = torch.tensor([50., 50., 50., 80.])
    gt[2] = gt[9]
    out = {'boxes': pc, 'scores': (torch.rand(k, generator=gen) * 32).round() / 32,
           'labels': torch.randint(0, 4, (k,), generator=gen)}
    return out, {'boxes': gt, 'labels': torch.randint(1, 4, (g,), generator=gen)}


@pytest.mark.parametrize("iou_min", [0.5, 0.95, 1e-6])
def test_sparse_oracle_equals_dense(iou_min):
    out, tgt = _box_case(400, 350, seed=3)
    want = port.apmeter_match(out, tgt, iou_min)
    got = sparse_match.apmeter_match_sparse(out, tgt, iou_min)
    assert len(want[4]) > 0
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    pm, c, r = _ellipses(120, 96, 128, seed=4)
    gm = synth.ellipse_masks(c + 0.8, r * 1.05, 96, 128)
    gm[7] = False
    gm[10:15] = pm[10:15].bool()                                  # identical masks: IoU 1
    mo = {'boxes': torch.zeros(120, 4), 'scores': torch.rand(120), 'labels': torch.ones(120, dtype=torch.int64),
          'masks': pm}
    mt = {'boxes': torch.zeros(120, 4), 'labels': torch.ones(120, dtype=torch.int64), 'masks': gm}
    want = mask_match.apmeter_match(mo, mt, iou_min)
    assert len(want[4]) > 0
    for masks in ((pm, gm), (_pack(pm), _pack(gm.to(torch.uint8)))):        # dense and packed inputs
        got = sparse_match.apmeter_match_sparse({**mo, 'masks': masks[0]}, {**mt, 'masks': masks[1]}, iou_min,
                                                'masks')
        for a, b in zip(got, want):
            assert torch.equal(a, b)


def _orderable(f: float) -> int:
    u = int(np.array(f, dtype=np.float32).view(np.uint32))
    return u | 0x80000000 if u < 0x80000000 else (~u) & 0xffffffff


@pytest.mark.parametrize("lo,hi,n", [(0.0, 1024.0, 3000), (-3e38, 3e38, 1), (-1e35, 1e35, 1001), (1e30, 3e38, 5),
                                     (-5.0, 5.0, 1)])
def test_grid_is_bounded_for_any_finite_extent(lo, hi, n):
    """The cell picker returns a grid of at most 2 n + 1024 cells with a normal fp32 1 / cell for every finite
    ground-truth extent, flat ones (zero height) included."""
    from hd_yolo_b200.metrics import _pick_grid
    for y1 in (hi, lo):
        stats = [_orderable(lo), _orderable(lo), _orderable(hi), _orderable(y1), n, 16 * 20 * n]
        ox, oy, inv, nx, ny = _pick_grid(stats)
        assert 1 <= nx * ny <= 2 * n + 1024
        assert np.isfinite(np.float32(inv)) and np.float32(inv) >= np.finfo(np.float32).tiny
        assert np.isfinite(np.float32(ox)) and np.isfinite(np.float32(oy))


def test_mask_canvas_mismatch_is_rejected_on_host():
    """The canvas check match_predictions(iou_type='masks') runs before any launch (on the device, a CPU tensor is
    refused before it; tests/test_gpu_match_binned.py checks the binned call itself)."""
    from hd_yolo_b200.metrics import _check_mask_inputs
    a, _, _ = _ellipses(4, 40, 50, seed=6)
    b, _, _ = _ellipses(3, 40, 60, seed=7)
    with pytest.raises(hdy.HdyError, match="canvas"):
        _check_mask_inputs({'masks': a}, {'masks': b}, 4, 3, 0.5)
    _check_mask_inputs({'masks': a}, {'masks': a[:3]}, 4, 3, 0.5)
