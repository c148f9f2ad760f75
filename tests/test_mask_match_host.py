"""CPU tests of matching by mask IoU: the oracle's mask_iou on hand-computable cases, and the argument checks the
C-ABI entry points of the mask path run on the host before anything is launched."""
import ctypes as C

import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import _lib
from oracle import mask_match


def test_mask_iou_known_answers():
    a = torch.zeros((4, 5, 6), dtype=torch.bool)
    b = torch.zeros((3, 5, 6))
    a[0, 0, 0] = True                       # 1 pixel
    a[1, :2, :2] = True                     # 2 x 2 block
    a[2, :, :] = True                       # the whole 30-pixel canvas
    b[0, 0, :2] = 0.7                       # 2 pixels
    b[1, :, :] = 0.5                        # exactly 0.5 is not set: empty
    b[2, 1:3, 1:4] = 1.0                    # 2 x 3 block
    iou = mask_match.mask_iou(a, b)
    assert iou.dtype == torch.float32 and iou.shape == (4, 3)
    inter = torch.tensor([[1, 0, 0], [2, 0, 1], [2, 0, 6], [0, 0, 0]])
    union = torch.tensor([[2, 1, 7], [4, 4, 9], [30, 30, 30], [2, 0, 6]])
    want = inter.float() / union.float()
    assert torch.equal(torch.isnan(iou), torch.isnan(want))
    assert torch.equal(torch.nan_to_num(iou, nan=-1.0), torch.nan_to_num(want, nan=-1.0))
    # [n, 1, H, W] and integer masks (set iff nonzero) give the same numbers
    assert torch.equal(torch.nan_to_num(mask_match.mask_iou(a[:, None].to(torch.uint8) * 7, (b > 0.5)[:, None]), nan=-1.0),
                       torch.nan_to_num(want, nan=-1.0))
    # the division is one fp32 rounding of exact integers: 1 / 3 in fp32
    c = torch.zeros((1, 1, 3), dtype=torch.bool)
    d = c.clone()
    c[0, 0, :2] = True
    d[0, 0, 1:] = True
    assert mask_match.mask_iou(c, d).item() == float(torch.tensor(1.0) / torch.tensor(3.0))
    assert mask_match.mask_iou(a[:0], b).shape == (0, 3) and mask_match.mask_iou(a, b[:0]).shape == (4, 0)


def test_apmeter_match_masks_known_answer():
    masks = torch.zeros((3, 8, 8), dtype=torch.bool)
    masks[0, :4, :4] = True
    masks[1, 4:, 4:] = True
    masks[2, :4, :2] = True                 # half of mask 0
    out = {'boxes': torch.zeros((3, 4)), 'scores': torch.tensor([0.2, 0.9, 0.5]), 'labels': torch.tensor([1, 2, 3]),
           'masks': masks}
    tgt = {'boxes': torch.zeros((2, 4)), 'labels': torch.tensor([1, 2]), 'masks': masks[:2]}
    s, l, p, t, i = mask_match.apmeter_match(out, tgt, 0.5)
    assert torch.equal(s, torch.tensor([0.9, 0.5, 0.2])) and torch.equal(l, torch.tensor([2, 3, 1]))
    # ranks: row 1 -> 0, row 2 -> 1, row 0 -> 2; pairs (0, 1) iou 1, (2, 0) iou 1, (1, 0) iou 0.5
    assert torch.equal(p, torch.tensor([0, 2, 1])) and torch.equal(t, torch.tensor([1, 0, 0]))
    assert torch.equal(i, torch.tensor([1.0, 1.0, 0.5]))
    # the default keeps the box path
    st = mask_match.APMeterState()
    st.add({k: v for k, v in out.items() if k != 'masks'}, {k: v for k, v in tgt.items() if k != 'masks'},
           iou_type='masks')
    assert st.n_match == 0 and st.n_pred == 3           # zero-area boxes: 0/0, no match


def _p(v):
    return C.c_void_p(v)


def test_mask_entry_points_check_arguments_on_host():
    lib = _lib.load()
    fake = _p(4096)                                     # never dereferenced: every call below fails its checks first
    # hdy_pack_masks_geometry(masks, dtype, K, H, W, geom, offsets, stream)
    assert lib.hdy_pack_masks_geometry(fake, _lib.HDY_F32, -1, 8, 8, fake, fake, None) == -1
    assert lib.hdy_pack_masks_geometry(fake, _lib.HDY_F32, 4, 0, 8, fake, fake, None) == -1
    assert lib.hdy_pack_masks_geometry(fake, 7, 4, 8, 8, fake, fake, None) == -1
    assert b"dtype" in lib.hdy_last_error()
    assert lib.hdy_pack_masks_geometry(None, _lib.HDY_U8, 4, 8, 8, fake, fake, None) == -1
    assert lib.hdy_pack_masks_geometry(fake, _lib.HDY_U8, 4, 8, 8, fake, None, None) == -1
    assert lib.hdy_pack_masks_geometry(fake, _lib.HDY_U8, 4, 8, 8, _p(4100), fake, None) == -1
    assert b"aligned" in lib.hdy_last_error()
    assert lib.hdy_pack_masks_geometry(fake, _lib.HDY_U8, 4, 65536, 65536, fake, fake, None) == -1
    # hdy_pack_masks(masks, dtype, K, H, W, geom, offsets, bits, capacity_words, status, stream)
    assert lib.hdy_pack_masks(fake, _lib.HDY_F16, -2, 8, 8, fake, fake, fake, 16, fake, None) == -1
    assert lib.hdy_pack_masks(fake, _lib.HDY_F16, 4, 8, 8, fake, fake, None, 16, fake, None) == -1
    assert lib.hdy_pack_masks(fake, _lib.HDY_F16, 4, 8, 8, fake, fake, fake, -1, fake, None) == -1
    assert lib.hdy_pack_masks(fake, _lib.HDY_F16, 4, 8, 8, _p(4104), fake, fake, 16, fake, None) == -1
    # hdy_mask_areas(geom, offsets, bits, K, areas, stream)
    assert lib.hdy_mask_areas(fake, fake, fake, -1, fake, None) == -1
    assert lib.hdy_mask_areas(fake, None, fake, 3, fake, None) == -1
    assert lib.hdy_mask_areas(_p(4104), fake, fake, 3, fake, None) == -1
    # hdy_match_mask_pairs(pred geom/offsets/bits/areas/order, P, gt geom/offsets/bits/areas, G, iou_min, cand_cap,
    #                      cand, cap, pair_keys, counts, status, stream)

    def match(P=10, G=10, iou_min=0.5, cand_cap=16, cap=16, pred_geom=fake, gt_bits=fake):
        return lib.hdy_match_mask_pairs(pred_geom, fake, fake, fake, None, P, fake, fake, gt_bits, fake, G, iou_min,
                                        cand_cap, fake, cap, fake, fake, fake, None)
    assert match(P=-1) == -1 and match(G=-3) == -1
    assert match(cand_cap=0) == -1 and match(cap=0) == -1
    assert match(iou_min=0.0) == -1 and b"iou_min" in lib.hdy_last_error()
    assert match(iou_min=-0.5) == -1 and match(iou_min=float('nan')) == -1
    assert match(P=70000, G=70000) == -1 and b"32 bits" in lib.hdy_last_error()
    assert match(gt_bits=None) == -1 and b"NULL" in lib.hdy_last_error()
    assert match(pred_geom=_p(4100)) == -1 and b"aligned" in lib.hdy_last_error()
    assert match(P=0) == 0 and match(G=0) == 0             # nothing to do: nothing is launched


def test_mask_matching_rejects_cpu_tensors_and_bad_arguments():
    out = {'boxes': torch.zeros(2, 4), 'scores': torch.zeros(2), 'labels': torch.zeros(2), 'masks': torch.zeros(2, 8, 8)}
    tgt = {'boxes': torch.zeros(2, 4), 'labels': torch.zeros(2), 'masks': torch.zeros(2, 8, 8)}
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, tgt, 0.5, iou_type='masks')
    with pytest.raises(hdy.HdyError):
        hdy.match_predictions(out, tgt, 0.5, iou_type='segm')
    with pytest.raises(hdy.HdyError):
        hdy.PackedMasks.from_dense(torch.zeros(2, 8, 8))
