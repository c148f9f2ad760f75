"""GPU tests of the scan and stream-compaction primitives, driven through the public calls that use them, at sizes
that cross every tile and chunk boundary: the radix sort (histogram scan), the ordered survivor selection, the seam
selection of the multi-GPU merge and the word offsets of the packed masks."""
import numpy as np
import pytest
import torch

from hd_yolo_b200 import slide as hs
from hd_yolo_b200._lib import HDY_SEAM_HDR_WORDS, HDY_SEAM_FAR_WORDS, HDY_SEAM_ROW_WORDS, ptr
from hd_yolo_b200.ops import _call, _stream

pytestmark = pytest.mark.gpu


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


@pytest.mark.parametrize("first_byte,n_bytes", [(0, 8), (4, 4)])
def test_sort_keys_large(cuda_device, first_byte, n_bytes):
    n = 5_000_011
    g = torch.Generator().manual_seed(17 + first_byte)
    lo = torch.randint(0, 2 ** 32, (n,), generator=g, dtype=torch.int64)
    hi = torch.randint(-2 ** 31, 2 ** 31, (n,), generator=g, dtype=torch.int64)
    hi[::3] = hi[1]                                   # many equal upper halves: ties the partial sort must keep stable
    hi[1::7] = torch.randint(-4, 4, (len(hi[1::7]),), generator=g)
    k = (hi << 32) | lo
    out = _u64(hs.sort_keys(k.to(cuda_device), first_byte=first_byte, n_bytes=n_bytes))
    ku = k.numpy().view(np.uint64)
    if n_bytes == 8:
        ref = np.sort(ku, kind="stable")
    else:
        ref = ku[np.argsort(ku >> np.uint64(32), kind="stable")]
    assert np.array_equal(out, ref)


@pytest.mark.parametrize("n", [1, 255, 1025, 4096 * 1024 + 7])
def test_kept_in_order(cuda_device, n):
    g = torch.Generator().manual_seed(n)
    state = torch.randint(1, 4, (n,), generator=g, dtype=torch.uint8)          # KEPT / SUPPRESSED / DROPPED
    scores = (torch.randint(16, 64, (n,), generator=g) / 64.0).float()         # coarse: many ties
    boxes = torch.rand((n, 4), generator=g) * 100.0
    idx, ob, os_, _ = hs._kept_in_order(state.to(cuda_device), boxes.to(cuda_device), scores.to(cuda_device), None, n)
    kept = torch.nonzero(state == hs.STATE_KEPT).flatten()
    order = torch.sort(scores[kept], descending=True, stable=True).indices   # ties: the lower row first
    ref = kept[order]
    assert torch.equal(idx.cpu(), ref)
    assert torch.equal(ob.cpu(), boxes[ref]) and torch.equal(os_.cpu(), scores[ref])


@pytest.mark.parametrize("cap_frac", [2.0, 0.5])
def test_seam_select(cuda_device, cap_frac):
    world, rank, far_cap = 5, 2, 2
    n = 3_000_017
    g = torch.Generator().manual_seed(3)
    xy = torch.rand((n, 2), generator=g) * 20000.0
    wh = torch.rand((n, 2), generator=g) * 40.0 + 1.0
    boxes = torch.cat([xy, xy + wh], 1)
    scores = torch.rand((n,), generator=g)
    rows = [700_000, 0, n, 1_234_567, 2]               # rank 1 has no rows: its rectangle is not tested
    rects = [[0.0, 0.0, 3000.0, 20000.0], [5000.0, 5000.0, 15000.0, 15000.0], [0.0, 0.0, 20000.0, 20000.0],
             [10000.0, 19000.0, 20000.0, 30000.0], [12000.5, 7000.25, 12000.5, 7000.25]]
    hb = HDY_SEAM_HDR_WORDS + far_cap * HDY_SEAM_FAR_WORDS
    summ = torch.zeros((world, hb), dtype=torch.int32)
    for q in range(world):
        summ[q, 0:4] = torch.tensor(rects[q], dtype=torch.float32).view(torch.int32)
        summ[q, 6:8] = torch.tensor([rows[q]], dtype=torch.int64).view(torch.int32)
    ref = torch.zeros((n,), dtype=torch.bool)
    for q in range(world):
        if q == rank or rows[q] == 0:
            continue
        x1, y1, x2, y2 = torch.tensor(rects[q], dtype=torch.float32)
        ref |= (boxes[:, 2] >= x1) & (boxes[:, 0] <= x2) & (boxes[:, 3] >= y1) & (boxes[:, 1] <= y2)
    sel_ref = torch.nonzero(ref).flatten()
    m = len(sel_ref)
    assert 10_000 < m < n // 2
    seam_cap = int(m * cap_frac)
    keep = min(m, seam_cap)
    dev = cuda_device
    sel = torch.full((seam_cap,), -1, dtype=torch.int32, device=dev)
    block = torch.full((HDY_SEAM_HDR_WORDS + seam_cap * HDY_SEAM_ROW_WORDS,), -1, dtype=torch.int32, device=dev)
    scratch = torch.empty((4097,), dtype=torch.int32, device=dev)
    db, ds, dsumm = boxes.to(dev), scores.to(dev), summ.to(dev)
    _call("hdy_seam_select", ptr(db), ptr(ds), n, ptr(dsumm), world, rank, far_cap, seam_cap, ptr(sel), ptr(block),
          ptr(scratch), _stream())
    block, sel = block.cpu(), sel.cpu()
    assert int(block[0]) == m and torch.equal(block[1:HDY_SEAM_HDR_WORDS], torch.zeros(HDY_SEAM_HDR_WORDS - 1,
                                                                                       dtype=torch.int32))
    assert torch.equal(sel[:keep].long(), sel_ref[:keep])
    pay = block[HDY_SEAM_HDR_WORDS:].view(seam_cap, HDY_SEAM_ROW_WORDS)[:keep]
    r = sel_ref[:keep]
    assert torch.equal(pay[:, 0:4], boxes[r].view(torch.int32))
    assert torch.equal(pay[:, 4], scores[r].view(torch.int32))
    assert torch.equal(pay[:, 5].long(), r + sum(rows[:rank]))
    assert bool((block[HDY_SEAM_HDR_WORDS + keep * HDY_SEAM_ROW_WORDS:] == -1).all())


def _check_offsets(geom, offsets):
    g = geom.cpu().long()
    words = ((g[:, 2] + 31) >> 5) * g[:, 3]
    ref = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(words, 0)])
    assert torch.equal(offsets.cpu(), ref)


@pytest.mark.parametrize("K", [1, 1024, 1025, 4096 * 1024 + 3])
def test_paste_geometry_offsets(cuda_device, K):
    g = torch.Generator().manual_seed(K)
    xy = torch.rand((K, 2), generator=g) * 1100.0 - 50.0
    boxes = torch.cat([xy, xy + torch.rand((K, 2), generator=g) * 90.0], 1).to(cuda_device)
    channel = torch.randint(-1, 3, (K,), generator=g, dtype=torch.int32).to(cuda_device)
    geom = torch.empty((K, 4), dtype=torch.int32, device=cuda_device)
    offsets = torch.full((K + 1,), -1, dtype=torch.int64, device=cuda_device)
    _call("hdy_paste_geometry", ptr(boxes), ptr(channel), K, 28, 1, 1024, 1024, ptr(geom), ptr(offsets), _stream())
    assert bool((geom[channel < 0] == 0).all()) and bool((geom[channel >= 0, 2] > 0).any())
    _check_offsets(geom, offsets)


@pytest.mark.parametrize("bs,max_det,slide_form", [(1, 700, False), (3, 1000, True), (1100, 4000, False),
                                                   (1100, 4000, True)])
def test_process_mask_geometry_offsets(cuda_device, bs, max_det, slide_form):
    g = torch.Generator().manual_seed(bs + max_det)
    K = bs * max_det
    counts = torch.randint(0, max_det + 1, (bs,), generator=g, dtype=torch.int32)
    xy = torch.rand((K, 2), generator=g) * 340.0 - 10.0
    boxes = torch.cat([xy, xy + torch.rand((K, 2), generator=g) * 60.0], 1)
    row_state = tile_offsets = None
    if slide_form:
        tile_offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(counts.long(), 0)]).to(cuda_device)
        row_state = torch.randint(1, 4, (int(counts.sum()),), generator=g, dtype=torch.uint8).to(cuda_device)
    dev = cuda_device
    db, dc = boxes.to(dev), counts.to(dev)
    geom = torch.full((K, 4), -1, dtype=torch.int32, device=dev)
    offsets = torch.full((K + 1,), -1, dtype=torch.int64, device=dev)
    _call("hdy_process_mask_geometry", ptr(db), ptr(dc), bs, max_det, 80, 80, 320, 320, 1, ptr(row_state),
          ptr(tile_offsets), ptr(geom), ptr(offsets), _stream())
    live = torch.arange(max_det)[None, :] < counts[:, None].long()
    if slide_form:
        kept = torch.zeros((bs, max_det), dtype=torch.bool)
        kept[live] = row_state.cpu() == hs.STATE_KEPT
        live = kept
    gc = geom.cpu().view(bs, max_det, 4)
    assert bool((gc[~live] == 0).all()) and bool((gc[live][:, 2] > 0).any())
    _check_offsets(geom, offsets)
