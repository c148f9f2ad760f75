"""GPU parity tests of the sharded whole-slide merge: W ranks emulated on one device through the real C-ABI kernels
(hdy_seam_* / hdy_merge_rounds / hdy_merge_finish) vs torchvision's dense NMS on the slide-wide
concatenation (what Ensemble.merge computes, metayolo/models/yolo.py:189-195) and vs the single-device merge."""
import os
import sys

import pytest
import torch
import torchvision

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from slide_synth import banded_detections  # noqa: E402

pytestmark = pytest.mark.gpu
CONF, IOU = 0.25, 0.45


def _ref_states(parts):
    boxes = torch.cat([p[0] for p in parts])
    scores = torch.cat([p[1] for p in parts])
    keep = scores > CONF
    idx = torch.nonzero(keep).flatten()
    kept = idx[torchvision.ops.nms(boxes[idx], scores[idx], IOU)]
    st = torch.full((len(scores),), 2, dtype=torch.uint8)
    st[~keep] = 3
    st[kept] = 1
    return st


@pytest.mark.parametrize("world,n", [(2, 2000), (4, 6000), (8, 12000)])
def test_emulated_ranks_on_device_match_dense_nms(cuda_device, world, n):
    from hd_yolo_b200 import dist as hdist
    import hd_yolo_b200 as hdy

    parts = banded_detections(world, seed=100 + world, n_nuclei=n, width=3000.0)
    ref = _ref_states(parts)
    dparts = [(b.to(cuda_device), s.to(cuda_device)) for b, s in parts]
    got = torch.cat([g.cpu() for g in hdist.merge_emulated(dparts, CONF, IOU)])
    assert torch.equal(got, ref)
    # single-device merge on the concatenation gives the same verdicts
    allb = torch.cat([p[0] for p in dparts])
    alls = torch.cat([p[1] for p in dparts])
    one = hdy.merge_nms(allb, alls, CONF, IOU).cpu()
    assert torch.equal(one, ref)


def test_emulated_ranks_with_empty_rank(cuda_device):
    from hd_yolo_b200 import dist as hdist

    parts = banded_detections(3, seed=5, n_nuclei=1500)
    parts[1] = (torch.zeros((0, 4)), torch.zeros((0,)))
    ref = _ref_states(parts)
    dparts = [(b.to(cuda_device), s.to(cuda_device)) for b, s in parts]
    got = torch.cat([g.cpu() for g in hdist.merge_emulated(dparts, CONF, IOU)])
    assert torch.equal(got, ref)
