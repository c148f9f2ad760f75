"""bench.py --dump-outputs on the GPU: what it writes for the last timed step is what the public API returns for the same
seeded inputs -- detections in the caller's order, and the masks of exactly those detections (tiles: mask index
tile * max_det + slot, proto and paste; slide: the survivor's slide row)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu
QUIET = ["--no-sub", "--no-cpu-baseline", "--no-torch-cuda", "--no-e2e"]
N_MASKS = 64       # masks compared pixel for pixel (each unpacked onto a whole canvas)


def _dump(tmp_path, *args):
    out = str(tmp_path / "dump")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", *QUIET, *args,
                        "--dump-outputs", out], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    d = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    return d


def _check_masks(d, pm, rows):
    """The dump's first windows / pixels against PackedMasks.to_dense() of the same mask rows."""
    from hd_yolo_b200.masks import PackedMasks
    rows = rows[:N_MASKS]
    sub = PackedMasks(pm.geom[rows].contiguous(), torch.cat([pm.offsets[rows], pm.offsets[-1:]]), pm.bits, pm.H, pm.W,
                      pm.status)
    dense = sub.to_dense().cpu().numpy()
    win, pix, o = d["mask_windows"], d["mask_pixels"], 0
    assert np.array_equal(win[:len(rows)], sub.geom.cpu().numpy().astype(np.float32))
    for i, (x0, y0, w, h) in enumerate(win.astype(np.int64)):
        if i == len(rows):
            break
        want = dense[i, y0:y0 + h, x0:x0 + w]
        assert np.array_equal(pix[o:o + w * h], want.reshape(-1).astype(np.float32)), i
        assert int(dense[i].sum()) == int(want.sum())          # nothing outside the window
        o += w * h
    assert pix[:o].sum() > 0


@pytest.mark.parametrize("masks", ["proto", "paste"])
def test_tiles_dump_is_the_last_steps_output(cuda_device, tmp_path, masks):
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import synth
    d = _dump(tmp_path, "--workload", "tiles640", "--masks", masks)
    # bench.py: tiles640 = 64 tiles of 640 px, ~1 000 candidates, cap 2048; --steps 1 replays the graph of input batch 0
    bs, tile, nc, nm = 64, 640, 4, 32
    extra = nm if masks == "proto" else 0
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=nc, no=5 + nc + extra)
    dets = synth.nuclei_logits(bs, tile, nc, 1000, seed=0, conf=0.25, extra=extra, generator_device="cuda")
    out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, 1000, cap=2048)
    lst = out.to_list()
    if masks == "proto":
        g = torch.Generator(device="cuda").manual_seed(77)
        protos = torch.randn((bs, nm, tile // 4, tile // 4), generator=g, device=cuda_device)
        pm = hdy.process_mask_packed(protos, out.extra, out.boxes, out.counts, (tile, tile), upsample=True)
    else:
        g = torch.Generator(device="cuda").manual_seed(78)
        logits = torch.randn((bs * out.max_det, 2, 28, 28), generator=g, device=cuda_device)
        live = torch.arange(out.max_det, device=cuda_device)[None, :] < out.counts[:, None]
        mi = torch.tensor([-1, 0, 0, 1, 1], dtype=torch.int32, device=cuda_device)
        ch = torch.where(live, mi[torch.where(live, out.labels, torch.zeros_like(out.labels)).clamp(min=0)],
                         torch.full_like(out.labels, -1, dtype=torch.int32)).reshape(-1)
        pm = hdy.paste_masks_packed(logits, out.boxes.reshape(-1, 4), (tile, tile), padding=1, channel=ch,
                                    apply_sigmoid=True)
    pm.check()
    assert np.array_equal(d["counts"], out.counts.cpu().numpy())
    assert np.array_equal(d["sample"], np.arange(sum(len(a['boxes']) for a in lst)))
    for k in ("boxes", "scores", "labels"):
        assert np.array_equal(d[k], torch.cat([a[k] for a in lst]).cpu().numpy().astype(d[k].dtype)), k
    slots = torch.cat([i * out.max_det + torch.arange(len(a['boxes']), device=cuda_device) for i, a in enumerate(lst)])
    _check_masks(d, pm, slots)


def test_slide_dump_is_the_last_steps_output(cuda_device, tmp_path):
    from hd_yolo_b200 import synth
    from hd_yolo_b200.pipeline import SlidePostprocessor
    import hd_yolo_b200 as hdy
    S = 3000
    d = _dump(tmp_path, "--slide-size", str(S))
    # bench.py: slide = 1024-px tiles, 64 px overlap, batches of 148, cap 3072, 32 prototypes; every tile's inputs are
    # seeded by its global index
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=5 + 4 + 32)
    post = SlidePostprocessor(spec, (S, S), (1024, 1024), 64, 0.25, 0.45, 3072, cap=3072, batch=148, device=cuda_device)
    n = int(post.rois.shape[0])
    dets = synth.slide_tile_logits(post.rois, 1024, 4, seed=1, conf=0.25, extra=32, device=cuda_device)
    protos = synth.slide_tile_protos(n, 1024, seed=1, device=cuda_device)
    r = post.run(lambda a, b: dets, ordered=True, proto_provider=lambda a, b: protos, mask_words_per_row=40.0)
    r['masks'].check()
    assert np.array_equal(d["counts"], [int(r['n']), int(r['boxes'].shape[0])])
    assert np.array_equal(d["sample"], np.arange(int(r['boxes'].shape[0])))
    for k in ("boxes", "scores", "labels"):
        assert np.array_equal(d[k], r[k].cpu().numpy().astype(d[k].dtype)), k
    _check_masks(d, r['masks'], r['index'] - int(r['base']))
