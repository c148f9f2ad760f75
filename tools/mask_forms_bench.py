"""One process_mask call of every output form, timed with CUDA events after warm-up, on tiles of the synthetic nuclei
field (synth.slide_tile_logits -> detect_postprocess, synth.slide_tile_protos):

  dense_upsampled  masks.process_mask_batch(upsample=True):  [bs, max_det, ih, iw] fp32 (4 * ih * iw bytes per slot)
  dense            masks.process_mask_batch(upsample=False): [bs, max_det, mh, mw] fp32
  packed           masks.process_mask_packed(upsample=False): bit planes at prototype resolution
  packed_upsampled masks.process_mask_packed(upsample=True):  the throughput form (slide pipeline, bench.py)

Each figure is the median over `rounds` rounds of the mean of `reps` back-to-back calls; the forms take turns inside
every round.  The dense times include the memset of the whole output.  The prototypes of 8 tiles of 640 px are 26 MB
and stay in L2 across calls.

usage: python tools/mask_forms_bench.py [--tiles 8] [--tile 640] [--max-det 1000] [--reps 20] [--rounds 5]
       (prints one JSON line)"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hd_yolo_b200 as hdy
from hd_yolo_b200 import masks as hm
from hd_yolo_b200 import synth
from hd_yolo_b200.slide import sliding_window_scanner

ap = argparse.ArgumentParser()
ap.add_argument("--tiles", type=int, default=8)
ap.add_argument("--tile", type=int, default=640)
ap.add_argument("--max-det", type=int, default=1000)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=5)
a = ap.parse_args()

dev = torch.device("cuda:0")
bs, tile, md, nm = a.tiles, a.tile, a.max_det, 32
rois = sliding_window_scanner((100000, 100000), (tile, tile), 64)[1000:1000 + bs]
spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=9 + nm)
dets = synth.slide_tile_logits(rois, tile, 4, seed=1, first_tile=1000, extra=nm, device=dev)
out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, md, cap=2048)
del dets
protos = synth.slide_tile_protos(bs, tile, seed=1, first_tile=1000, device=dev)
shape = (tile, tile)

forms = {
    "dense_upsampled": lambda: hm.process_mask_batch(protos, out.extra, out.boxes, out.counts, shape, upsample=True),
    "dense": lambda: hm.process_mask_batch(protos, out.extra, out.boxes, out.counts, shape, upsample=False),
    "packed": lambda: hm.process_mask_packed(protos, out.extra, out.boxes, out.counts, shape, upsample=False),
    "packed_upsampled": lambda: hm.process_mask_packed(protos, out.extra, out.boxes, out.counts, shape, upsample=True),
}
for fn in forms.values():   # warm-up: module loads, allocator, the workspace
    for _ in range(3):
        r = fn()
    del r
torch.cuda.synchronize()

e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
ms = {k: [] for k in forms}
for _ in range(a.rounds):
    for k, fn in forms.items():
        e0.record()
        for _ in range(a.reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        del r
        ms[k].append(e0.elapsed_time(e1) / a.reps)

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
rec = {
    "gpu": torch.cuda.get_device_name(dev), "power_limit": power,
    "batch": {"tiles": bs, "tile": tile, "max_det": md, "detections": int(out.counts.sum())},
    "ms_per_call": {k: statistics.median(v) for k, v in ms.items()},
    "ms_per_call_rounds": ms,
}
print(json.dumps(rec))
