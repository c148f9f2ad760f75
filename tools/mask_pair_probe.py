"""The two kernels of one packed, upsampled mask call on slide batches (148 tiles of the synthetic nuclei field, as
tools/mask_batch_probe.py builds them), timed with CUDA events and torch.profiler:

  (a) the whole call (masks.process_mask_packed: windows and offsets, binning, clear, regions, upsample), ms per
      batch;
  (b) the region kernel alone (proto_patch*), ms and GB/s against its algorithmic bytes (prototypes of the non-empty
      regions read once, coefficients of the live slots, patches written);
  (c) the upsample kernel alone (mask_upsample_pack2*), ms;
  (d) eight consecutive batches alternating over three streams, as SlidePostprocessor.masks runs them, ms per batch;
      the torch.profiler trace of (d) is written to OUT/pair_trace.pt.trace.json and the time during which a region
      kernel runs beside an upsample kernel of another stream is read from its kernel intervals.

usage: python tools/mask_pair_probe.py OUT_DIR [max_det]   (prints one JSON line, also written to OUT/pair_probe.json)"""
import json
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hd_yolo_b200 as hdy
from hd_yolo_b200 import masks as hm
from hd_yolo_b200 import synth
from hd_yolo_b200.ops import scratch_slot
from hd_yolo_b200.slide import sliding_window_scanner

out_dir = sys.argv[1]
md = int(sys.argv[2]) if len(sys.argv) > 2 else 3072
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")
bs, tile, nm, n_batches, n_streams = 148, 1024, 32, 8, 3
rois = sliding_window_scanner((100000, 100000), (tile, tile), 64)[1000:1000 + bs]
spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=4, no=9 + nm)
dets = synth.slide_tile_logits(rois, tile, 4, seed=1, first_tile=1000, extra=nm, device=dev)
out = hdy.detect_postprocess(dets, spec, 0.25, 0.45, md, cap=4096)
del dets
# distinct prototype maps per batch (1.24 GB each, 10x the L2), the detections of one batch for all of them
protos = [synth.slide_tile_protos(bs, tile, seed=1, first_tile=1000 + i * bs, device=dev) for i in range(n_batches)]
cap_words = int(bs * md * 40)


def call(p):
    return hm.process_mask_packed(p, out.extra, out.boxes, out.counts, (tile, tile), upsample=True,
                                  capacity_words=cap_words)


def kind(name):
    if "proto_patch" in name:
        return "region"
    if "mask_upsample_pack2" in name:
        return "upsample"
    return None


for p in protos:
    call(p)
torch.cuda.synchronize()
# (a) the whole call, one stream
reps = 3 * n_batches
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(reps):
    pm = call(protos[i % n_batches])
e1.record()
torch.cuda.synchronize()
pm.check()
call_ms = e0.elapsed_time(e1) / reps


def kernel_intervals(fn, trace):
    """(kind, start us, end us, stream) of the region and upsample kernels fn() launches, from a torch.profiler trace"""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        evs = json.load(f)["traceEvents"]
    return [(kind(e["name"]), e["ts"], e["ts"] + e["dur"], e["args"].get("stream")) for e in evs
            if e.get("cat") == "kernel" and kind(e.get("name", ""))]


# (b), (c): kernel durations of single-stream calls
single = kernel_intervals(lambda: [call(p) for p in protos], os.path.join(out_dir, "single_trace.pt.trace.json"))
dur = {k: [b - a for kk, a, b, _ in single if kk == k] for k in ("region", "upsample")}
region_ms = sum(dur["region"]) / max(len(dur["region"]), 1) / 1000.0
upsample_ms = sum(dur["upsample"]) / max(len(dur["upsample"]), 1) / 1000.0

# algorithmic bytes of the region kernel: prototypes of the non-empty regions (clipped to the plane) read once,
# coefficients of the live slots read, patches of the live slots written (what reaches the upsample)
mh = mw = tile // 4
rn = (mh + 23) // 24
ws, _ = hm._pm_workspace(dev, bs, md)
slots = bs * md
off_kr = 256 + ((slots * 4 + 255) & ~255)
kr = ws[off_kr:off_kr + slots * 16].view(torch.int32).view(slots, 4)
live = (kr[:, 2] > kr[:, 0]) & (kr[:, 3] > kr[:, 1])
n_live = int(live.sum())
touched = torch.zeros((bs, rn, rn), dtype=torch.bool, device=dev)
krl = kr[live].long()
tiles = torch.nonzero(live).squeeze(1) // md
for dy in range(2):
    for dx in range(2):
        ry = torch.minimum((krl[:, 1] // 24) + dy, (krl[:, 3] - 1) // 24)
        rx = torch.minimum((krl[:, 0] // 24) + dx, (krl[:, 2] - 1) // 24)
        touched[tiles, ry, rx] = True
widths = torch.tensor([min(24, mw - 24 * i) for i in range(rn)], device=dev)
region_px = (widths[None, :, None] * widths[None, None, :]).expand(bs, rn, rn)[touched].sum()
region_bytes = int(region_px) * nm * protos[0].element_size() + n_live * (nm * 4 + 16 * 16 * 4)

# (d) eight batches over three streams, batch i on stream i % 3 (the word cursor is not shared here: each call has
# its own output, so this times the kernels' overlap, not the pipeline's bookkeeping)
streams = [torch.cuda.Stream() for _ in range(n_streams)]


def pair_run():
    cur = torch.cuda.current_stream()
    for s in streams:
        s.wait_stream(cur)
    for i in range(n_batches):
        # a scratch set (workspace) of its own per stream, as the pipeline gives each of its lanes
        with torch.cuda.stream(streams[i % n_streams]), scratch_slot(8 + i % n_streams):
            call(protos[i])
    for s in streams:
        cur.wait_stream(s)


pair_run()
torch.cuda.synchronize()
times = []
for _ in range(5):
    e0.record()
    pair_run()
    e1.record()
    torch.cuda.synchronize()
    times.append(e0.elapsed_time(e1) / n_batches)
trace = os.path.join(out_dir, "pair_trace.pt.trace.json")
pair = kernel_intervals(pair_run, trace)
regions = [(a, b, s) for k, a, b, s in pair if k == "region"]
ups = [(a, b, s) for k, a, b, s in pair if k == "upsample"]
overlap_us = 0.0
for a0, a1, sa in regions:
    for b0, b1, sb in ups:
        if sb != sa:
            overlap_us += max(0.0, min(a1, b1) - max(a0, b0))
rec = {
    "gpu": torch.cuda.get_device_name(dev),
    "batch": {"tiles": bs, "max_det": md, "live_slots": n_live, "kept_per_tile": float(out.counts.float().mean())},
    "a_call_ms": call_ms,
    "b_region_ms": region_ms,
    "b_region_alg_bytes": region_bytes,
    "b_region_gbs": region_bytes / region_ms / 1e6,
    "c_upsample_ms": upsample_ms,
    "d_three_streams_ms_per_batch": min(times),
    "d_three_streams_ms_per_batch_all": times,
    "d_region_beside_upsample_us": overlap_us,
    "d_region_us": sum(b - a for a, b, _ in regions),
    "d_upsample_us": sum(b - a for a, b, _ in ups),
    "trace": os.path.basename(trace),
}
line = json.dumps(rec)
print(line)
with open(os.path.join(out_dir, "pair_probe.json"), "w") as f:
    f.write(line + "\n")
