#!/usr/bin/env python
"""Benchmark of the post-processing hot path (BASELINE.json metric: post-proc tiles/s & boxes/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload slide|tiles640|tiles1024|hnet] [--masks proto|none]
                    [--dtype f32|f16] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores

--dump-outputs DIR writes what the last timed step returned (detections in the caller's order, mask pixels) as .npy
files; the inputs are seeded, so two builds run with the same arguments can be compared output for output.

slide (default; BASELINE.json configs[3], the configuration the north-star target is quoted on): one "step" = a whole
synthetic 100k x 100k px slide (11 025 tiles of 1024 px, 64 px overlap, ~3 000 nuclei per tile) cut from one global
nuclei field: per-tile decode+filter+compact -> NMS -> score/label select of this rank's tile rows, append in slide
coordinates, exact slide-level merge NMS (seam exchange over NCCL when N > 1), then process_mask (32-prototype
contraction, sigmoid, crop, bilinear upsample, > 0.5, bit-packed) for the rows the merge KEPT.  Strong scaling.
Short runs of tiles640 / tiles1024 (configs[1] / configs[2]) and of the multi-scale RoIAlign (SURVEY 8f) are attached as
sub-records unless --no-sub.

tiles640 / tiles1024: one "step" = one pass of the per-tile path over one batch of synthetic head outputs (masks
included).  Weak scaling (every rank processes its own batches; the path has no cross-tile dependency).

Prints ONE JSON line on rank 0:
  value     : whole-job tiles/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e       : the same through the public API with HOST (pinned) inputs: H2D of the step's inputs and D2H of its
              results inside the timed region
  roofline  : the dominant HBM-bound call: algorithmic bytes per launch / its CUDA-event time (measured live)
  stages    : every C-ABI call of the step with its time, algorithmic bytes and achieved GB/s
  pipeline  : the whole step's algorithmic bytes / its time, against the HBM peak (the north star's "% of roofline")
  cpu_baseline : oracle port (the reference's torch/torchvision CPU path) on a bounded sample
  torch_cuda   : diagnostic, not product: the same port on CUDA tensors (ATen / torchvision CUDA kernels) -- the
                 library GPU path SURVEY 2b names as the bar
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# NCCL (NCCL_DEBUG=VERSION/INFO) or any library may write to fd 1: the JSON line goes to a private duplicate of stdout,
# everything else that is written to fd 1 lands on stderr -- rank 0 prints ONE JSON line whatever the environment asks.
_JSON_FD = None


def _protect_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)

WORKLOADS = {
    # BASELINE.json configs[1]: 640x640 tiles, batch 64, 3 anchor levels, 32 prototypes, ~1k candidates/tile
    "tiles640": dict(tile=640, bs=64, n_cand=1000, conf=0.25, iou=0.45, max_det=1000, nc=4, cap=2048),
    # BASELINE.json configs[2]: 1024x1024 dense-nuclei tiles, batch 128, ~3k candidates/tile
    "tiles1024": dict(tile=1024, bs=128, n_cand=3000, conf=0.25, iou=0.45, max_det=3000, nc=4, cap=4096),
    # BASELINE.json configs[3]: whole slide, 1024-px tiles, 64-px overlap, ~3k candidates/tile
    # (148 tiles per batch: the per-tile NMS runs one CTA per tile, one per SM)
    # (the field holds at most 55 x 55 = 3 025 nuclei per tile, so max_det = cap = 3072 never binds)
    # (cap 3072: the per-tile NMS instance that shares an SM with the filter of the next batch; an overflow raises)
    "slide": dict(tile=1024, bs=148, n_cand=3000, conf=0.25, iou=0.45, max_det=3072, nc=4, cap=3072, overlap=64),
    # BASELINE.json configs[4]: hnet multi-level heads (RCNN-style 10x structures + 40x nuclei), cross-level merge
    "hnet": dict(tile=1024, bs=16, n_cand=3000, conf=0.25, iou=0.45, max_det=4096, nc=4, cap=4096, overlap=64),
}
NM = 32            # prototypes
L2_BYTES = 126e6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="slide", choices=list(WORKLOADS))
    ap.add_argument("--masks", default=None, choices=["proto", "paste", "none"],
                    help="mask stage (default: proto; --impl reference: paste, the reference's own mask path)")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f16"],
                    help="element type of the head outputs (logits, prototypes) as they arrive; f16 = a half() model, "
                         "the reference's GPU default (val_nuclei.py:109,115-116).  Arithmetic is fp32 either way.")
    ap.add_argument("--slide-size", type=int, default=100000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", "--no-slide", dest="no_sub", action="store_true",
                    help="no sub-records (slide: tiles640/tiles1024 runs; tiles: the short slide run)")
    ap.add_argument("--no-torch-cuda", action="store_true")
    ap.add_argument("--proto-pool", type=int, default=592,
                    help="slide: distinct prototype maps (tile t reads map t mod pool; 592 x 8.4 MB = 5 GB, 40x L2)")
    ap.add_argument("--layout", type=int, default=0, choices=[0, 1],
                    help="tiles workloads: 0 = the reference's permuted [bs,na,ny,nx,no] head tensors, 1 = the 1x1 "
                         "conv's native [bs,na*no,ny,nx] output (the yolo_head.py:141-145 permute copy skipped)")
    ap.add_argument("--slide-streams", type=int, default=3,
                    help="slide workload: tile batches alternate over this many streams (SlidePostprocessor(streams=))")
    ap.add_argument("--inflight", type=int, default=3, help="steps in flight (CUDA graphs on separate streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 or "
                         "float64; a fixed, seeded sample of the detections and masks of a large step; with --gpus > 1 the part of "
                         "rank 0)")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl == "reference" or a.workload == "hnet"):
        ap.error("--dump-outputs covers --impl ours on the slide, tiles640 and tiles1024 workloads")
    if a.masks is None:
        a.masks = "paste" if a.impl == "reference" else "proto"
    if a.steps is None:
        a.steps = 5 if a.workload in ("slide", "hnet") else 200
    if a.warmup is None:
        a.warmup = 3 if a.workload in ("slide", "hnet") else 10
    return a


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed regions run (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
MASK_CHUNK = 300    # detections per paste / process_mask call on the CPU: the dense [k,1,H,W] fp32 canvases the
                    # reference allocates are 4 MB each at 1024 px (12.6 GB for one tile's 3 000 detections)


def _cpu_tile_pass(dets, second, wl, masks, tile_px, device=None):
    """The reference's per-tile path for a batch of tiles (oracle port, torch/torchvision ops on `device`):
    compute_proposals -> level pad/cat -> nms_per_image -> hierarchical scores + select
      -> masks == "paste": mask select (yolo_head.py:346-353) + paste_masks_in_image (val_nuclei.py:169-176) > 0.5
         masks == "proto": upstream process_mask (contraction, sigmoid, crop, upsample, > 0.5)
    Returns [(boxes, scores, labels, n_mask_pixels)] per tile."""
    import torch
    from oracle import port
    from hd_yolo_b200 import synth
    nc = wl["nc"]
    preds = port.compute_proposals(dets, synth.ANCHORS_3, synth.STRIDES_3)
    cat = port.concat_levels(preds)
    if masks == "proto":    # mask coefficients travel raw (no sigmoid), as in the device path
        raw = torch.cat([d.reshape(d.shape[0], -1, d.shape[-1]) for d in dets], 1)
        cat[..., 5 + nc:5 + nc + NM] = raw[..., 5 + nc:5 + nc + NM]
    res = port.nms_per_image(cat, nc, wl["conf"], wl["iou"], wl["max_det"])
    out = []
    for i, r in enumerate(res):
        s, l = port.select_scores(r['scores'][:, :1 + nc].clone(), wl["conf"], port.default_descendants(nc))
        k, px = len(r['boxes']), 0
        for c0 in range(0, k if masks != "none" else 0, MASK_CHUNK):
            c1 = min(c0 + MASK_CHUNK, k)
            if masks == "proto":
                coef = r['extra'][c0:c1, :NM]   # extra = raw coefficient channels + level id; coefficients first
                m = port.process_mask(second[i].float(), coef.float(), r['boxes'][c0:c1].clone(), (tile_px, tile_px),
                                      upsample=True)
            else:
                sel = port.mask_select(second[i][c0:c1].float(), l[c0:c1],
                                       torch.tensor([-1, 0, 0, 1, 1], device=l.device))
                m = port.paste_masks_in_image(sel, r['boxes'][c0:c1], (tile_px, tile_px), padding=1) > 0.5
            px += int(m.sum())
        out.append((r['boxes'], s, l, px))
    return out


def cpu_sample(workload, wl, masks, n_tiles, dtype="f32", device="cpu", slide_size=100000):
    """A bounded sample of the workload as CPU (or `device`) tensors + a function running the reference path on it.
    slide: the first n_tiles tiles of the slide's first tile row (adjacent: their overlap bands hold duplicates), the
    per-tile path, then merge_outputs + Ensemble.merge over them."""
    import torch
    from oracle import port
    from hd_yolo_b200 import synth
    from hd_yolo_b200.slide import sliding_window_scanner
    tile, nc = wl["tile"], wl["nc"]
    extra = NM if masks == "proto" else 0
    td = torch.float16 if (dtype == "f16" and device != "cpu") else torch.float32   # CPU NMS/sigmoid: fp32 only
    rois = None
    if workload == "slide":
        rois = sliding_window_scanner((slide_size, slide_size), (tile, tile), wl["overlap"])[:n_tiles]
        dets = synth.slide_tile_logits(rois, tile, nc, seed=1, first_tile=0, conf=wl["conf"], extra=extra,
                                       device=device)
    else:
        dets = [d.to(device) for d in synth.nuclei_logits(n_tiles, tile, nc, wl["n_cand"], seed=1, conf=wl["conf"],
                                                          extra=extra)]
    if dtype == "f16":       # the same fp16-rounded numbers the GPU arm reads
        dets = [d.half().to(td) for d in dets]
    g = torch.Generator().manual_seed(8)
    second = None
    if masks == "proto":
        second = synth.slide_tile_protos(n_tiles, tile, seed=1, first_tile=0, nm=NM, device=device)
        if dtype == "f16":
            second = second.half().to(td)
    elif masks == "paste":
        second = torch.randn((n_tiles, min(wl["max_det"], wl["cap"]), 2, 28, 28), generator=g).to(device)

    def run():
        res = _cpu_tile_pass([d.float() for d in dets], second, wl, masks, tile)
        if workload == "slide":
            tiles = [{'boxes': b, 'scores': sc, 'labels': l, 'roi': rois[i].to(b.device)}
                     for i, (b, sc, l, _) in enumerate(res)]
            port.ensemble_merge([{'det': port.merge_outputs(tiles)}],
                                {'conf_thres': wl["conf"], 'iou_thres': wl["iou"], 'max_det': 10 ** 9})
        return res

    what = "compute_proposals + level cat + nms_per_image + score select" + \
        {"proto": " + process_mask(upsample) > 0.5", "paste": " + mask_select + paste_masks_in_image > 0.5",
         "none": ""}[masks] + (" + merge_outputs + Ensemble.merge over the sample's tiles" if workload == "slide" else "")
    return run, what


def time_cpu(workload, wl, masks, budget_s, max_passes, threads=None, dtype="f32", n_tiles=None, slide_size=100000):
    """Bounded CPU timing of the oracle port on `threads` host threads (default: all).  Every pass is a whole sample;
    nothing is extrapolated.  Returns a dict for the JSON line."""
    import torch
    torch.set_num_threads(threads or os.cpu_count() or 1)
    if n_tiles is None:
        n_tiles = 2 if (masks != "none" and wl["tile"] >= 1024) else (4 if masks != "none" else 8)
    run, what = cpu_sample(workload, wl, masks, n_tiles, dtype, "cpu", slide_size)
    global MASK_CHUNK
    keep, MASK_CHUNK = MASK_CHUNK, 64
    try:                                    # warm the allocator / thread pools on a cheaper configuration of the same
        wrun, _ = cpu_sample(workload, dict(wl, max_det=64), masks, 1, dtype, "cpu", slide_size)
        wrun()
    finally:
        MASK_CHUNK = keep
    passes, t0 = 0, time.perf_counter()
    while passes < 1 or (passes < max_passes and (time.perf_counter() - t0) * (passes + 1) / passes < budget_s):
        run()
        passes += 1
    dt = time.perf_counter() - t0
    return {"value": n_tiles * passes / dt, "unit": "tiles/s", "cores": torch.get_num_threads(), "kind": "port",
            "ms_per_pass": 1e3 * dt / passes, "tiles_per_pass": n_tiles, "passes": passes,
            "sample": f"{n_tiles} tiles x {passes} timed passes of oracle/port.py ({what}; torch {torch.__version__} CPU "
                      f"+ torchvision; mask canvases in chunks of {MASK_CHUNK} detections; one process)"}


def time_torch_cuda(workload, wl, masks, dtype, device, n_tiles=4, passes=3, slide_size=100000):
    """DIAGNOSTIC, not the product and not the reference arm: the same oracle port on CUDA tensors (ATen's and
    torchvision's CUDA kernels) on this GPU -- the library GPU path SURVEY 2b names as the bar to beat."""
    import torch
    run, what = cpu_sample(workload, wl, masks, n_tiles, dtype, device, slide_size)
    run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(passes):
        run()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": n_tiles * passes / dt, "unit": "tiles/s", "ms_per_pass": 1e3 * dt / passes,
            "tiles_per_pass": n_tiles, "passes": passes,
            "what": f"oracle/port.py on CUDA tensors ({what}); wall clock around synchronised passes, one GPU"}


def cpu_merge_scaling(boxes, scores, tile, n_cols, conf, iou, grids=(2, 3, 4, 6, 8), budget_s=25.0):
    """SURVEY 8d: the reference's slide merge (Ensemble.merge, yolo.py:165-204 = one dense torchvision.ops.nms over
    everything merge_outputs concatenated) is O(n^2) -- 338 s at 2e5 boxes -- so it is timed on g x g tile sub-slides
    of the SAME detections and reported with its measured exponent instead of an extrapolated full-slide number.
    boxes [n,4] / scores [n] / tile [n] (tile index in the slide's row-major grid of n_cols columns): CPU tensors in
    merge_outputs' order.  Returns a dict for the JSON line."""
    import math
    import torch
    from oracle import port
    torch.set_num_threads(os.cpu_count() or 1)
    rows, cols = tile // n_cols, tile % n_cols
    pts, t_start = [], time.perf_counter()
    for g in grids:
        sel = (rows < g) & (cols < g)
        b, sc = boxes[sel].contiguous(), scores[sel].contiguous()
        if len(b) < 16:
            continue
        if pts and time.perf_counter() - t_start + pts[-1][2] * (len(b) / pts[-1][1]) ** 2 > budget_s:
            break                                   # the next size would not fit the budget
        labels = torch.zeros((len(b),), dtype=torch.int64)
        t0 = time.perf_counter()
        r = port.ensemble_merge([{'det': {'boxes': b, 'scores': sc, 'labels': labels}}],
                                {'conf_thres': conf, 'iou_thres': iou, 'max_det': 10 ** 9})['det']
        pts.append((g * g, int(len(b)), time.perf_counter() - t0, int(len(r['boxes']))))
    out = {"what": "oracle port of Ensemble.merge (dense torchvision.ops.nms) on g x g tile sub-slides of the bench's "
                   "own detections, all host threads", "cores": torch.get_num_threads(),
           "tiles": [p[0] for p in pts], "boxes": [p[1] for p in pts], "seconds": [round(p[2], 4) for p in pts],
           "kept": [p[3] for p in pts]}
    if len(pts) >= 2:
        xs = [math.log(p[1]) for p in pts]
        ys = [math.log(max(p[2], 1e-9)) for p in pts]
        mx, my = sum(xs) / len(xs), sum(ys) / len(ys)
        den = sum((x - mx) ** 2 for x in xs)
        out["exponent"] = round(sum((x - mx) * (y - my) for x, y in zip(xs, ys)) / den, 3) if den > 0 else None
    return out


def common_config(args, wl, masks):
    """The keys both arms print under "config" (same keys, same workload parameters)."""
    cfg = {"workload": args.workload, "tile": wl["tile"], "candidates_per_tile": wl["n_cand"], "conf": wl["conf"],
           "iou": wl["iou"], "max_det": wl["max_det"], "masks": masks, "dtype_in": args.dtype}
    if args.workload == "slide":
        cfg.update({"slide_px": args.slide_size, "overlap": wl["overlap"]})
    return cfg


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation (oracle port: same torch/torchvision calls) on all
    host threads of ONE process; each step is one pass over a bounded sample of the workload, --steps passes timed
    whole -- ms_per_step is the measured time of one sample pass."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    masks = args.masks
    wk = args.workload if args.workload != "hnet" else "tiles1024"
    r = time_cpu(wk, wl, masks, budget_s=float("inf"), max_passes=args.steps, dtype=args.dtype,
                 slide_size=args.slide_size)
    other = None
    if masks in ("paste", "proto"):      # the other mask variant beside it (one pass)
        om = "proto" if masks == "paste" else "paste"
        o = time_cpu(wk, wl, om, budget_s=1.0, max_passes=1, dtype=args.dtype, n_tiles=1, slide_size=args.slide_size)
        other = {"masks": om, "value": o["value"], "unit": "tiles/s", "ms_per_pass": o["ms_per_pass"],
                 "tiles_per_pass": o["tiles_per_pass"]}
    v = r["value"]
    cfg = common_config(args, wl, masks)
    cfg["note"] = ("masks=paste is the reference's own mask path (yolo_head.py:346-353 + torchvision "
                   "paste_masks_in_image, val_nuclei.py:169-176); masks=proto is upstream yolov5's process_mask, "
                   "which the reference does not contain.  One CPU process whatever --gpus says.")
    line = {
        "impl": "reference", "metric": "postproc_tiles_per_s", "value": v, "unit": "tiles/s", "n_gpus": args.gpus,
        "steps": r["passes"], "steps_requested": args.steps, "warmup": 1, "ms_per_step": r["ms_per_pass"],
        "tiles_per_step": r["tiles_per_pass"], "higher_is_better": True,
        "scaling": "strong" if args.workload == "slide" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": v, "unit": "tiles/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": v, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "boxes_per_s": v * wl["n_cand"], "other_mask_variant": other,
    }
    _emit(line)


# ------------------------------------------------------------------------------------------------ helpers
class Ctx:
    pass


try:
    _ORIG_AFFINITY = os.sched_getaffinity(0)
except Exception:   # not on Linux
    _ORIG_AFFINITY = set()


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs next to GPU `index` (sysfs local_cpulist of its PCI function) before any pinned
    host buffer is allocated: first-touch then places the e2e staging buffers on the GPU's own NUMA node, which is
    worth up to 1.4x of H2D bandwidth on a two-socket box.  Returns a short description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus and len(cpus) < len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return f"bound to the {len(cpus)} CPUs local to GPU {index}"
        return "all CPUs are local to the GPU (single NUMA node)"
    except Exception as e:  # no sysfs entry / no PCI ids: leave the affinity alone
        return f"unchanged ({type(e).__name__})"


def make_ctx(args):
    c = Ctx()
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.rank = int(os.environ.get("RANK", "0"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(c.local)
    c.affinity = bind_to_gpu_numa_node(c.local)
    c.dev = torch.device("cuda", c.local)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=c.dev)
    assert c.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={c.world}: launch with torch.distributed.run"

    def barrier():
        if c.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, side_streams=()):
        """CUDA events around `steps` calls, barrier + synchronize on both sides, max over ranks (ms).  Work that fn
        issues on side_streams is ordered after the start event and before the end event."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main = torch.cuda.current_stream()
        e0.record()
        for s_ in side_streams:
            s_.wait_event(e0)
        for i in range(steps):
            fn(i)
        for s_ in side_streams:
            main.wait_stream(s_)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if c.world > 1:
            t = torch.tensor([ms], device=c.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    c.barrier, c.timed = barrier, timed
    return c


def load_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (of fallback)"


DUMP_ROWS = 1 << 19     # detections written by --dump-outputs (a seeded sample above that)
DUMP_MASKS = 2048       # of which the first DUMP_MASKS also have their mask pixels written
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, boxes, scores, labels, mask_rows, masks, extra):
    """--dump-outputs: the detections of the last timed step in the order the caller receives them (boxes [K,4],
    scores [K], labels [K]) and their masks (row mask_rows[k] of the PackedMasks `masks`, or None).  Above DUMP_ROWS
    detections a fixed, seeded sample is written (sample.npy: the positions in [0, K)); the masks of the first
    DUMP_MASKS detections of the sample are unpacked to 0/1 pixels (mask_windows.npy: x0, y0, w, h; mask_pixels.npy:
    every window row-major, one after the other).  `extra`: further small arrays, written as they are."""
    import numpy as np
    import torch
    K = int(boxes.shape[0])
    pos = np.arange(K) if K <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(K, DUMP_ROWS, replace=False))
    sel = torch.from_numpy(pos).to(boxes.device)
    arrays = dict(extra)
    arrays.update(sample=pos.astype(np.float64), boxes=boxes[sel].float().cpu().numpy(),
                  scores=scores[sel].float().cpu().numpy(), labels=labels[sel].cpu().numpy().astype(np.float32))
    if masks is not None:
        rows = mask_rows[sel[:DUMP_MASKS]].to(torch.int64)
        g = masks.geom[rows].to(torch.int64)
        wpr = (g[:, 2] + 31) >> 5                          # 32-bit words per mask row
        words = wpr * g[:, 3]
        owner = torch.repeat_interleave(torch.arange(rows.numel(), device=rows.device), words)
        j = torch.arange(int(words.sum()), device=rows.device) - (torch.cumsum(words, 0) - words)[owner]
        bits = np.unpackbits(masks.bits[masks.offsets[rows][owner] + j].cpu().numpy().view(np.uint8), bitorder="little")
        g, wpr = g.cpu().numpy(), wpr.cpu().numpy()
        pix, o = [], 0
        for (_, _, w, h), n in zip(g, wpr):                # pixel (x, y) of a window is bit x of its row y
            pix.append(bits[o:o + h * n * 32].reshape(h, n * 32)[:, :w].reshape(-1))
            o += h * n * 32
        arrays["mask_windows"] = g.astype(np.float32)
        arrays["mask_pixels"] = (np.concatenate(pix) if pix else np.zeros((0,), np.uint8)).astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ tiles workloads
def run_tiles(args, wl, c, dump=None):
    import torch
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import masks as hmasks
    from hd_yolo_b200 import ops, synth

    masks = args.masks
    extra = NM if masks == "proto" else 0
    nc, tile, bs, K, W = wl["nc"], wl["tile"], wl["bs"], args.steps, max(args.warmup, 3)
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=nc, no=5 + nc + extra)
    shapes = synth.level_shapes(tile, synth.STRIDES_3)
    N = spec.rows_per_tile(shapes)
    mh = mw = tile // 4
    td = torch.float16 if args.dtype == "f16" else torch.float32
    esz = 2 if args.dtype == "f16" else 4
    if args.dtype == "f16" and args.layout == 1:
        raise SystemExit("--dtype f16 reads layout 0 only")
    in_bytes = bs * N * spec.no * esz + (bs * NM * mh * mw * esz if masks == "proto" else 0) + \
        (bs * min(wl["max_det"], wl["cap"]) * 2 * 28 * 28 * 4 if masks == "paste" else 0)
    R = max(2, args.inflight, int(2.5 * L2_BYTES / in_bytes) + 1)   # rotate input batches so that reads miss L2
    batches = [[d.to(td) for d in synth.nuclei_logits(bs, tile, nc, wl["n_cand"], seed=1000 * c.rank + r,
                                                      conf=wl["conf"], extra=extra, generator_device="cuda")]
               for r in range(R)]
    if args.layout == 1:   # the same logits as the head's 1x1 conv leaves them: [bs, na*no, ny, nx]
        batches = [[d.permute(0, 1, 4, 2, 3).reshape(d.shape[0], -1, d.shape[2], d.shape[3]).contiguous() for d in b]
                   for b in batches]
    protos = None
    if masks == "proto":
        g = torch.Generator(device="cuda").manual_seed(77 + c.rank)
        protos = [torch.randn((bs, NM, mh, mw), generator=g, device=c.dev).to(td) for _ in range(R)]
    md_slots = min(wl["max_det"], wl["cap"])
    mlogits = None
    if masks == "paste":
        # reference variant A (yolo_head.py:321-353 + torchvision paste_masks_in_image): one 2-channel 28x28 mask
        # logit map per detection slot, as the RoI mask head would produce them
        g = torch.Generator(device="cuda").manual_seed(78 + c.rank)
        mlogits = [torch.randn((bs * md_slots, 2, 28, 28), generator=g, device=c.dev) for _ in range(R)]
        mask_indices = torch.tensor([-1, 0, 0, 1, 1], dtype=torch.int32, device=c.dev)
        slot_ids = torch.arange(md_slots, device=c.dev)[None, :]
    state = {"cap_words": None}

    def step(i, dets=None, pr=None):
        out = hdy.detect_postprocess(dets if dets is not None else batches[i % R], spec, wl["conf"], wl["iou"],
                                     wl["max_det"], cap=wl["cap"], layout=args.layout)
        pm = None
        if masks == "proto":
            pm = hmasks.process_mask_packed(pr if pr is not None else protos[i % R], out.extra, out.boxes, out.counts,
                                            (tile, tile), upsample=True, capacity_words=state["cap_words"])
        elif masks == "paste":
            # M1: channel = mask_indices[labels.clamp(min=0)], empty beyond counts; M2+M3 fused and bit-packed
            live = slot_ids < out.counts[:, None]            # slots beyond counts hold uninitialised labels
            ch = mask_indices[torch.where(live, out.labels, torch.zeros_like(out.labels)).clamp(min=0)]
            ch = torch.where(live, ch, torch.full_like(ch, -1)).reshape(-1)
            pm = hmasks.paste_masks_packed(pr if pr is not None else mlogits[i % R], out.boxes.reshape(-1, 4),
                                           (tile, tile), padding=1, channel=ch, apply_sigmoid=True,
                                           capacity_words=state["cap_words"])
        return out, pm

    # size the packed-mask buffer once (the only call that reads a size back), then never sync inside a step
    out, pm = step(0)
    out.to_list()                      # raises on candidate-capacity overflow
    words = 0
    if pm is not None:
        words = int(pm.offsets[-1].item())
        state["cap_words"] = int(words * 1.2) + 1024

    sampler = ClockSampler(c.local)
    sampler.start()
    for i in range(W):
        out, pm = step(i)
    if pm is not None:
        pm.check()
    # The step is launch-bound on the host at these sizes (7 C-ABI calls + ~25 small allocations per step), so the
    # public API offers CUDA-graph capture of a fixed-shape step (hdy.CapturedStep); one graph per rotating input batch.
    # Every graph has its own scratch slot, so two steps can be in flight on two streams: the per-tile NMS occupies
    # only `bs` of the 148 SMs and the tails of the other kernels leave SMs idle, which the neighbouring step fills.
    graphs = [hdy.CapturedStep(lambda r=r: step(r), slot=r) for r in range(R)]
    side = [torch.cuda.Stream() for _ in range(max(1, args.inflight))]

    def gstep(i):
        return graphs[i % R]()

    def gstep2(i):
        return graphs[i % R](stream=side[(i % R) % len(side)])

    for i in range(W):
        gstep(i)
    ms_serial = c.timed(gstep, K)
    for i in range(W):
        gstep2(i)
    torch.cuda.synchronize()
    ops.profile.reset()
    ms = c.timed(gstep2, K, side_streams=side)
    launches = ops.profile.launches
    if dump and c.rank == 0:        # the last timed step replayed graph (K-1) mod R, whose outputs stay in place
        o, p = graphs[(K - 1) % R].out
        live = torch.arange(o.max_det, device=c.dev)[None, :] < o.counts[:, None]
        rows = torch.nonzero(live.reshape(-1)).flatten()     # tile-major; mask index = tile * max_det + slot
        dump_outputs(dump, o.boxes.reshape(-1, 4)[rows], o.scores.reshape(-1)[rows], o.labels.reshape(-1)[rows], rows,
                     p, {"counts": o.counts.cpu().numpy().astype("float64")})
    tiles_per_s = c.world * bs * K / (ms * 1e-3)
    torch.cuda.synchronize()
    out, pm = gstep(0)

    # ---- per-call CUDA-event times of the same step, un-graphed.  A GPU-side sleep is queued first so that the
    #      host runs ahead and the event pairs bracket back-to-back kernels, not launch gaps.
    ops.profile.enabled = True
    ops.profile.reset()

    def pstep(i):
        torch.cuda._sleep(3_000_000)
        step(i)

    c.timed(pstep, min(K, 50))
    prof = ops.profile.summary()
    ops.profile.enabled = False
    cand = float(out.cand_counts[:bs].float().mean())
    kept = float(out.counts.float().mean())
    ne = spec.no - 5 - nc
    alg = {   # algorithmic bytes per launch (DESIGN.md section 3)
        # layout 1: only the objectness plane is streamed, survivors gather their four box logits
        "hdy_filter_compact_logits": bs * (esz * N * spec.no + 24 * cand) if args.layout == 0
        else bs * (4 * N + (16 + 24) * cand),
        "hdy_nms_tiles": bs * (24 * cand + 28 * kept),
        "hdy_gather_logits": bs * kept * ((4 + esz) * (1 + nc + ne) + 4),
        "hdy_gather_select_logits": bs * kept * ((4 + esz) * (1 + nc + ne) + 4 + 4 + 8),
        "hdy_select_scores": bs * kept * (4 * (1 + nc) * 2 + 4 + 8),
        "hdy_process_mask_geometry": bs * min(wl["max_det"], wl["cap"]) * (16 + 16 + 8),
        "hdy_process_mask_packed": bs * (esz * NM * mh * mw + kept * (4 * NM + 16 + 8)) + 4 * words,
        "hdy_zero_i32": 4 * (bs + 1),
        "hdy_paste_geometry": bs * md_slots * (16 + 16 + 8 + 4),
        "hdy_paste_masks_packed": bs * kept * (28 * 28 * 4 + 16 + 8) + 4 * words,
    }
    peak, peak_src = load_peak()
    stages = {}
    for name, (calls, tot) in prof.items():
        t = tot / calls
        a = alg.get(name)
        stages[name] = {"ms": t, "alg_bytes": a, "gbs": (a / (t * 1e-3) / 1e9) if a else None}
    hbm_bound = [k for k in stages if k in ("hdy_filter_compact_logits", "hdy_process_mask_packed",
                                            "hdy_paste_masks_packed")]
    dom = max(hbm_bound, key=lambda k: stages[k]["ms"])
    dom_ms, dom_bytes = stages[dom]["ms"], alg[dom]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    step_bytes = sum(v["alg_bytes"] for v in stages.values() if v["alg_bytes"])
    traffic = None
    try:   # DRAM bytes per launch of the dominant call, from the committed ncu --set full capture of this workload
        tr = "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else \
            "r01_traffic.json"
        traffic = json.load(open(os.path.join(ROOT, "profiles", tr)))[args.workload][dom]["bytes"]
        if args.dtype != "f32" or (masks != "proto" and dom == "hdy_filter_compact_logits" and
                                   args.workload != "tiles1024"):
            traffic = None
    except Exception:
        pass

    # ---- e2e: host (pinned) inputs, H2D + D2H inside the timed region ---------------------------------------
    e2e = None
    if not args.no_e2e:
        host = [[d.cpu().pin_memory() for d in b] for b in batches[:2]]
        second = protos if protos is not None else mlogits
        host_p = [p.cpu().pin_memory() for p in second[:2]] if second is not None else None
        stage = [torch.empty_like(d) for d in batches[0]]
        stage_p = torch.empty_like(second[0]) if second is not None else None
        md = out.max_det
        h = {"boxes": torch.empty((bs, md, 4), dtype=torch.float32).pin_memory(),
             "scores": torch.empty((bs, md), dtype=torch.float32).pin_memory(),
             "labels": torch.empty((bs, md), dtype=torch.int64).pin_memory(),
             "counts": torch.empty((bs,), dtype=torch.int32).pin_memory()}
        if pm is not None:
            h["geom"] = torch.empty(tuple(pm.geom.shape), dtype=torch.int32).pin_memory()
            h["offsets"] = torch.empty(tuple(pm.offsets.shape), dtype=torch.int64).pin_memory()
            h["bits"] = torch.empty((state["cap_words"],), dtype=torch.int32).pin_memory()

        # Two staging sets and two graphs: the H2D copy of step i+1 runs on a copy stream while step i computes and
        # reads back (PCIe is full duplex), as a serving loop would; every byte of every step is still copied inside
        # the timed region.
        stage2 = [torch.empty_like(d) for d in batches[0]]
        stage_p2 = torch.empty_like(second[0]) if second is not None else None
        stages_e = [(stage, stage_p), (stage2, stage_p2)]
        graphs_e = [hdy.CapturedStep(lambda: step(0, stage, stage_p), slot=0),
                    hdy.CapturedStep(lambda: step(0, stage2, stage_p2), slot=1)]
        copy_stream = torch.cuda.Stream()
        ready = [None, None]     # H2D of the set finished
        freed = [None, None]     # the graph that read the set finished

        def issue_h2d(i):
            k = i % 2
            st, stp = stages_e[k]
            with torch.cuda.stream(copy_stream):
                if freed[k] is not None:
                    copy_stream.wait_event(freed[k])
                for s, hh in zip(st, host[i % 2]):
                    s.copy_(hh, non_blocking=True)
                if stp is not None:
                    stp.copy_(host_p[i % 2], non_blocking=True)
                ready[k] = torch.cuda.Event()
                ready[k].record(copy_stream)

        pending = {"next": None}

        def e2e_step(i):
            if pending["next"] != i:      # first step of a run: nothing was prefetched
                issue_h2d(i)
            k = i % 2
            cur = torch.cuda.current_stream()
            cur.wait_event(ready[k])
            o, p = graphs_e[k]()
            freed[k] = torch.cuda.Event()
            freed[k].record(cur)
            issue_h2d(i + 1)              # overlaps the read-back below and the next replay's wait
            pending["next"] = i + 1
            h["boxes"].copy_(o.boxes, non_blocking=True)
            h["scores"].copy_(o.scores, non_blocking=True)
            h["labels"].copy_(o.labels, non_blocking=True)
            h["counts"].copy_(o.counts, non_blocking=True)
            if p is not None:
                h["geom"].copy_(p.geom, non_blocking=True)
                h["offsets"].copy_(p.offsets, non_blocking=True)
                h["bits"][:p.bits.numel()].copy_(p.bits, non_blocking=True)

        Ke = max(3, min(K, 50))
        for i in range(3):
            e2e_step(i)
        pending["next"] = None
        torch.cuda.synchronize()
        ms_e = c.timed(e2e_step, Ke, side_streams=(copy_stream,))
        d2h = sum(t.numel() * t.element_size() for k, t in h.items() if k != "bits") + (words * 4 if pm is not None else 0)
        e2e = {"value": c.world * bs * Ke / (ms_e * 1e-3), "unit": "tiles/s", "h2d_bytes_per_step": in_bytes,
               "d2h_bytes_per_step": d2h, "steps": Ke, "ms_per_step": ms_e / Ke}
        del host, host_p, stage, stage_p, stage2, stage_p2, stages_e, graphs_e, h
    clocks = sampler.stop()

    line = {
        "metric": "postproc_tiles_per_s", "value": tiles_per_s, "unit": "tiles/s", "n_gpus": c.world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**common_config(args, wl, masks), "tiles_per_step_per_gpu": bs, "levels": 3,
                   "layout": "permuted [bs,na,ny,nx,no] (what the reference's Detect.forward hands over)"
                   if args.layout == 0 else "conv-native [bs,na*no,ny,nx] (yolo_head.py:141-145 permute skipped)",
                   "rows_per_tile": N, "channels": spec.no, "prototypes": NM if masks == "proto" else 0,
                   "candidates_per_tile": round(cand, 1), "kept_per_tile": round(kept, 1), "conf": wl["conf"],
                   "iou": wl["iou"], "max_det": wl["max_det"], "cap": wl["cap"],
                   "stages": "decode+filter+compact, nms, score/label select" +
                             (", process_mask (proto contraction, sigmoid, crop, upsample, >0.5, bit-packed)" if masks == "proto" else "") +
                             (", mask select + paste_masks_in_image > 0.5 (28x28 mask logits, bit-packed)" if masks == "paste" else ""),
                   "l2": f"{R} rotating input batches ({R * in_bytes / 1e6:.0f} MB) > 126 MB L2",
                   "launch": f"one CUDA graph per input batch (hdy.CapturedStep), replayed; {len(side)} steps in "
                             "flight on as many streams (each graph has its own scratch slot)",
                   "ms_per_step_one_stream": ms_serial / K},
        "boxes_per_s": tiles_per_s * cand,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0, "traffic": traffic,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms},
        "stages": stages,
        "pipeline": {"algorithmic_bytes_per_step": step_bytes, "achieved_gbs": step_bytes / (ms / K * 1e-3) / 1e9,
                     "frac_of_peak": step_bytes / (ms / K * 1e-3) / 1e9 / peak},
        "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }
    del batches, protos, mlogits, graphs
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------ slide workload
def _timed_phase(c, fn, reps):
    """max-over-ranks CUDA-event time of `reps` calls of fn (ms per call)."""
    return c.timed(lambda i: fn(), reps) / reps


def run_slide(args, wl, c, steps, warmup, want_e2e, want_cpu_merge=False, masks="proto", want_stages=True, dump=None):
    import numpy as np
    import torch
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import ops, synth
    from hd_yolo_b200.pipeline import SlidePostprocessor
    from hd_yolo_b200.slide import fold_digest, kept_digest, mask_digest

    nc, tile, bs = wl["nc"], wl["tile"], wl["bs"]
    with_masks = masks == "proto"
    extra = NM if with_masks else 0
    td = torch.float16 if args.dtype == "f16" else torch.float32
    esz = 2 if args.dtype == "f16" else 4
    spec = hdy.HeadSpec(synth.ANCHORS_3, synth.STRIDES_3, nc=nc, no=5 + nc + extra)
    S = args.slide_size
    post = SlidePostprocessor(spec, (S, S), (tile, tile), wl["overlap"], wl["conf"], wl["iou"], wl["max_det"],
                              cap=wl["cap"], batch=bs, rank=c.rank, world=c.world, device=c.dev,
                              capacity=None, streams=args.slide_streams)
    t0, t1 = post.tile_range
    n_tiles = int(post.rois.shape[0])
    mh = tile // 4
    # this rank's head outputs for the whole slide, resident in HBM (N=1, fp32, 41 channels: 11 025 tiles x 10.6 MB =
    # 117 GB); every tile's bytes are a function of its global index alone, however the slide is sharded
    store = []
    for a in range(t0, t1, bs):
        b = min(a + bs, t1)
        store.append(synth.slide_tile_logits(post.rois[a:b], tile, nc, seed=1, first_tile=a, conf=wl["conf"],
                                             extra=extra, device=c.dev, dtype=td))
    in_bytes = sum(sum(t.numel() * t.element_size() for t in dets) for dets in store)
    pool, P = None, 0
    if with_masks:
        # prototype maps: tile t reads map (t mod P) of a pool P x 8.4 MB (fp32) >> L2, rows [P, P + bs) repeat rows
        # [0, bs) so that a batch is always one contiguous slice.  (The unique maps of 11 025 tiles would take 92 GB
        # next to 117 GB of logits.)  The mapping is by GLOBAL tile index: the same for every number of ranks.
        P = max(bs, min(args.proto_pool, n_tiles))
        pool = torch.empty((P + bs, NM, mh, mh), dtype=td, device=c.dev)
        for p0 in range(0, P, 64):
            p1 = min(p0 + 64, P)
            pool[p0:p1] = synth.slide_tile_protos(p1 - p0, tile, seed=1, first_tile=p0, nm=NM, device=c.dev, dtype=td)
        pool[P:] = pool[:bs]
        in_bytes += (t1 - t0) * NM * mh * mh * esz

    def provider(a, b):
        return store[(a - t0) // bs]

    def protos(a, b):
        return pool[a % P:a % P + (b - a)]

    res = {}

    def step(i):
        res.pop("r", None)              # the previous slide's results are released before the next ones are allocated
        res["r"] = post.run(provider, ordered=True, proto_provider=protos if with_masks else None,
                            mask_words_per_row=40.0)

    for i in range(max(warmup, 3)):     # the slide-sized temporaries settle in the caching allocator after ~3 passes
        step(i)
    if with_masks:
        res["r"]["masks"].check()
    ops.profile.reset()
    ms = c.timed(step, steps)
    launches = ops.profile.launches
    r = res["r"]
    n_local = int(r["n"])
    if dump and c.rank == 0:        # this rank's survivors in score order, their masks by slide row
        dump_outputs(dump, r["boxes"], r["scores"], r["labels"], r["index"] - int(r["base"]),
                     r["masks"] if with_masks else None,
                     {"counts": np.array([n_local, int(r["boxes"].shape[0])], dtype=np.float64)})
    seam_rows, exchanges = r.get("seam_rows"), r.get("exchanges")
    dg = kept_digest(r["state"], r["base"])
    words_local = int(r["masks"].offsets[n_local]) if with_masks else 0
    md = mask_digest(r["masks"], r["state"], r["base"]) if with_masks else torch.zeros_like(dg)
    del r
    res.clear()                         # the phases below allocate their own results: release the slide's first
    # phases (each timed alone, max over ranks)
    reps = max(2, min(steps, 3))
    ms_detect = _timed_phase(c, lambda: post.detect(provider, keep_batches=with_masks), reps)

    def merge_only():
        res.pop("m", None)
        res["m"] = post.merge(ordered=True)

    ms_merge = _timed_phase(c, merge_only, reps)
    ms_masks = _timed_phase(c, lambda: post.masks(protos, res["m"]["state"], words_per_row=40.0), reps) \
        if with_masks else 0.0
    res.clear()
    cand_local = 0
    stages = None
    if want_stages:
        # per-call CUDA-event times of one more (untimed) pass: every C-ABI call bracketed by events on its stream
        ns, post.n_streams = post.n_streams, 1       # one stream: a call's events then bracket its own kernels only
        ops.profile.enabled = True
        ops.profile.reset()
        step(0)
        prof = ops.profile.summary()
        ops.profile.enabled = False
        post.n_streams = ns
        res.clear()
        stages = {k: {"calls": n, "ms_total": t} for k, (n, t) in prof.items()}
        cand_local = int(sum(int(b[2].cand_counts[:-1].sum()) for b in post._batches)) if post._batches else 0
    cpu_merge = None
    if want_cpu_merge and c.rank == 0 and c.world == 1:
        try:   # a reported baseline must never take the GPU record down with it
            n_cols = int((post.rois[:, 1] == post.rois[0, 1]).sum())        # tiles in the first grid row
            tl = post.acc.tile[:n_local]
            tl = torch.where(tl >= 0, tl, ~tl).to(torch.int64)              # fragile rows carry ~tile
            sub = ((tl // n_cols) < 8) & ((tl % n_cols) < 8)      # the largest sub-slide cpu_merge_scaling may time
            cpu_merge = cpu_merge_scaling(post.acc.boxes[:n_local][sub].cpu(), post.acc.scores[:n_local][sub].cpu(),
                                          tl[sub].cpu(), n_cols, wl["conf"], wl["iou"], budget_s=12.0)
        except Exception as e:   # noqa: BLE001
            cpu_merge = {"error": f"{type(e).__name__}: {e}"}
    tot = torch.cat([torch.tensor([n_local, in_bytes, cand_local, words_local], dtype=torch.int64, device=c.dev), dg, md])
    if c.world > 1:
        import torch.distributed as dist
        dist.all_reduce(tot)
    n_all, in_all, cand_all, words_all = [int(v) for v in tot[:4].tolist()]
    digest, mdigest = fold_digest(tot[4:7]), fold_digest(tot[7:10])
    kept_all = digest["kept"]
    N_rows = spec.rows_per_tile(synth.level_shapes(tile, synth.STRIDES_3))
    alg = {   # algorithmic bytes of ONE slide, all ranks together (DESIGN.md 3): totals over all launches of a call
        "hdy_filter_compact_logits": n_tiles * esz * N_rows * spec.no + 24 * cand_all,
        "hdy_nms_tiles": 24 * cand_all + 29 * n_all,
        "hdy_gather_select_logits": n_all * ((esz + 4) * (1 + nc + extra) + 4 + 4 + 8),
        "hdy_merge_append": n_all * (29 + 32),
        "hdy_merge_nms": n_all * (28 + 1),
        "hdy_seam_build": n_all * (28 + 1),
        "hdy_merge_select_ordered": n_all + 8 * kept_all,
        "hdy_sort_keys_bytes": kept_all * 8 * 2 * 4,
        "hdy_merge_gather": kept_all * (8 + 28 + 36),
        "hdy_process_mask_geometry": n_all * (16 + 1) + n_tiles * wl["cap"] * 24,
        "hdy_process_mask_rows": n_all * (24 + 24),
        "hdy_process_mask_packed": n_tiles * esz * NM * mh * mh + kept_all * (4 * NM + 16 + 24) + 4 * words_all,
    }
    step_bytes = sum(v for k, v in alg.items() if stages is None or k in stages)
    peak, peak_src = load_peak()
    out = {"tiles": n_tiles, "tiles_per_s": n_tiles * steps / (ms * 1e-3), "ms_per_slide": ms / steps,
           "detect_ms": ms_detect, "merge_ms": ms_merge, "masks_ms": ms_masks, "detections": n_all, "kept": kept_all,
           "candidates": cand_all, "mask_words": words_all, "digest": digest, "mask_digest": mdigest,
           "input_bytes": in_all, "slide_px": S, "tile": tile, "overlap": wl["overlap"], "dtype_in": args.dtype,
           "masks": masks, "proto_pool": P,
           "seam_rows": seam_rows, "exchanges": exchanges, "gpu_launches": launches,
           "boxes_per_s": cand_all * steps / (ms * 1e-3) if cand_all else n_all * steps / (ms * 1e-3),
           "pipeline": {"algorithmic_bytes_per_step": step_bytes,
                        "achieved_gbs": step_bytes / (ms / steps * 1e-3) / 1e9 / c.world,
                        "frac_of_peak": step_bytes / (ms / steps * 1e-3) / 1e9 / c.world / peak,
                        "note": "per GPU: the slide's algorithmic bytes / ranks / time, against one GPU's HBM peak"}}
    if stages is not None:
        for k, v in stages.items():     # rank 0's calls process 1/world of the slide's bytes
            a_b = alg.get(k)
            v["alg_bytes_total"] = (a_b / c.world) if a_b else None
            v["gbs"] = (a_b / c.world / (v["ms_total"] * 1e-3) / 1e9) if a_b and v["ms_total"] > 0 else None
            v["ms"] = v["ms_total"] / max(v["calls"], 1)
        out["stages"] = stages
        hbm = [k for k in stages if k in ("hdy_filter_compact_logits", "hdy_process_mask_packed")]
        if hbm:
            dom = max(hbm, key=lambda k: stages[k]["ms_total"])
            calls, t_tot = stages[dom]["calls"], stages[dom]["ms_total"]
            per_launch = alg[dom] / c.world / calls
            ach = per_launch / (t_tot / calls * 1e-3) / 1e9
            traffic = None
            try:   # DRAM bytes per launch of the dominant call, from the committed ncu --set full capture
                traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["slide"][dom]["bytes"]
            except Exception:
                pass
            out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                               "frac": ach / peak, "frac_of_nominal_8000": ach / 8000.0, "traffic": traffic,
                               "peak_source": peak_src, "algorithmic_bytes_per_launch": per_launch,
                               "kernel_ms": t_tot / calls, "launches_per_step": calls}
    if cpu_merge is not None:
        out["cpu_merge"] = cpu_merge
    if want_e2e:
        # host-resident head outputs: every batch is copied H2D inside the timed region (4 pinned host batches are
        # reused in rotation, bytes are counted for every copy), the slide's survivors and their masks are read back
        nrot = min(4, len(store))
        host = [[t.cpu().pin_memory() for t in store[k]] for k in range(nrot)]
        nst = max(1, args.slide_streams)
        stg = [[torch.empty_like(t) for t in store[0]] for _ in range(nst)]
        host_p = [pool[k * bs:(k + 1) * bs].cpu().pin_memory() for k in range(min(4, P // bs))] if with_masks else None
        stg_p = [torch.empty_like(pool[:bs]) for _ in range(nst)] if with_masks else None   # one per stream

        def provider_h(a, b):
            k = ((a - t0) // bs)
            src = host[k % nrot]
            stage = stg[k % nst]
            n = b - a
            for s_, h in zip(stage, src):
                s_[:n].copy_(h[:n], non_blocking=True)
            return [s_[:n] for s_ in stage] if n < bs else stage

        def protos_h(a, b):
            k = ((a - t0) // bs)
            n = b - a
            sp = stg_p[k % nst]               # batch k runs on stream k % streams (SlidePostprocessor.masks)
            sp[:n].copy_(host_p[k % len(host_p)][:n], non_blocking=True)
            return sp[:n]

        hb, pinned = {}, {}

        def back(k, t):
            # results are read back into pinned host buffers that persist across slides (a pageable .cpu() of
            # ~1 GB costs more than the whole H2D stream: fresh pages + a staged copy)
            buf = pinned.get(k)
            if buf is None or buf.shape[0] < t.shape[0]:
                buf = torch.empty((int(t.shape[0] * 1.05) + 1,) + tuple(t.shape[1:]), dtype=t.dtype).pin_memory()
                pinned[k] = buf
            buf[:t.shape[0]].copy_(t, non_blocking=True)
            hb[k] = buf[:t.shape[0]]

        def e2e_step(i):
            rr = post.run(provider_h, ordered=True, proto_provider=protos_h if with_masks else None,
                          mask_words_per_row=40.0)
            for k in ("boxes", "scores", "labels", "index"):
                back(k, rr[k])
            if with_masks:
                pm = rr["masks"]
                back("mask_geom", pm.geom)
                back("mask_offsets", pm.offsets)
                back("mask_bits", pm.bits[:words_local + 1])

        e2e_step(0)
        Ke = max(1, min(steps, 2))
        ms_e = c.timed(e2e_step, Ke)
        d2h = torch.tensor([sum(t.numel() * t.element_size() for t in hb.values()), in_bytes], dtype=torch.int64,
                           device=c.dev)
        if c.world > 1:
            import torch.distributed as dist
            dist.all_reduce(d2h)
        out["e2e"] = {"value": n_tiles * Ke / (ms_e * 1e-3), "unit": "tiles/s", "h2d_bytes_per_step": int(d2h[1]),
                      "d2h_bytes_per_step": int(d2h[0]), "steps": Ke, "ms_per_step": ms_e / Ke}
        del host, stg, host_p, stg_p, pinned, hb
    del store, pool
    post._batches = []
    res.clear()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ main
def main():
    args = parse()
    _protect_stdout()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    c = make_ctx(args)
    peak, peak_src = load_peak()
    masks = args.masks

    if args.workload == "slide":
        if masks == "paste":
            raise SystemExit("--workload slide takes --masks proto or none")
        sampler = ClockSampler(c.local)
        sampler.start()
        s = run_slide(args, wl, c, args.steps, args.warmup, want_e2e=not args.no_e2e,
                      want_cpu_merge=not args.no_cpu_baseline, masks=masks, dump=args.dump_outputs)
        clocks = sampler.stop()
        cfg = common_config(args, wl, masks)
        cfg.update({"tiles": s["tiles"], "tiles_per_step_per_gpu": s["tiles"] / c.world, "detections": s["detections"],
                    "kept": s["kept"], "digest": s["digest"], "mask_digest": s["mask_digest"],
                    "stages": "per tile: decode+filter+compact, nms, score/label select; append in slide coordinates; "
                              "exact slide-level merge NMS (4 all-gathers of fixed-size seam blocks over NCCL when "
                              "N>1)" + ("; process_mask (proto contraction, sigmoid, crop, upsample, >0.5, bit-packed) "
                                        "for the KEPT rows" if masks == "proto" else ""),
                    "l2": f"{s['input_bytes'] / 1e9:.1f} GB of head outputs resident in HBM, each read once per step" +
                          (f" (prototype maps: tile t reads map t mod {s['proto_pool']})" if masks == "proto" else ""),
                    "launch": f"tile batches of {wl['bs']} alternate over {args.slide_streams} streams "
                              "(SlidePostprocessor(streams=)), appends chained by events"})
        line = {
            "metric": "postproc_tiles_per_s", "value": s["tiles_per_s"], "unit": "tiles/s", "n_gpus": c.world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": s["ms_per_slide"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "boxes_per_s": s["boxes_per_s"], "roofline": s.get("roofline"), "stages": s.get("stages"),
            "pipeline": s["pipeline"], "slide": {k: v for k, v in s.items() if k not in ("stages", "roofline", "e2e")},
            "e2e": s.get("e2e"), "gpu_launches": s["gpu_launches"], "clocks": clocks,
        }
        if not args.no_sub and args.dtype == "f32":
            # the same slide with fp16 head outputs -- what the reference's GPU path hands over (half=True,
            # val_nuclei.py:109,115-116); widened on load, fp32 arithmetic: half the HBM and PCIe bytes
            hargs = argparse.Namespace(**vars(args))
            hargs.dtype = "f16"
            h = run_slide(hargs, wl, c, 2, 2, want_e2e=not args.no_e2e, want_cpu_merge=False, masks=masks,
                          want_stages=False)
            line["slide_f16"] = {k: h[k] for k in ("tiles_per_s", "ms_per_slide", "detect_ms", "merge_ms", "masks_ms",
                                                   "kept", "digest", "mask_digest", "input_bytes", "pipeline", "e2e")
                                 if k in h}
        if not args.no_sub:
            for name, st, wu in (("tiles640", 100, 10), ("tiles1024", 40, 5)):
                targs = argparse.Namespace(**vars(args))
                targs.workload, targs.steps, targs.warmup, targs.no_e2e, targs.no_sub = name, st, wu, True, True
                t = run_tiles(targs, WORKLOADS[name], c)
                line[name] = {k: t[k] for k in ("value", "unit", "ms_per_step", "boxes_per_s", "roofline", "stages",
                                                "pipeline", "gpu_launches", "config")}
            if c.rank == 0:
                try:   # SURVEY 8f rank 1: the gather in front of the mask head, exact order vs tensor cores (DESIGN 3.8b)
                    from tools.roi_bench import run_roi
                    torch.cuda.empty_cache()
                    line["roi_align"] = run_roi(dev=c.dev, with_torchvision=False)
                except Exception as e:   # noqa: BLE001  (a sub-record must never take the line down)
                    line["roi_align"] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()
    elif args.workload == "hnet":
        from tools.hnet_bench import run_hnet     # configs[4]: kept in its own file
        line = run_hnet(args, wl, c, common_config, load_peak, ClockSampler)
    else:
        line = run_tiles(args, wl, c, dump=args.dump_outputs)
        if not args.no_sub:
            sargs = argparse.Namespace(**vars(args))
            line["slide"] = run_slide(sargs, WORKLOADS["slide"], c, steps=3, warmup=2, want_e2e=False,
                                      want_cpu_merge=False, masks="proto" if masks == "proto" else "none",
                                      want_stages=False)

    try:   # the CPU legs use every core the process started with, not just the GPU's NUMA node
        os.sched_setaffinity(0, _ORIG_AFFINITY)
    except Exception:
        pass
    wk = args.workload if args.workload != "hnet" else "tiles1024"
    if c.rank == 0 and not args.no_torch_cuda:
        try:   # diagnostics must never take the record down
            line["torch_cuda"] = time_torch_cuda(wk, wl, masks, args.dtype, c.dev,
                                                 n_tiles=2 if wl["tile"] >= 1024 else 8, slide_size=args.slide_size)
        except Exception as e:   # noqa: BLE001
            line["torch_cuda"] = {"error": f"{type(e).__name__}: {e}"}
        torch.cuda.empty_cache()
    cpu = None
    if c.rank == 0 and not args.no_cpu_baseline:
        try:
            cpu = time_cpu(wk, wl, masks, budget_s=25.0, max_passes=20, dtype=args.dtype, slide_size=args.slide_size)
            # the reference's own mask path (variant A) beside it, and its own thread cap: min(8, ncpu - 1)
            # (metayolo/__init__.py:21,31)
            if masks == "proto":
                p = time_cpu(wk, wl, "paste", budget_s=1.0, max_passes=1, dtype=args.dtype, n_tiles=1,
                             slide_size=args.slide_size)
                cpu["paste_variant"] = {"value": p["value"], "ms_per_pass": p["ms_per_pass"], "tiles_per_pass": 1}
            t8 = min(8, max(1, (os.cpu_count() or 2) - 1))
            p8 = time_cpu(wk, wl, "none", budget_s=3.0, max_passes=3, threads=t8, dtype=args.dtype,
                          slide_size=args.slide_size)
            cpu["no_masks_reference_threads"] = {"value": p8["value"], "threads": p8["cores"]}
        except Exception as e:   # noqa: BLE001
            cpu = {"error": f"{type(e).__name__}: {e}", "kind": "port"}
    line["cpu_baseline"] = cpu
    if isinstance(line.get("e2e"), dict):
        line["e2e"]["host_affinity"] = c.affinity
    if c.rank == 0:
        _emit(line)
    if c.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
