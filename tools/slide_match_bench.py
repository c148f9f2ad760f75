"""Times binned matching (match_predictions(..., binned=True)) at slide scale: ~2.85e7 predictions against a
ground-truth field of the same size, both from hd_yolo_b200.synth.slide_nuclei (the global nuclei field of
slide_tile_logits, pitch 18.7 px, over a ~99 840^2 px region; predictions are the field jittered by up to 2 px).
Both plane sets are GBs, far larger than L2: every pass reads HBM.

Reported, after one warm-up call of each form, over five calls: CUDA-event times of every library call
(hd_yolo_b200.ops.profile) and of the whole match_predictions call, the caching allocator's segment allocations and
frees in each call, and (one more call under torch.profiler) the host operations that take the most CPU time, for ground-truth binning (hdy_match_bin_* + the cell sort), the box pass and the
mask pass; the algorithmic bytes of each, computed from the shapes below (each input read once, each output written
once); and the share of the 7.7 TB/s data-sheet HBM bound that gives.  The card's name and power limit are read in the
same run.

Usage: python tools/slide_match_bench.py OUTDIR [side_px]   -> OUTDIR/slide_match_bench.json"""
import json
import os
import subprocess
import sys
from collections import defaultdict

import torch

HBM_PEAK_GBS = 7700.0       # B200 data sheet (HGX B200, one GPU); not a measured figure


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


_ALLOC_KEYS = ("segment.all.allocated", "segment.all.freed", "num_alloc_retries", "num_device_alloc",
               "num_device_free")


def _alloc_counts(dev):
    st = torch.cuda.memory_stats(dev)
    return {k: st.get(k, 0) for k in _ALLOC_KEYS}


def _host_time_by_op(fn, dev, top=8):
    """CPU self time of the slowest host-side operations of one fn() call (torch.profiler, CPU and CUDA activities):
    where time outside the kernels goes (cudaMalloc / cudaFree of the caching allocator, synchronising reads)."""
    from torch.profiler import ProfilerActivity, profile as tprof
    torch.cuda.synchronize(dev)
    with tprof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize(dev)
    ev = sorted(prof.key_averages(), key=lambda e: -e.self_cpu_time_total)[:top]
    return [{"op": e.key, "calls": e.count, "self_cpu_ms": e.self_cpu_time_total / 1e3} for e in ev]


def _profiled(fn, dev):
    """fn() once with per-call CUDA events on; returns (result, total ms, {entry point: ms}, allocator deltas)."""
    from hd_yolo_b200.ops import profile
    torch.cuda.synchronize(dev)
    before = _alloc_counts(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profile.records.clear()
    profile.enabled = True
    a.record()
    res = fn()
    b.record()
    profile.enabled = False
    torch.cuda.synchronize(dev)
    per = defaultdict(float)
    for name, s, e in profile.records:
        per[name] += s.elapsed_time(e)
    profile.records.clear()
    after = _alloc_counts(dev)
    return res, a.elapsed_time(b), dict(per), {k: after[k] - before[k] for k in _ALLOC_KEYS}


def run(out_dir, side=99840):
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import synth
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rec = {"card": _card(), "hbm_peak_GBs_datasheet": HBM_PEAK_GBS, "region_px": [side, side]}
    region = (0, 0, side, side)
    gt = synth.slide_nuclei(region, device=dev)
    pred = synth.slide_nuclei(region, jitter=2.0, seed=1, device=dev)
    pred['scores'] = (pred['scores'] * 4096).round() / 4096
    P, G = len(pred['boxes']), len(gt['boxes'])
    pw, gw = int(pred['masks'].offsets[-1]), int(gt['masks'].offsets[-1])
    rec.update({"P": P, "G": G, "pred_plane_GB": pw * 4 / 1e9, "gt_plane_GB": gw * 4 / 1e9})
    torch.cuda.synchronize(dev)
    # bytes each pass must move at least: its inputs once, its outputs once
    box_in = 16 * (P + G) + 4 * P
    mask_in = 4 * (pw + gw) + (16 + 8 + 4) * (P + G) + 4 * P     # planes, geom + offsets + areas, rank order
    for iou_type in ('boxes', 'masks'):
        f = lambda: hdy.match_predictions(pred, gt, 0.5, iou_type=iou_type, binned=True)
        f()                                                          # warm-up
        runs = []
        for _ in range(5):
            m, total, per, alloc = _profiled(f, dev)
            runs.append((total, per, alloc))
        n = int(m['ious'].shape[0])
        binning = sum(v for k, v in per.items() if k.startswith("hdy_match_bin_"))
        passes = {k: v for k, v in per.items() if not k.startswith("hdy_match_bin_")}
        nbytes = (box_in if iou_type == 'boxes' else mask_in) + 16 * n
        pass_ms = sum(v for k, v in passes.items() if k in ("hdy_match_boxes_binned", "hdy_match_mask_candidates_binned",
                                                             "hdy_match_mask_exact_list"))
        rec[iou_type] = {
            "pairs": n, "call_ms_runs": [r[0] for r in runs], "kernel_ms_runs": [sum(r[1].values()) for r in runs],
            "allocator_deltas_runs": [r[2] for r in runs], "per_entry_point_ms": per,
            "host_ops_one_call": _host_time_by_op(f, dev),
            "binning_ms_without_cell_sort": binning, "pair_pass_ms": pass_ms,
            "pair_pass_algorithmic_GB": nbytes / 1e9,
            "pair_pass_share_of_hbm_bound": nbytes / (pass_ms * 1e-3) / (HBM_PEAK_GBS * 1e9),
        }
        del m
    gb_bin = 16 * G * 3 + 8 * 4 * G                                 # three reads of the boxes, ~4 entries per nucleus
    rec["binning_algorithmic_GB_estimate"] = gb_bin / 1e9
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "slide_match_bench.json"), "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    run(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 99840)
