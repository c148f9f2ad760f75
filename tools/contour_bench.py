"""Times PackedMasks.contours() at slide scale: the ~2.85e7 nuclei of hd_yolo_b200.synth.slide_nuclei over a
~99 840^2 px region (tight windows, 12-30 px ellipses).  The planes are GBs, far larger than L2: every pass reads HBM.

Reported, after one warm-up call, over five calls: the CUDA-event time of each entry point (hd_yolo_b200.ops.profile)
and of the whole contours() call (which includes the one device->host read of the totals and the output allocations);
the algorithmic bytes of each entry point, computed from the shapes below (planes, windows and offsets read once per
pass, every output written once); and the share of the 7.7 TB/s data-sheet HBM bound that gives.  Also, measured on the
host: save_geojson's time and file size for a region of ~1e5 nuclei.  The card's name and power limit are read in the
same run.

Usage: python tools/contour_bench.py OUTDIR [side_px]   -> OUTDIR/contour_bench.json"""
import json
import os
import subprocess
import sys
import tempfile
import time
from collections import defaultdict

import torch

HBM_PEAK_GBS = 7700.0       # B200 data sheet (HGX B200, one GPU); not a measured figure


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def _profiled(fn, dev):
    """fn() once with per-call CUDA events on; returns (result, total ms, {entry point: ms})."""
    from hd_yolo_b200.ops import profile
    torch.cuda.synchronize(dev)
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
    return res, a.elapsed_time(b), dict(per)


def run(out_dir, side=99840):
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import synth
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rec = {"card": _card(), "hbm_peak_GBs_datasheet": HBM_PEAK_GBS, "region_px": [side, side]}
    pm = synth.slide_nuclei((0, 0, side, side), device=dev)['masks']
    K, words = len(pm), int(pm.offsets[-1])
    rec.update({"masks": K, "plane_GB": words * 4 / 1e9})
    f = pm.contours
    c = f()                                                          # warm-up
    R, V = int(c.mask_rings[-1]), int(c.xy.shape[0])
    del c
    runs = []
    for _ in range(5):
        c, total, per = _profiled(f, dev)
        runs.append((total, per))
        del c
    # bytes each entry point must move at least: planes + windows + offsets once, its outputs once
    planes = 4 * words + (16 + 8) * K
    nbytes = {"hdy_mask_contour_sizes": planes + 16 * (K + 1),
              "hdy_mask_contours": planes + 16 * (K + 1) + 8 * (R + 1) + 4 * R + 8 * V}
    best = {k: min(r[1][k] for r in runs) for k in nbytes}
    rec.update({
        "rings": R, "vertices": V, "vertices_per_mask": V / K,
        "call_ms_runs": [r[0] for r in runs], "kernel_ms_runs": [sum(r[1].values()) for r in runs],
        "per_entry_point_ms_runs": [r[1] for r in runs],
        "algorithmic_GB": {k: v / 1e9 for k, v in nbytes.items()},
        "share_of_hbm_bound_best_run": {k: nbytes[k] / (best[k] * 1e-3) / (HBM_PEAK_GBS * 1e9) for k in nbytes},
    })
    del pm
    torch.cuda.empty_cache()
    # GeoJSON of a region of ~1e5 nuclei: host time of the writer only (the contours are traced before)
    reg = synth.slide_nuclei((0, 0, 5914, 5914), device=dev)
    rc = reg['masks'].contours()
    torch.cuda.synchronize(dev)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "region.geojson")
        t0 = time.perf_counter()
        n = hdy.save_geojson(path, reg, rc)
        dt = time.perf_counter() - t0
        size = os.path.getsize(path)
    rec["geojson_region"] = {"nuclei": len(reg['masks']), "features": n, "vertices": int(rc.xy.shape[0]),
                             "host_s": dt, "bytes": size, "MB_per_s": size / dt / 1e6}
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "contour_bench.json"), "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    run(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 99840)
