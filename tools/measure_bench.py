"""Times PackedMasks.measure() at slide scale: the ~2.85e7 nuclei of hd_yolo_b200.synth.slide_nuclei over a ~99 840^2 px
region (tight windows, 12-30 px ellipses).  The planes are GBs, far larger than L2: every pass reads HBM.

Reported, after one warm-up call, over five calls: the CUDA-event time of hdy_mask_measure (hd_yolo_b200.ops.profile)
and, in the same run on the same planes, of hdy_mask_areas (the plane-read floor: one popcount pass); the time of the
whole measure() call (its one 4-byte device->host read and the output allocations included) and of columns(); the
algorithmic bytes of hdy_mask_measure, computed from the shapes below (planes, windows and offsets read once, 116 B of
exact fields written per mask), and the share of the 7.7 TB/s data-sheet HBM bound that gives.  The card's name and
power limit are read in the same run.

Time breakdown: csrc/measure.cu built with -DHDY_MEASURE_STAGES=1 runs only the sums and corner patterns of the small
path, with =2 also the two hull chains (the library is 3: also the hull, the calipers and the perimeter).  Build such a
library with ``HDY_NVCC_EXTRA=-DHDY_MEASURE_STAGES=n bash hd_yolo_b200/csrc/build.sh`` and pass a tag, so that its
record goes to a file of its own; only its kernel times mean anything, its hull fields are not written.

Usage: python tools/measure_bench.py OUTDIR [side_px] [tag]   -> OUTDIR/r08_measure_bench[_tag].json"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from contour_bench import HBM_PEAK_GBS, _card, _profiled  # noqa: E402

FIELD_BYTES = 4 + 16 + 40 + 16 + 24 + 16        # area, bbox, moments, quads, hull, hull_len per mask


def run(out_dir, side=99840, tag=""):
    import hd_yolo_b200 as hdy  # noqa: F401
    from hd_yolo_b200 import synth
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rec = {"card": _card(), "hbm_peak_GBs_datasheet": HBM_PEAK_GBS, "region_px": [side, side], "build": tag or "library"}
    pm = synth.slide_nuclei((0, 0, side, side), device=dev)['masks']
    K, words = len(pm), int(pm.offsets[-1])
    rec.update({"masks": K, "plane_GB": words * 4 / 1e9})
    m = pm.measure()                                                 # warm-up
    m.columns()
    pm.areas()
    del m
    runs = []
    for _ in range(5):
        m, total, per = _profiled(pm.measure, dev)
        _, cols_ms, _ = _profiled(m.columns, dev)
        _, _, per_a = _profiled(pm.areas, dev)
        runs.append({"measure_call_ms": total, "columns_ms": cols_ms, "hdy_mask_measure_ms": per["hdy_mask_measure"],
                     "hdy_mask_areas_ms": per_a["hdy_mask_areas"]})
        del m
    nbytes = 4 * words + (16 + 8) * K + FIELD_BYTES * K
    best = min(r["hdy_mask_measure_ms"] for r in runs)
    best_a = min(r["hdy_mask_areas_ms"] for r in runs)
    rec.update({
        "runs": runs, "best_hdy_mask_measure_ms": best, "best_hdy_mask_areas_ms": best_a,
        "measure_over_areas": best / best_a, "algorithmic_GB": nbytes / 1e9,
        "share_of_hbm_bound_best_run": nbytes / (best * 1e-3) / (HBM_PEAK_GBS * 1e9),
    })
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "r08_measure_bench" + (f"_{tag}" if tag else "") + ".json"), "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    run(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 99840, sys.argv[3] if len(sys.argv) > 3 else "")
