"""Times matching by mask IoU at the scale of a crowded 1024-px tile: k = g = 3 000 nuclei (filled ellipses 12-36 px
across, hd_yolo_b200.synth.nuclei_match_case; predictions are jittered copies of the ground truth plus false
positives).  CUDA events, warm-up, dense inputs (3.1-12.6 GB) far larger than L2; the packed planes (~1 MB) are not.

  * PackedMasks.from_dense on fp32 and uint8 masks: the geometry pass alone (reads every dense byte once: HBM-bound)
    and the whole call (+ the bit pass and one 8-byte host read), as GB/s of the dense bytes against the HBM peak;
  * match_predictions(iou_type='masks') from PackedMasks inputs, with its candidate and match counts;
  * the library-GPU leg a torch user would write: dense fp32 overlap matmul on CUDA (TF32 off), threshold, sort and
    where -- its pairs are compared with ours;
  * for scale, oracle/mask_match.py's matching on the CPU at a smaller stated case, and ours on the same case.

Usage: python tools/mask_match_bench.py OUTDIR [k] [size]   -> OUTDIR/mask_match_bench.json"""
import json
import os
import subprocess
import sys
import time

import torch

HBM_PEAK_GBS = 7700.0       # B200 data sheet (HGX B200, one GPU); not a measured figure


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def _timed(fn, n, dev):
    for _ in range(2):
        fn()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize(dev)
    return a.elapsed_time(b) / n


def torch_match(pred, gt, scores, iou_min=0.5):
    """Dense fp32 masks on CUDA, the way a torch user would match them: overlap matmul, IoU, sort, where."""
    order = torch.sort(scores, descending=True, stable=True).indices
    p, g = pred.flatten(1), gt.flatten(1)
    inter = p @ g.T
    iou = inter / (p.sum(1)[:, None] + g.sum(1)[None, :] - inter)
    iou = iou[order]
    pi, ti = torch.where(iou >= iou_min)
    ious, o2 = torch.sort(iou[pi, ti], descending=True, stable=True)
    return pi[o2], ti[o2], ious


def run(k=3000, size=1024, cpu_k=300, cpu_size=512, dev=None):
    import hd_yolo_b200 as hdy
    from hd_yolo_b200 import _lib, synth
    from hd_yolo_b200.masks import PackedMasks
    from hd_yolo_b200.metrics import _mask_pairs
    from hd_yolo_b200.ops import _call, _stream
    dev = dev if dev is not None else torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rec = {"card": _card(), "k": k, "g": k, "canvas": [size, size], "hbm_peak_GBs_datasheet": HBM_PEAK_GBS}
    out, tgt = synth.nuclei_match_case(k, k, size, seed=1, device=dev)
    torch.cuda.synchronize(dev)

    # 1. dense -> packed
    geom = torch.empty((k, 4), dtype=torch.int32, device=dev)
    offsets = torch.empty((k + 1,), dtype=torch.int64, device=dev)
    for name, dense, code in (("fp32", out['masks'].float(), _lib.HDY_F32),
                              ("uint8", out['masks'].to(torch.uint8), _lib.HDY_U8)):
        nbytes = dense.numel() * dense.element_size()
        t_geom = _timed(lambda: _call("hdy_pack_masks_geometry", dense.data_ptr(), code, k, size, size,
                                      geom.data_ptr(), offsets.data_ptr(), _stream()), 10, dev)
        t_all = _timed(lambda: PackedMasks.from_dense(dense), 10, dev)
        rec[f"from_dense_{name}"] = {
            "dense_GB": nbytes / 1e9,
            "ms_geometry_pass": t_geom, "GBs_geometry_pass": nbytes / t_geom / 1e6,
            "share_of_hbm_peak_geometry_pass": nbytes / t_geom / 1e6 / HBM_PEAK_GBS,
            "ms_whole_call": t_all, "GBs_whole_call": nbytes / t_all / 1e6}
        del dense
    pp, pg = PackedMasks.from_dense(out['masks']), PackedMasks.from_dense(tgt['masks'])
    rec["packed_MB"] = (pp.nbytes() + pg.nbytes()) / 1e6

    # 2. matching from PackedMasks inputs
    op, tp = {**out, 'masks': pp}, {**tgt, 'masks': pg}
    t_match = _timed(lambda: hdy.match_predictions(op, tp, 0.5, iou_type='masks'), 20, dev)
    got = hdy.match_predictions(op, tp, 0.5, iou_type='masks')
    order32 = got['order'].to(torch.int32).contiguous()
    _, needs = _mask_pairs(pp, pg, order32, k, k, 0.5)(max(4 * k, 1024))
    n_match, n_cand = needs.tolist()
    rec["match_predictions_masks"] = {"ms": t_match, "candidates": n_cand, "matches": n_match,
                                      "window_pairs_tested": k * k}

    # 3. the library-GPU leg on dense fp32 masks (TF32 off: exact integer sums, comparable pair for pair)
    torch.backends.cuda.matmul.allow_tf32 = False
    pf, gf = out['masks'].float(), tgt['masks'].float()
    t_torch = _timed(lambda: torch_match(pf, gf, out['scores']), 3, dev)
    pi, ti, ious = torch_match(pf, gf, out['scores'])
    rec["torch_dense_fp32_matmul"] = {
        "ms": t_torch, "dense_GB": 2 * pf.numel() * 4 / 1e9,
        "pairs_identical_to_ours": bool(torch.equal(pi, got['pred_idx']) and torch.equal(ti, got['true_idx']) and
                                        torch.equal(ious, got['ious']))}
    del pf, gf, out, tgt

    # 4. for scale: the CPU oracle on a smaller case, and ours on the same case
    from oracle import mask_match
    co, ct = synth.nuclei_match_case(cpu_k, cpu_k, cpu_size, seed=2, device="cpu")
    t0 = time.perf_counter()
    ref = mask_match.apmeter_match(co, ct, 0.5)
    t_cpu = (time.perf_counter() - t0) * 1e3
    do, dt = {a: v.to(dev) for a, v in co.items()}, {a: v.to(dev) for a, v in ct.items()}
    so, st = {**do, 'masks': PackedMasks.from_dense(do['masks'])}, {**dt, 'masks': PackedMasks.from_dense(dt['masks'])}
    t_small = _timed(lambda: hdy.match_predictions(so, st, 0.5, iou_type='masks'), 20, dev)
    small = hdy.match_predictions(so, st, 0.5, iou_type='masks')
    rec["cpu_oracle_small_case"] = {
        "k": cpu_k, "g": cpu_k, "canvas": [cpu_size, cpu_size], "threads": torch.get_num_threads(),
        "ms_cpu_oracle": t_cpu, "ms_ours_from_packed": t_small, "matches": int(len(ref[4])),
        "identical": bool(torch.equal(small['pred_idx'].cpu(), ref[2]) and torch.equal(small['ious'].cpu(), ref[4]))}
    return rec


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    outdir = sys.argv[1]
    a = [int(v) for v in sys.argv[2:4]]
    r = run(*a)
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "mask_match_bench.json"), "w") as f:
        json.dump(r, f, indent=1)
    print(json.dumps(r))
