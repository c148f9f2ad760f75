"""ORACLE (test infrastructure): the seeded cases of tests/test_oracle_vs_reference.py and their stored answers.

Every case builds its inputs from a fixed seed and runs them through an implementation with the signatures of
oracle/port.py (``port`` itself, or ``reference_impl(ref_shim.load())``).  ``python -m oracle.live_cases SOURCE``
(SOURCE = reference | port) stores, for every input and output tensor of every case, a SHA-256 of its dtype, shape
and bytes in tests/golden/live_cases.npz, with SOURCE beside them: a bit-exact record that takes a few KB where the
tensors themselves (random fp32 boxes and IoU matrices) would take ~0.4 MB.

The stored file was written with SOURCE = port: the reference tree was not available when it was written.  Cases
nms_*, box_* and merge_* are the inputs on which the live test compared the port with the reference bit for bit when
that test was added (f185083); oracle/port.py has not changed since (last change ab6dfbb).  Case proposals_* takes new
inputs: the live test used to draw its inputs after building the reference's Detect module, so they depended on that
module's weight initialisation; compute_proposals is also pinned on the reference's own outputs in
tests/golden/detect_*.npz.
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch

from hd_yolo_b200 import synth

NMS_CASES = [(0, 3000, 4, 0.2), (1, 800, 7, 0.05), (2, 50, 1, 0.5)]
YOLO_KW = [dict(), dict(agnostic=True), dict(multi_label=True), dict(classes=[0])]
SCALE_CASES = [((640, 640), (480, 720), None), ((320, 512), (777, 333), ((0.5, 0.5), (10.0, 20.0)))]
SCAN_CASES = [((3000, 2500), (1024, 1024), 64), ((700, 900), (512, 512), 0), ((100000, 100000), (1024, 1024), 64)]
MERGE_PARAMS = {'conf_thres': 0.3, 'iou_thres': 0.45, 'max_det': 500}
GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "live_cases.npz")


def digest(t: torch.Tensor) -> np.ndarray:
    """SHA-256 of dtype, shape and bytes: equal digests <=> the same tensor bit for bit."""
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.view(torch.uint8).numpy().tobytes() if t.numel() else b"")
    return np.frombuffer(h.digest(), dtype=np.uint8)


def reference_impl(ref):
    """The reference's functions (ref_shim.load()) behind oracle/port.py's signatures."""
    def compute_proposals(dets, anchors, strides):
        det = ref.Detect(ch=[8] * len(strides), anchors=anchors, strides=strides, nc=dets[0].shape[-1] - 5, masks={},
                         is_scripting=True)
        det.eval()
        with torch.no_grad():
            return det.compute_proposals([d.clone() for d in dets])

    return types.SimpleNamespace(
        nms_per_image=lambda p, nc, conf, iou, md: ref.nms_per_image(p, nc, conf_thres=conf, iou_thres=iou, max_det=md),
        non_max_suppression=ref.non_max_suppression, box_iou=ref.box_iou, xywh2xyxy=ref.xywh2xyxy,
        scale_coords=ref.scale_coords, sliding_window_scanner=ref.sliding_window_scanner,
        merge_outputs=lambda tiles: ref.Detect.merge_outputs(None, tiles),
        ensemble_merge=lambda parts, params: ref.Ensemble([], nms_params=params).merge(parts),
        compute_proposals=compute_proposals)


def nms_case(impl, seed, n, nc, conf):
    g = torch.Generator().manual_seed(seed)
    c = torch.rand((2, n, 2), generator=g) * 600
    wh = torch.rand((2, n, 2), generator=g) * 40 + 1
    sc = torch.rand((2, n, 1 + nc), generator=g)
    extra = torch.rand((2, n, 2), generator=g)
    preds = torch.cat([c, wh, sc, extra], -1)
    y5 = torch.cat([c, wh, sc], -1)
    out = {f"nms{seed}_in_preds": preds}
    for i, r in enumerate(impl.nms_per_image(preds.clone(), nc, conf, 0.45, 300)):
        out.update({f"nms{seed}_npi{i}_{k}": r[k] for k in ("boxes", "scores", "extra")})
    for j, kw in enumerate(YOLO_KW):
        for i, r in enumerate(impl.non_max_suppression(y5.clone(), conf, 0.45, max_det=300, **kw)):
            out[f"nms{seed}_yolo{j}_{i}"] = r
    return out


def box_case(impl):
    g = torch.Generator().manual_seed(5)
    a = torch.rand((300, 4), generator=g) * 500
    b = torch.rand((200, 4), generator=g) * 500
    a[:, 2:] += a[:, :2]
    b[:, 2:] += b[:, :2]
    out = {"box_in_a": a, "box_in_b": b, "box_iou": impl.box_iou(a, b), "box_xywh2xyxy": impl.xywh2xyxy(a)}
    for i, (img1, img0, rp) in enumerate(SCALE_CASES):
        out[f"box_scale{i}"] = impl.scale_coords(img1, a.clone(), img0, rp)
    return out


def merge_case(impl):
    out = {f"merge_scan{i}": impl.sliding_window_scanner(*c) for i, c in enumerate(SCAN_CASES)}
    g = torch.Generator().manual_seed(9)
    tiles = []
    for t in range(6):
        k = 150
        c = torch.rand((k, 2), generator=g) * 512
        wh = torch.rand((k, 2), generator=g) * 30 + 8
        tiles.append({'boxes': torch.cat([c - wh / 2, c + wh / 2], 1), 'scores': torch.rand((k,), generator=g),
                      'labels': torch.randint(1, 5, (k,), generator=g),
                      'roi': torch.tensor([(t % 3) * 448.0, (t // 3) * 448.0, 0.0, 0.0])})
    for t, d in enumerate(tiles):
        out.update({f"merge_in{t}_{k}": d[k] for k in ("boxes", "scores", "labels")})
    m = impl.merge_outputs([{k: (v.clone() if torch.is_tensor(v) else v) for k, v in t.items()} for t in tiles])
    e = impl.ensemble_merge([{'det': m}], dict(MERGE_PARAMS))['det']
    for k in ("boxes", "scores", "labels"):
        out[f"merge_tiles_{k}"], out[f"merge_ensemble_{k}"] = m[k], e[k]
    return out


def proposals_case(impl):
    g = torch.Generator().manual_seed(3)
    dets = [torch.randn((2, 3, 160 // s, 160 // s, 5 + 4), generator=g) for s in synth.STRIDES_3]
    out = {f"proposals_in{i}": d for i, d in enumerate(dets)}
    out.update({f"proposals_out{i}": p for i, p in
                enumerate(impl.compute_proposals([d.clone() for d in dets], synth.ANCHORS_3, synth.STRIDES_3))})
    return out


def all_cases(impl):
    out = {}
    for c in NMS_CASES:
        out.update(nms_case(impl, *c))
    for case in (box_case, merge_case, proposals_case):
        out.update(case(impl))
    return out


def main(argv):
    if argv[1:] not in (["reference"], ["port"]):
        raise SystemExit("usage: python -m oracle.live_cases reference|port")
    if argv[1] == "reference":
        from . import ref_shim
        impl = reference_impl(ref_shim.load())
    else:
        from . import port as impl
    arrays = {k: digest(v) for k, v in all_cases(impl).items()}
    np.savez_compressed(GOLDEN, source=np.array(argv[1]), **arrays)
    print(f"{GOLDEN}: {len(arrays)} tensors from the {argv[1]}, {os.path.getsize(GOLDEN)} bytes")


if __name__ == "__main__":
    main(sys.argv)
