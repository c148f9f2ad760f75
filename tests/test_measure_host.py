"""CPU tests of mask morphometry: oracle/morphology.py on known answers and against cv2 and oracle/contours.py over
random masks, MaskMeasurements' derived columns against the oracle's, save_geojson(measurements=), and the host-side
argument checks of hdy_mask_measure."""
import ctypes
import json
import math

import cv2
import numpy as np
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import _lib
from hd_yolo_b200.masks import MaskContours, MaskMeasurements, PackedMasks
from oracle import contours as oc
from oracle import morphology as om


def _mm(windows):
    """MaskMeasurements of the oracle's exact fields (CPU tensors)."""
    f = om.measure(windows)
    geom = torch.tensor([[x0, y0, m.shape[1], m.shape[0]] for x0, y0, m in windows], dtype=torch.int32).reshape(-1, 4)
    return MaskMeasurements(geom, f["area"], f["bbox"], f["moments"], f["quads"], f["hull"][:, 0],
                            f["hull"][:, 2].to(torch.int32), f["hull"][:, 1], f["hull_len"][:, 0], f["hull_len"][:, 1])


def _disc(r):
    n = 2 * r + 3
    yy, xx = np.mgrid[:n, :n]
    return np.hypot(xx + 0.5 - n / 2, yy + 0.5 - n / 2) <= r


def test_known_answers():
    px = _mm([(5, 7, np.ones((1, 1), bool))]).columns()
    want = {"area": 1, "perimeter": 4, "perimeter_smooth": 2 * math.sqrt(2), "convex_area": 1, "feret_max": math.sqrt(2),
            "feret_min": 1, "eccentricity": 0, "centroid_x": 5.5, "centroid_y": 7.5, "euler": 1, "convex_perimeter": 4,
            "major_axis": 0, "minor_axis": 0, "solidity": 1, "extent": 1}
    for k, v in want.items():
        assert float(px[k][0]) == pytest.approx(v, rel=1e-15, abs=0), k
    bar = _mm([(0, 0, np.ones((1, 3), bool))])
    c = bar.columns()
    assert bar.moments[0].tolist() == [3, 0, 5, 0, 0] and bar.quads[0].tolist() == [4, 4, 0, 0]
    assert int(bar.feret_max2[0]) == 10 and float(c["feret_min"][0]) == 1 and float(c["perimeter"][0]) == 8
    assert float(c["orientation"][0]) == 0 and float(c["eccentricity"][0]) == 1
    assert float(c["major_axis"][0]) == pytest.approx(4 * math.sqrt(2 / 3), rel=1e-15) and float(c["minor_axis"][0]) == 0
    tall = _mm([(0, 0, np.ones((3, 1), bool))]).columns()
    assert float(tall["orientation"][0]) == pytest.approx(math.pi / 2, rel=1e-15)
    sq = _mm([(0, 0, np.ones((2, 2), bool))])
    assert sq.quads[0].tolist() == [4, 4, 0, 0] and int(sq.convex_area2[0]) == 8 and int(sq.hull_verts[0]) == 4
    assert float(sq.feret_min[0]) == 2 and int(sq.feret_max2[0]) == 8
    ell = _mm([(0, 0, np.array([[1, 0], [1, 1]], bool))])
    assert ell.quads[0].tolist() == [5, 2, 1, 0] and int(ell.convex_area2[0]) == 7 and int(ell.hull_verts[0]) == 5
    assert float(ell.convex_perimeter[0]) == 6 + math.sqrt(2) and float(ell.feret_min[0]) == 2
    assert float(ell.columns()["solidity"][0]) == 6 / 7
    cb = (np.add.outer(np.arange(3), np.arange(3)) % 2 == 0)                     # four saddles
    c = _mm([(0, 0, cb)])
    assert c.quads[0].tolist() == [12, 0, 0, 4] and int(c.euler[0]) == 5 and float(c.perimeter[0]) == 20
    assert int(c.convex_area2[0]) == 18 and int(c.hull_verts[0]) == 4
    yy, xx = np.mgrid[:21, :21]
    r = np.hypot(yy - 10, xx - 10)
    ring = (r < 10) & (r >= 6) | (r < 2)                                           # a ring with an island
    c = _mm([(0, 0, ring)])
    assert int(c.euler[0]) == 1                                                     # 2 components - 1 hole
    rings, _ = oc.mask_rings(ring)
    assert float(c.perimeter[0]) == sum(np.abs(np.roll(v, -1, 0) - v).sum() for v in rings)
    for rad, lo, hi in ((6, 0.82, 0.84), (20, 0.86, 0.88)):                        # the documented disc values
        d = _mm([(0, 0, _disc(rad))]).columns()
        assert lo < float(d["circularity"][0]) < hi
        assert float(d["eccentricity"][0]) < 0.05


def test_oracle_against_cv2_and_contours():
    rng = np.random.default_rng(0)
    for _ in range(1500):
        h, w = (int(v) for v in rng.integers(1, 16, 2))
        m = rng.random((h, w)) < rng.random()
        f = om.measure_window(3, 4, m)
        if not m.any():
            assert f["area"] == 0 and f["hull"] == [0, 0, 0]
            continue
        mo = cv2.moments(m.astype(np.uint8), binaryImage=True)
        assert [mo["m00"], mo["m10"], mo["m01"], mo["m20"], mo["m02"], mo["m11"]] == \
            [f["area"]] + f["moments"][:2] + f["moments"][2:]
        ys, xs = np.nonzero(m)
        corners = np.concatenate([np.stack([xs + a, ys + b], 1) for a in (0, 1) for b in (0, 1)]).astype(np.int32)
        assert cv2.contourArea(cv2.convexHull(corners)) == f["hull"][0] / 2
        n1, n2, n3, nd = f["quads"]
        rings, parent = oc.mask_rings(m)
        assert n1 + n2 + n3 + 2 * nd == sum(int(np.abs(np.roll(v, -1, 0) - v).sum()) for v in rings)
        assert (n1 - n3 + 2 * nd) % 4 == 0
        assert (n1 - n3 + 2 * nd) // 4 == sum(p < 0 for p in parent) - sum(p >= 0 for p in parent)
        assert n1 + n3 + 2 * nd == oc.local_vertex_count(m) == sum(len(v) for v in rings)
        hull = om.convex_hull(m)
        assert len(hull) == f["hull"][2] and hull[0] == min(hull, key=lambda p: (p[1], p[0]))
        bw, bh = f["bbox"][2] - f["bbox"][0], f["bbox"][3] - f["bbox"][1]
        assert max(bw, bh) ** 2 <= f["hull"][1] <= bw * bw + bh * bh and f["hull_len"][1] <= min(bw, bh)
        assert 2 * f["area"] <= f["hull"][0] <= 2 * bw * bh


def test_derived_columns_equal_oracle():
    rng = np.random.default_rng(1)
    wins = [(int(rng.integers(0, 50)), int(rng.integers(0, 50)), rng.random((int(h), int(w))) < rng.random())
            for h, w in rng.integers(1, 30, (300, 2))]
    wins.append((2, 2, np.zeros((4, 4), bool)))
    m = _mm(wins)
    want = om.columns(om.measure(wins), m.geom)
    got = m.columns()
    assert list(got) == list(want)
    for k in want:
        g = got[k].double().numpy()
        assert np.allclose(g, want[k], rtol=1e-12, atol=1e-12 if k == "orientation" else 0, equal_nan=True), k
    assert torch.isnan(got["centroid_x"][-1]) and torch.isnan(got["solidity"][-1]) and int(got["area"][-1]) == 0


def _square_contours(n):
    sq = [[0, 0], [2, 0], [2, 2], [0, 2]]
    return MaskContours(torch.arange(n + 1, dtype=torch.int64), torch.arange(0, 4 * n + 1, 4, dtype=torch.int64),
                        torch.tensor(sq * n, dtype=torch.int32), torch.full((n,), -1, dtype=torch.int32))


def test_save_geojson_measurements(tmp_path):
    c = _square_contours(3)
    res = {"scores": torch.tensor([0.5, 0.25, 0.75])}
    plain, again = str(tmp_path / "a.geojson"), str(tmp_path / "b.geojson")
    hdy.save_geojson(plain, res, c, chunk_rows=2)
    hdy.save_geojson(again, res, c, chunk_rows=2, measurements=None)
    assert open(plain, "rb").read() == open(again, "rb").read()
    meas = {"area": torch.tensor([4, 0, 9], dtype=torch.int32),
            "solidity": torch.tensor([1.0, float("nan"), float("inf")], dtype=torch.float64)}
    path = str(tmp_path / "m.geojson")
    assert hdy.save_geojson(path, res, c, chunk_rows=2, measurements=meas) == 3
    text = open(path).read()
    assert "NaN" not in text and "Infinity" not in text
    feats = json.loads(text)["features"]
    assert [f["properties"]["measurements"] for f in feats] == [{"area": 4, "solidity": 1.0},
                                                                {"area": 0, "solidity": None},
                                                                {"area": 9, "solidity": None}]
    assert feats[0]["properties"]["score"] == 0.5
    wins = [(0, 0, np.ones((2, 2), bool)), (0, 0, np.zeros((2, 2), bool)), (0, 0, np.ones((2, 3), bool))]
    m = _mm(wins)
    hdy.save_geojson(path, res, c, measurements=m)
    props = [f["properties"]["measurements"] for f in json.load(open(path))["features"]]
    assert list(props[0]) == list(m.columns()) and props[1]["centroid_x"] is None and props[2]["area"] == 6
    with pytest.raises(hdy.HdyError):
        hdy.save_geojson(path, res, c, measurements={"area": torch.zeros(2)})


def test_measure_argument_checks():
    lib = _lib.load()
    buf = (ctypes.c_int64 * 8)()
    geom = (ctypes.c_int32 * 8)()
    mis = ctypes.c_void_p(ctypes.addressof(geom) + 4 if ctypes.addressof(geom) % 16 == 0 else ctypes.addressof(geom))
    args = [buf] * 6
    assert lib.hdy_mask_measure(None, None, None, -1, *args, None) == -1
    assert b"negative K" in lib.hdy_last_error()
    assert lib.hdy_mask_measure(None, None, None, 0, *[None] * 6, None) == 0
    assert lib.hdy_mask_measure(None, None, None, 1, *args, None) == -1
    assert b"NULL" in lib.hdy_last_error()
    assert lib.hdy_mask_measure(geom, buf, buf, 1, buf, buf, buf, buf, None, buf, None) == -1
    assert b"NULL" in lib.hdy_last_error()
    assert lib.hdy_mask_measure(mis, buf, buf, 1, *args, None) == -1
    assert b"aligned" in lib.hdy_last_error()
    pm = PackedMasks(torch.zeros((1, 4), dtype=torch.int32), torch.zeros(2, dtype=torch.int64),
                     torch.zeros(1, dtype=torch.int32), 8, 8, torch.zeros(1, dtype=torch.int32))
    with pytest.raises(hdy.HdyError, match="CUDA"):
        pm.measure()
