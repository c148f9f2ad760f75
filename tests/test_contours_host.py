"""CPU tests of mask contours: the contract's identities on oracle/contours.py over random masks, save_geojson on
hand-built MaskContours, and the host-side argument checks of hdy_mask_contour_sizes / hdy_mask_contours."""
import ctypes
import json

import numpy as np
import pytest
import torch

import hd_yolo_b200 as hdy
from hd_yolo_b200 import _lib
from hd_yolo_b200.masks import MaskContours, PackedMasks
from oracle import contours as oc


def _random_masks(n, side, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        h, w = (int(v) for v in rng.integers(1, side + 1, 2))
        yield rng.random((h, w)) < rng.random()


def test_oracle_identities_on_random_masks():
    """Areas add up to the pixel count, even-odd filling gives the mask back, one exterior ring per 4-connected
    component, one hole ring per bounded 8-connected background component, the local vertex count, and the start
    order."""
    holes = 0
    for m in _random_masks(1500, 13, seed=0):
        rings, parent = oc.mask_rings(m)
        areas = [oc.signed_area(v) for v in rings]
        assert sum(areas) == m.sum()
        assert (oc.rasterize_even_odd(rings, *m.shape) == m).all()
        assert sum(a > 0 for a in areas) == oc.component_count(m)
        n_holes = sum(a < 0 for a in areas)
        assert n_holes == oc.hole_count(m)
        holes += n_holes
        assert sum(len(v) for v in rings) == oc.local_vertex_count(m)
        starts = [(int(v[0, 1]), int(v[0, 0])) for v in rings]
        assert starts == sorted(set(starts))
        for r, v in enumerate(rings):
            keys = [(int(y), int(x)) for x, y in v]
            assert keys[0] == min(keys) and keys.count(keys[0]) == 1
            turns = np.diff(np.concatenate([v, v[:1]]), axis=0)
            assert ((turns[:, 0] == 0) ^ (turns[:, 1] == 0)).all()            # unit-axis edges
            assert ((turns[:, 0] == 0) != np.roll(turns[:, 0] == 0, 1)).all()  # no collinear vertices
            assert (parent[r] < 0) == (areas[r] > 0)
            if parent[r] >= 0:
                x, y = v[0]
                assert m[y - 1, x] and parent[r] < r                         # the pixel above is its component's
    assert holes > 200


def test_oracle_hand_cases():
    px = np.ones((1, 1), bool)
    rings, parent = oc.mask_rings(px)
    assert [v.tolist() for v in rings] == [[[0, 0], [1, 0], [1, 1], [0, 1]]] and parent == [-1]
    # a saddle: two exterior rings touching at (1, 1), each turning right there
    rings, parent = oc.mask_rings(np.array([[1, 0], [0, 1]], bool))
    assert [v.tolist() for v in rings] == [[[0, 0], [1, 0], [1, 1], [0, 1]], [[1, 1], [2, 1], [2, 2], [1, 2]]]
    # a frame: exterior ring, then its hole (clockwise read with y up: negative area), parent = the exterior
    frame = np.ones((3, 3), bool)
    frame[1, 1] = False
    rings, parent = oc.mask_rings(frame)
    assert [v.tolist() for v in rings] == [[[0, 0], [3, 0], [3, 3], [0, 3]], [[1, 1], [1, 2], [2, 2], [2, 1]]]
    assert parent == [-1, 0] and oc.signed_area(rings[1]) == -1.0
    assert oc.mask_rings(np.zeros((3, 4), bool)) == ([], [])


def _contours(rings_per_row):
    """MaskContours from [[(ring [n, 2], parent_local)] per row]."""
    mr, rv, xy, par = [0], [0], [], []
    for rows in rings_per_row:
        base = mr[-1]
        for v, p in rows:
            xy += list(v)
            rv.append(rv[-1] + len(v))
            par.append(-1 if p < 0 else base + p)
        mr.append(base + len(rows))
    return MaskContours(torch.tensor(mr, dtype=torch.int64), torch.tensor(rv, dtype=torch.int64),
                        torch.tensor(xy, dtype=torch.int32).reshape(-1, 2), torch.tensor(par, dtype=torch.int32))


SQ = [[0, 0], [4, 0], [4, 4], [0, 4]]
HOLE = [[1, 1], [1, 2], [2, 2], [2, 1]]
SQ2 = [[10, 0], [12, 0], [12, 2], [10, 2]]


@pytest.mark.parametrize("chunk_rows", [1, 2, 3, 65536])
def test_save_geojson(tmp_path, chunk_rows):
    rows = [[(SQ, -1)], [], [(SQ, -1), (HOLE, 0), (SQ2, -1)], [(SQ, -1), (SQ2, -1), [[11, 1], [11, 2], [12, 2], [12, 1]]]]
    rows[3][2] = (rows[3][2], 1)                              # a hole of the second exterior
    c = _contours(rows)
    res = {'scores': torch.tensor([0.5, 0.25, 0.75, 1.0]), 'labels': torch.tensor([1, 2, 3, 4]),
           'index': torch.tensor([100, 101, 102, 103])}
    path = str(tmp_path / "out.geojson")
    assert hdy.save_geojson(path, res, c, chunk_rows=chunk_rows) == 3
    doc = json.load(open(path))
    assert doc["type"] == "FeatureCollection" and len(doc["features"]) == 3
    f0, f2, f3 = doc["features"]
    assert f0["properties"] == {"index": 100, "score": 0.5, "label": 1}
    assert f0["geometry"] == {"type": "Polygon", "coordinates": [SQ + [SQ[0]]]}
    assert f2["properties"]["index"] == 102                   # the empty row 1 is omitted
    assert f2["geometry"] == {"type": "MultiPolygon", "coordinates": [[SQ + [SQ[0]], HOLE + [HOLE[0]]],
                                                                      [SQ2 + [SQ2[0]]]]}
    h3 = [[11, 1], [11, 2], [12, 2], [12, 1], [11, 1]]
    assert f3["geometry"] == {"type": "MultiPolygon", "coordinates": [[SQ + [SQ[0]]], [SQ2 + [SQ2[0]], h3]]}
    assert not (tmp_path / "out.geojson.tmp").exists()
    # no 'index' entry: the row number; nothing to write: an empty collection
    assert hdy.save_geojson(path, {}, c, chunk_rows=chunk_rows) == 3
    assert [f["properties"] for f in json.load(open(path))["features"]] == [{"index": 0}, {"index": 2}, {"index": 3}]
    assert hdy.save_geojson(path, {}, _contours([[], []])) == 0
    assert json.load(open(path)) == {"type": "FeatureCollection", "features": []}
    with pytest.raises(hdy.HdyError):
        hdy.save_geojson(path, {'scores': torch.zeros(3)}, c)


def test_save_geojson_round_trips_oracle_rings(tmp_path):
    """Rings of random masks written and read back fill their masks again, each Feature on its own window."""
    masks = list(_random_masks(60, 12, seed=3))
    wins = [(5 * i, 7, m) for i, m in enumerate(masks)]
    ref = oc.contours(wins)
    c = MaskContours(ref['mask_rings'], ref['ring_verts'], ref['xy'], ref['parent'])
    path = str(tmp_path / "r.geojson")
    n = hdy.save_geojson(path, {}, c, chunk_rows=7)
    feats = json.load(open(path))["features"]
    assert n == len(feats) == sum(int(m.any()) for m in masks)
    for f in feats:
        x0, y0, m = wins[f["properties"]["index"]]
        polys = f["geometry"]["coordinates"]
        if f["geometry"]["type"] == "Polygon":
            polys = [polys]
        rings = [np.array(r[:-1]) - [x0, y0] for p in polys for r in p]
        assert all(r[0] == r[-1] for p in polys for r in p)
        assert (oc.rasterize_even_odd(rings, *m.shape) == m).all()


def test_contour_argument_checks():
    lib = _lib.load()
    buf = (ctypes.c_int64 * 4)()
    geom = (ctypes.c_int32 * 8)()
    mis = ctypes.c_void_p(ctypes.addressof(geom) + 4 if ctypes.addressof(geom) % 16 == 0 else ctypes.addressof(geom))
    assert lib.hdy_mask_contour_sizes(None, None, None, -1, buf, buf, None) == -1
    assert b"negative K" in lib.hdy_last_error()
    assert lib.hdy_mask_contour_sizes(None, None, None, 1, buf, buf, None) == -1
    assert b"NULL" in lib.hdy_last_error()
    assert lib.hdy_mask_contour_sizes(geom, buf, buf, 1, None, buf, None) == -1
    assert lib.hdy_mask_contour_sizes(mis, buf, buf, 1, buf, buf, None) == -1
    assert b"aligned" in lib.hdy_last_error()
    assert lib.hdy_mask_contours(None, None, None, -2, buf, buf, buf, buf, buf, None) == -1
    assert lib.hdy_mask_contours(None, None, None, 1, buf, buf, buf, buf, buf, None) == -1
    assert lib.hdy_mask_contours(mis, buf, buf, 1, buf, buf, buf, buf, buf, None) == -1
    assert lib.hdy_mask_contours(None, None, None, 0, buf, buf, None, None, None, None) == -1
    pm = PackedMasks(torch.zeros((1, 4), dtype=torch.int32), torch.zeros(2, dtype=torch.int64),
                     torch.zeros(1, dtype=torch.int32), 8, 8, torch.zeros(1, dtype=torch.int32))
    with pytest.raises(hdy.HdyError, match="CUDA"):
        pm.contours()
