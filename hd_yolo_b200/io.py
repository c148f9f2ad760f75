"""Compact on-disk format for post-processing results (SURVEY 8f rank 3: the reference pickles Python dicts of CPU
tensors with ``torch.save``, evaluation.py:225 -- 4 MB of dense fp32 mask per nucleus at 1024 px if masks are kept).

One little-endian file: a JSON header line (magic, version, array table with dtype / shape / byte offset, free-form
``meta``) padded to 64 bytes, then the raw arrays, each 64-byte aligned.  Detections are the struct-of-arrays the
package works in (``boxes`` fp32 [k,4], ``scores`` fp32 [k], ``labels`` int64 stored as int16, optional ``index``);
masks are the cropped bit planes of ``PackedMasks`` (geom / offsets / bits), ~100-300 bytes per nucleus.  Host-side
only (CUDA tensors are read back once); loading memory-maps the file and returns CPU tensors.

``save_geojson`` writes the boundary polygons of PackedMasks.contours() as one RFC 7946 FeatureCollection, the format
slide viewers, annotation tools and morphometry code read; with ``measurements`` (PackedMasks.measure()) each Feature
also carries its row of the morphometry table.
"""
from __future__ import annotations

import json
import math
import os
from typing import Dict, Optional, Tuple, Union

import numpy as np
import torch

from ._lib import HdyError
from .masks import MaskContours, MaskMeasurements, PackedMasks

__all__ = ["save_detections", "load_detections", "save_geojson"]

MAGIC = "hd_yolo_b200.detections"
VERSION = 1
_ALIGN = 64
# label -100 ("unclassified", yolo_head.py:345) and class ids up to 32767 fit int16
_STORE_AS = {"labels": np.int16}


def _np(t: torch.Tensor) -> np.ndarray:
    return t.detach().cpu().contiguous().numpy()


def save_detections(path: str, result: Dict[str, torch.Tensor], masks: Optional[PackedMasks] = None,
                    meta: Optional[dict] = None) -> int:
    """Writes `result` ('boxes' [k,4], 'scores' [k], optional 'labels' [k], 'index' [k], any other tensor entry) and
    optionally the bit-packed masks of the same k detections.  Returns the file size in bytes."""
    arrays = {}
    for name, t in result.items():
        if not isinstance(t, torch.Tensor):
            continue
        a = _np(t)
        if name in _STORE_AS:
            if a.size and (a.min() < np.iinfo(_STORE_AS[name]).min or a.max() > np.iinfo(_STORE_AS[name]).max):
                raise HdyError(f"'{name}' does not fit {_STORE_AS[name].__name__}")
            a = a.astype(_STORE_AS[name])
        arrays[name] = (a, str(t.dtype).replace("torch.", ""))
    k = int(result["boxes"].shape[0])
    if masks is not None:
        if len(masks) != k:
            raise HdyError(f"{len(masks)} masks for {k} detections")
        masks.check()
        words = int(masks.offsets[-1].item())
        arrays["mask_geom"] = (_np(masks.geom), "int32")
        arrays["mask_offsets"] = (_np(masks.offsets), "int64")
        arrays["mask_bits"] = (_np(masks.bits[:words]), "int32")
    table, off = [], 0
    for name, (a, orig) in arrays.items():
        off = (off + _ALIGN - 1) // _ALIGN * _ALIGN
        table.append({"name": name, "dtype": a.dtype.str, "shape": list(a.shape), "offset": off, "restore": orig})
        off += a.nbytes
    header = {"magic": MAGIC, "version": VERSION, "count": k, "arrays": table, "meta": meta or {},
              "mask_canvas": [masks.H, masks.W] if masks is not None else None}
    head = (json.dumps(header) + "\n").encode()
    head += b" " * ((-len(head)) % _ALIGN)
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(head)
        for entry, (a, _) in zip(table, arrays.values()):
            f.seek(len(head) + entry["offset"])
            f.write(a.tobytes())
    os.replace(tmp, path)          # a reader never sees a half-written file
    return os.path.getsize(path)


def load_detections(path: str, mmap: bool = True) -> Tuple[Dict[str, torch.Tensor], Optional[PackedMasks], dict]:
    """-> (result dict of CPU tensors, PackedMasks on the CPU or None, meta).  `PackedMasks.to_dense()` needs the
    tensors on a CUDA device (`.geom.cuda()` ...): the file itself never holds dense masks."""
    with open(path, "rb") as f:
        line = f.readline()
    try:
        header = json.loads(line)
    except Exception as e:
        raise HdyError(f"{path}: not a detections file") from e
    if header.get("magic") != MAGIC or header.get("version") != VERSION:
        raise HdyError(f"{path}: magic/version mismatch ({header.get('magic')}, {header.get('version')})")
    base = (len(line) + _ALIGN - 1) // _ALIGN * _ALIGN
    out: Dict[str, torch.Tensor] = {}
    for e in header["arrays"]:
        n = int(np.prod(e["shape"])) if e["shape"] else 1
        if mmap and n:
            a = np.memmap(path, dtype=np.dtype(e["dtype"]), mode="r", offset=base + e["offset"], shape=tuple(e["shape"]))
            a = np.array(a)        # one sequential read; the tensors own their memory
        else:
            a = np.fromfile(path, dtype=np.dtype(e["dtype"]), count=n, offset=base + e["offset"]).reshape(e["shape"])
        out[e["name"]] = torch.from_numpy(np.ascontiguousarray(a)).to(getattr(torch, e["restore"]))
    masks = None
    if header.get("mask_canvas"):
        H, W = header["mask_canvas"]
        masks = PackedMasks(out.pop("mask_geom"), out.pop("mask_offsets"), out.pop("mask_bits"), int(H), int(W),
                            torch.zeros((1,), dtype=torch.int32))
    return out, masks, header.get("meta", {})


def _json_number(v):
    """JSON has no NaN or infinity: such a value is written as null."""
    return v if not isinstance(v, float) or math.isfinite(v) else None


def save_geojson(path: str, result: Dict[str, torch.Tensor], contours: MaskContours, chunk_rows: int = 65536,
                 measurements: Union[MaskMeasurements, Dict[str, torch.Tensor], None] = None) -> int:
    """Writes one RFC 7946 FeatureCollection with a Feature per row of `contours` that has a ring: a Polygon for one
    exterior ring, a MultiPolygon for several, each exterior followed by its holes, every ring closed by repeating its
    first vertex.  Coordinates are canvas pixel corners (x, y).  Properties: 'index' (``result['index']`` if present,
    else the row), 'score' and 'label' (``result['scores']`` / ``result['labels']`` if present).  `contours` may be on
    the CPU or a CUDA device; it is read back `chunk_rows` rows at a time and the text is streamed to `path` + '.tmp',
    then renamed.  `measurements` (a MaskMeasurements, whose ``columns()`` are written, or a dict of [K] tensors) adds
    ``properties.measurements = {name: value}`` to each Feature, the key QuPath reads; non-finite values are written as
    null.  Returns the number of Features written."""
    K = len(contours)
    cols = {}
    for key, name in (("index", "index"), ("scores", "score"), ("labels", "label")):
        t = result.get(key)
        if isinstance(t, torch.Tensor):
            if t.shape[0] != K:
                raise HdyError(f"result['{key}'] has {t.shape[0]} rows, contours {K}")
            cols[name] = t
    if isinstance(measurements, MaskMeasurements):
        measurements = measurements.columns()
    for key, t in (measurements or {}).items():
        if not isinstance(t, torch.Tensor) or t.dim() != 1 or t.shape[0] != K:
            raise HdyError(f"measurements['{key}'] must be a [{K}] tensor")
    if chunk_rows < 1:
        raise HdyError("chunk_rows must be >= 1")
    n = 0
    tmp = path + ".tmp"
    with open(tmp, "w") as f:
        f.write('{"type": "FeatureCollection", "features": [')
        for a in range(0, K, chunk_rows):
            b = min(a + chunk_rows, K)
            mr = contours.mask_rings[a:b + 1].cpu().tolist()
            r0, r1 = mr[0], mr[-1]
            rv = contours.ring_verts[r0:r1 + 1].cpu().numpy()
            xy = contours.xy[int(rv[0]):int(rv[-1])].cpu().numpy().tolist()
            parent = contours.parent[r0:r1].cpu().numpy().tolist()
            props = {name: t[a:b].cpu().tolist() for name, t in cols.items()}
            meas = {name: t[a:b].cpu().tolist() for name, t in measurements.items()} if measurements else None
            v0 = int(rv[0])
            for i in range(a, b):
                lo, hi = mr[i - a], mr[i - a + 1]
                if lo == hi:
                    continue
                polys, at = [], {}
                for r in range(lo, hi):
                    ring = xy[int(rv[r - r0]) - v0:int(rv[r - r0 + 1]) - v0]
                    ring.append(ring[0])
                    p = parent[r - r0]
                    if p < 0:
                        at[r] = len(polys)
                        polys.append([ring])
                    else:
                        polys[at[p]].append(ring)
                geometry = ({"type": "Polygon", "coordinates": polys[0]} if len(polys) == 1 else
                            {"type": "MultiPolygon", "coordinates": polys})
                pr = {"index": props["index"][i - a] if "index" in props else i}
                for name in ("score", "label"):
                    if name in props:
                        pr[name] = props[name][i - a]
                if meas is not None:
                    pr["measurements"] = {name: _json_number(v[i - a]) for name, v in meas.items()}
                f.write((",\n" if n else "\n") +
                        json.dumps({"type": "Feature", "geometry": geometry, "properties": pr}, separators=(",", ":")))
                n += 1
        f.write("\n]}\n")
    os.replace(tmp, path)
    return n
