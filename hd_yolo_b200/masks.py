"""Host-side mirror of the reference's mask post-processing over the C-ABI kernels (csrc/mask.cu).

Same names, argument meaning and return structures as the functions they replace:

* ``mask_select``            -- mask tail of Detect.compute_outputs (metayolo/models/yolo_head.py:332, 346-353)
* ``paste_masks_in_image``   -- torchvision.models.detection.roi_heads.paste_masks_in_image as the reference calls
                                it (metayolo/val_nuclei.py:169-176, metayolo/models/evaluation.py:122-123)
* ``process_mask``           -- ultralytics/yolov5 v7 utils/segment/general.py::process_mask (north-star extension;
                                the reference does not vendor it)

plus the bit-packed variants the throughput numbers use (``paste_masks_packed``, ``process_mask_packed``), which
fuse the ``> 0.5`` threshold (M3) and write box-cropped bit planes instead of [k,H,W] fp32 canvases.
No CPU fallback: CPU tensors raise HdyError.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import HdyError, ptr
from .ops import _Scratch, _aligned16, _call, _need_cuda, _need_head_tensor, _stream

_pm_scratch = _Scratch()

__all__ = ["MaskContours", "MaskMeasurements", "PackedMasks", "mask_select", "paste_masks_in_image", "paste_masks_packed", "process_mask",
           "process_mask_batch", "process_mask_packed", "SlideMaskBuilder"]


@dataclass
class MaskContours:
    """Boundary polygons of K masks (PackedMasks.contours(); contract in include/hd_yolo_b200.h and DESIGN §3.10).

    The rings of mask i are mask_rings[i] .. mask_rings[i+1]-1; ring r's vertices are xy[ring_verts[r]:ring_verts[r+1]]
    (x, y) pixel corners on the canvas, y down, starting at the least one in (y, x) order, not closed.  Exterior rings
    have positive shoelace area (counter-clockwise read with y up); parent[r] = -1 for them, else the index of the
    exterior ring of the hole's component."""

    mask_rings: torch.Tensor   # [K+1] int64
    ring_verts: torch.Tensor   # [R+1] int64
    xy: torch.Tensor           # [V, 2] int32
    parent: torch.Tensor       # [R] int32

    def __len__(self):
        return self.mask_rings.shape[0] - 1


@dataclass
class MaskMeasurements:
    """Morphometry of K masks (PackedMasks.measure(); contract in include/hd_yolo_b200.h and DESIGN §3.10b).

    Pixel (x, y) is the unit square [x, x+1] x [y, y+1] of the canvas, y down; dx = x - gx and dy = y - gy are pixel
    indices relative to the window (gx, gy, w, h) = geom[i].  The fields are exact, computed on the device:

    * area [K] i32; bbox [K, 4] i32 (x0, y0, x1, y1), the tight box of the set pixels, x1 / y1 exclusive;
    * moments [K, 5] i64: sum dx, sum dy, sum dx^2, sum dy^2, sum dx*dy over the set pixels;
    * quads [K, 4] i32: over the (w+1)(h+1) corners of the window, the 2 x 2 pixel patterns around each corner with n1
      (one set), n2 (two sharing an edge), n3 (three) and nD (two on a diagonal) set pixels;
    * convex_area2 [K] i64, hull_verts [K] i32, feret_max2 [K] i64: twice the area, the vertex count and the largest
      squared vertex distance of the convex hull of the set pixels' squares;
    * convex_perimeter, feret_min [K] f64: the hull's edge lengths summed in order from its least vertex in (y, x)
      order, and its least caliper width.

    The derived columns are fp64 expressions of those, computed with torch on access (A = area):

    * centroid = (gx + sum dx / A + 0.5, gy + sum dy / A + 0.5), the centroid of the pixel squares;
    * perimeter = n1 + n2 + n3 + 2 nD, the length of the contours() rings, holes included;
    * perimeter_smooth = n2 + (n1 + n3 + 2 nD) sqrt(1/2), the marching-squares contour through the pixel-edge midpoints;
    * euler = (n1 - n3 + 2 nD) / 4: 4-connected components minus holes;
    * convex_area = convex_area2 / 2; solidity = A / convex_area; extent = A / bbox area;
    * equivalent_diameter = sqrt(4 A / pi); circularity = 4 pi A / perimeter_smooth^2, not clamped: a digital disc
      gives 0.83 at radius 6 and 0.87 at radius 20, not 1;
    * mx = sum dx / A, c20 = sum dx^2 / A - mx^2, c02 likewise, c11 = sum dx dy / A - mx my: the central second moments
      of the pixel centres; l1, l2 = (c20 + c02) / 2 +- sqrt(((c20 - c02) / 2)^2 + c11^2), l2 clamped at 0;
      major_axis, minor_axis = 4 sqrt(l1), 4 sqrt(l2) (skimage's axis_major_length); eccentricity = sqrt(1 - l2 / l1),
      0 when l1 = 0; orientation = atan2(2 c11, c20 - c02) / 2, the major axis' angle from +x toward +y, in
      (-pi/2, pi/2];
    * feret_max = sqrt(feret_max2).

    Rows with area 0 give NaN for the centroid and every ratio."""

    geom: torch.Tensor              # [K, 4] int32: the windows the moments are relative to
    area: torch.Tensor              # [K] int32
    bbox: torch.Tensor              # [K, 4] int32
    moments: torch.Tensor           # [K, 5] int64
    quads: torch.Tensor             # [K, 4] int32
    convex_area2: torch.Tensor      # [K] int64
    hull_verts: torch.Tensor        # [K] int32
    feret_max2: torch.Tensor        # [K] int64
    convex_perimeter: torch.Tensor  # [K] float64
    feret_min: torch.Tensor         # [K] float64

    def __len__(self):
        return self.area.shape[0]

    def _q(self):
        q = self.quads.long()
        return q[:, 0], q[:, 1], q[:, 2], q[:, 3]

    @property
    def centroid(self) -> torch.Tensor:
        """[K, 2] float64 (x, y) in canvas pixels: the coordinates of the contours() polygons."""
        A, m, g = self.area.double(), self.moments.double(), self.geom.double()
        return torch.stack([g[:, 0] + m[:, 0] / A + 0.5, g[:, 1] + m[:, 1] / A + 0.5], 1)

    @property
    def perimeter(self) -> torch.Tensor:
        n1, n2, n3, nd = self._q()
        return (n1 + n2 + n3 + 2 * nd).double()

    @property
    def perimeter_smooth(self) -> torch.Tensor:
        n1, n2, n3, nd = self._q()
        return n2.double() + (n1 + n3 + 2 * nd).double() * math.sqrt(0.5)

    @property
    def euler(self) -> torch.Tensor:
        n1, _, n3, nd = self._q()
        return (n1 - n3 + 2 * nd) // 4

    @property
    def convex_area(self) -> torch.Tensor:
        return self.convex_area2.double() / 2

    @property
    def solidity(self) -> torch.Tensor:
        return self.area.double() / self.convex_area

    @property
    def extent(self) -> torch.Tensor:
        b = self.bbox.long()
        return self.area.double() / ((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])).double()

    @property
    def equivalent_diameter(self) -> torch.Tensor:
        return torch.sqrt(4 * self.area.double() / math.pi)

    @property
    def circularity(self) -> torch.Tensor:
        ps = self.perimeter_smooth
        return 4 * math.pi * self.area.double() / (ps * ps)

    def _central(self):
        A, m = self.area.double(), self.moments.double()
        mx, my = m[:, 0] / A, m[:, 1] / A
        return m[:, 2] / A - mx * mx, m[:, 3] / A - my * my, m[:, 4] / A - mx * my

    def _eigen(self):
        c20, c02, c11 = self._central()
        d = (c20 - c02) / 2
        half, root = (c20 + c02) / 2, torch.sqrt(d * d + c11 * c11)
        return half + root, torch.clamp(half - root, min=0.0)

    @property
    def major_axis(self) -> torch.Tensor:
        return 4 * torch.sqrt(self._eigen()[0])

    @property
    def minor_axis(self) -> torch.Tensor:
        return 4 * torch.sqrt(self._eigen()[1])

    @property
    def eccentricity(self) -> torch.Tensor:
        l1, l2 = self._eigen()
        return torch.where(l1 == 0, torch.zeros_like(l1), torch.sqrt(1 - l2 / l1))

    @property
    def orientation(self) -> torch.Tensor:
        c20, c02, c11 = self._central()
        return torch.atan2(2 * c11, c20 - c02) / 2

    @property
    def feret_max(self) -> torch.Tensor:
        return torch.sqrt(self.feret_max2.double())

    def columns(self) -> Dict[str, torch.Tensor]:
        """The user-facing columns, one [K] tensor each, in table order.  ``save_detections(path, {**result,
        **m.columns()}, masks)`` stores them beside the detections; ``save_geojson(..., measurements=m)`` writes them
        into each Feature's properties."""
        c = self.centroid
        return {"centroid_x": c[:, 0], "centroid_y": c[:, 1], "area": self.area, "perimeter": self.perimeter,
                "perimeter_smooth": self.perimeter_smooth, "euler": self.euler, "convex_area": self.convex_area,
                "convex_perimeter": self.convex_perimeter, "solidity": self.solidity, "extent": self.extent,
                "equivalent_diameter": self.equivalent_diameter, "circularity": self.circularity,
                "major_axis": self.major_axis, "minor_axis": self.minor_axis, "eccentricity": self.eccentricity,
                "orientation": self.orientation, "feret_max": self.feret_max, "feret_min": self.feret_min}


@dataclass
class PackedMasks:
    """Box-cropped bit planes (include/hd_yolo_b200.h, "Cropped bit-packed layout").

    geom[i] = (x0, y0, w, h): the window of mask i inside the (H, W) canvas; offsets[i] = first 32-bit word of
    mask i inside ``bits``; row r of mask i is ceil(w/32) words, pixel (x, y) is bit (x-x0)&31 of word
    offsets[i] + (y-y0)*ceil(w/32) + ((x-x0)>>5)."""

    geom: torch.Tensor      # [K, 4] int32
    offsets: torch.Tensor   # [K+1] int64
    bits: torch.Tensor      # [words] int32 (bit pattern of uint32)
    H: int
    W: int
    status: torch.Tensor    # [1] int32 device status word (HDY_STATUS_OVERFLOW)

    def __len__(self):
        return self.geom.shape[0]

    def check(self) -> None:
        if int(self.status.item()) & _lib.HDY_STATUS_OVERFLOW:
            raise HdyError("bit-plane capacity overflow: pass a larger capacity_words")

    def to_dense(self) -> torch.Tensor:
        """[K, H, W] uint8 canvas of 0/1 (what ``paste_masks_in_image(...) > 0.5`` holds)."""
        K = len(self)
        out = torch.empty((K, self.H, self.W), dtype=torch.uint8, device=self.geom.device)
        if K:
            _call("hdy_unpack_masks", ptr(self.geom), ptr(self.offsets), ptr(self.bits), K, self.H, self.W, ptr(out),
                  _stream(), launches=2)
        return out

    def nbytes(self) -> int:
        return self.bits.numel() * 4 + self.geom.numel() * 4 + self.offsets.numel() * 8

    @classmethod
    def from_dense(cls, masks: torch.Tensor) -> "PackedMasks":
        """The inverse of ``to_dense()``: [K, H, W] or [K, 1, H, W] CUDA masks -> PackedMasks with TIGHT windows (the
        bounding rectangle of the set pixels; an empty mask gets w = h = 0).  fp32 / fp16 pixels are set iff > 0.5
        (``paste_masks_in_image(...) > 0.5``), uint8 / bool pixels iff nonzero.  One 8-byte device->host read (the
        total word count)."""
        if not isinstance(masks, torch.Tensor) or not masks.is_cuda:
            raise HdyError("masks must be a CUDA tensor: hd_yolo_b200 has no CPU fallback")
        codes = {torch.float32: _lib.HDY_F32, torch.float16: _lib.HDY_F16, torch.uint8: _lib.HDY_U8,
                 torch.bool: _lib.HDY_U8}
        if masks.dtype not in codes:
            raise HdyError(f"masks must be float32, float16, uint8 or bool (got {masks.dtype})")
        if masks.dim() == 4 and masks.shape[1] == 1:
            masks = masks[:, 0]
        if masks.dim() != 3:
            raise HdyError(f"masks must be [K, H, W] or [K, 1, H, W], got {tuple(masks.shape)}")
        K, H, W = (int(s) for s in masks.shape)
        if H < 1 or W < 1:
            raise HdyError(f"empty canvas {H} x {W}")
        dev = masks.device
        src = masks.contiguous()
        if src.dtype == torch.bool:
            src = src.view(torch.uint8)
        geom = torch.empty((K, 4), dtype=torch.int32, device=dev)
        offsets = torch.empty((K + 1,), dtype=torch.int64, device=dev)
        status = torch.zeros((1,), dtype=torch.int32, device=dev)
        _call("hdy_pack_masks_geometry", ptr(src), codes[masks.dtype], K, H, W, ptr(geom), ptr(offsets), _stream(),
              launches=3)
        words = int(offsets[K].item())
        bits = torch.empty((max(words, 1),), dtype=torch.int32, device=dev)
        if K:
            _call("hdy_pack_masks", ptr(src), codes[masks.dtype], K, H, W, ptr(geom), ptr(offsets), ptr(bits), words,
                  ptr(status), _stream())
        return cls(geom, offsets, bits[:words], H, W, status)

    def areas(self) -> torch.Tensor:
        """[K] int32: set pixels per mask (bits beyond a row's width are ignored, whatever they hold)."""
        K = len(self)
        out = torch.empty((K,), dtype=torch.int32, device=self.geom.device)
        if K:
            _call("hdy_mask_areas", ptr(_aligned16(self.geom.contiguous())), ptr(self.offsets),
                  ptr(self._bits_nonempty()), K, ptr(out), _stream())
        return out

    def contours(self) -> MaskContours:
        """The boundary polygons of every mask, traced on the device (csrc/contours.cu).  One 16-byte device->host read
        (the ring and vertex totals).  Rows: ``masks.select(rows).contours()``."""
        if not self.geom.is_cuda:
            raise HdyError("contours() needs the planes on a CUDA device: hd_yolo_b200 has no CPU fallback")
        self.check()
        K, dev = len(self), self.geom.device
        geom, bits = _aligned16(self.geom.contiguous()), self._bits_nonempty()
        mask_rings = torch.empty((K + 1,), dtype=torch.int64, device=dev)
        vert_off = torch.empty((K + 1,), dtype=torch.int64, device=dev)
        _call("hdy_mask_contour_sizes", ptr(geom), ptr(self.offsets), ptr(bits), K, ptr(mask_rings), ptr(vert_off),
              _stream(), launches=4)
        R, V = torch.stack([mask_rings[K], vert_off[K]]).tolist()
        if R >= 2 ** 31:
            raise HdyError(f"{R} rings: parent indices are int32, trace fewer rows at a time")
        ring_verts = torch.empty((R + 1,), dtype=torch.int64, device=dev)
        parent = torch.empty((max(R, 1),), dtype=torch.int32, device=dev)
        xy = torch.empty((max(V, 1), 2), dtype=torch.int32, device=dev)
        _call("hdy_mask_contours", ptr(geom), ptr(self.offsets), ptr(bits), K, ptr(mask_rings), ptr(vert_off),
              ptr(ring_verts), ptr(parent), ptr(xy), _stream(), launches=2)
        return MaskContours(mask_rings, ring_verts, xy[:V], parent[:R])

    def measure(self) -> MaskMeasurements:
        """Area, box, moments, corner patterns, convex hull and calipers of every mask, on the device
        (csrc/measure.cu), with the derived columns as properties of the result.  Window sides up to 32 768; a larger
        window raises.  One 4-byte device->host read (the least area, and the overflow flag of the planes).  Rows:
        ``masks.select(rows).measure()``."""
        if not self.geom.is_cuda:
            raise HdyError("measure() needs the planes on a CUDA device: hd_yolo_b200 has no CPU fallback")
        K, dev = len(self), self.geom.device
        geom, bits = _aligned16(self.geom.contiguous()), self._bits_nonempty()
        area = torch.empty((K,), dtype=torch.int32, device=dev)
        bbox = torch.empty((K, 4), dtype=torch.int32, device=dev)
        moments = torch.empty((K, 5), dtype=torch.int64, device=dev)
        quads = torch.empty((K, 4), dtype=torch.int32, device=dev)
        hull = torch.empty((K, 3), dtype=torch.int64, device=dev)
        hull_len = torch.empty((K, 2), dtype=torch.float64, device=dev)
        flag = (self.status[:1] & _lib.HDY_STATUS_OVERFLOW) * -2
        if K:
            _call("hdy_mask_measure", ptr(geom), ptr(self.offsets), ptr(bits), K, ptr(area), ptr(bbox), ptr(moments),
                  ptr(quads), ptr(hull), ptr(hull_len), _stream(), launches=2)
            flag = torch.minimum(flag, area.amin().view(1))
        low = int(flag.item())
        if low == -2:
            raise HdyError("bit-plane capacity overflow: pass a larger capacity_words")
        if low < 0:
            row = int(torch.nonzero(area < 0)[0, 0])
            w, h = self.geom[row, 2:].tolist()
            raise HdyError(f"mask {row} has a {w} x {h} window: measure() takes window sides up to 32768")
        return MaskMeasurements(self.geom, area, bbox, moments, quads, hull[:, 0], hull[:, 2].to(torch.int32),
                                hull[:, 1], hull_len[:, 0], hull_len[:, 1])

    def select(self, rows) -> "PackedMasks":
        """The masks of `rows` (index tensor or sequence), in that order, sharing `bits`: geom[rows] and offsets[rows]
        address them, offsets[-1] stays the total word count.  Turns a slide result into matcher input:
        ``res['masks'].select(res['index'] - res['base'])``."""
        rows = torch.as_tensor(rows, dtype=torch.int64, device=self.geom.device)
        if rows.dim() != 1:
            raise HdyError(f"rows must be one-dimensional, got {tuple(rows.shape)}")
        return PackedMasks(self.geom[rows].contiguous(), torch.cat([self.offsets[rows], self.offsets[-1:]]), self.bits,
                           self.H, self.W, self.status)

    @classmethod
    def cat(cls, parts, origins, canvas) -> "PackedMasks":
        """Masks of several canvases placed on one: part i's canvas (its H x W) goes to (x, y) = origins[i] of the
        (H, W) `canvas` and must lie inside it -- e.g. the ground truth of several annotated regions of a slide on the
        slide canvas.  Rows in part order; windows move by the origin (empty windows stay empty), offsets by the words
        of the parts before; `bits` is the parts' planes one after another.  The status word is the OR of the parts'."""
        parts, origins = list(parts), [tuple(int(v) for v in o) for o in origins]
        if not parts or len(parts) != len(origins):
            raise HdyError(f"cat takes one origin per part ({len(parts)} parts, {len(origins)} origins)")
        H, W = _hw(canvas)
        for p, (x, y) in zip(parts, origins):
            if x < 0 or y < 0 or x + p.W > W or y + p.H > H:
                raise HdyError(f"a {p.H} x {p.W} canvas at (x, y) = ({x}, {y}) does not fit the {H} x {W} canvas")
        geoms, offs, bits, base = [], [], [], 0
        for p, (x, y) in zip(parts, origins):
            g = p.geom.clone()
            live = (g[:, 2] > 0) & (g[:, 3] > 0)
            g[:, 0] += torch.where(live, x, 0).to(g.dtype)
            g[:, 1] += torch.where(live, y, 0).to(g.dtype)
            geoms.append(g)
            offs.append(p.offsets[:-1] + base)
            bits.append(p.bits)
            base += int(p.bits.numel())
        dev = parts[0].geom.device
        status = parts[0].status.clone()
        for p in parts[1:]:
            status |= p.status
        offsets = torch.cat(offs + [torch.tensor([base], dtype=torch.int64, device=dev)])
        return cls(torch.cat(geoms).contiguous(), offsets, torch.cat(bits), H, W, status)

    def _bits_nonempty(self) -> torch.Tensor:
        """`bits`, or one zero word when no mask has any (an empty tensor has no device address)."""
        return self.bits if self.bits.numel() else torch.zeros((1,), dtype=torch.int32, device=self.bits.device)


def _hw(shape) -> Tuple[int, int]:
    if isinstance(shape, int):
        return int(shape), int(shape)
    return int(shape[0]), int(shape[1])


def _boxes4(boxes: torch.Tensor, k: int, name="boxes") -> torch.Tensor:
    _need_cuda(boxes, name)
    if boxes.dim() != 2 or boxes.shape[1] < 4 or boxes.shape[0] != k:
        raise HdyError(f"{name} must be [{k}, 4], got {tuple(boxes.shape)}")
    b = boxes[:, :4]
    return _aligned16(b.contiguous())


# ------------------------------------------------------------------------------------------------ M1
def mask_select(mask_logits: torch.Tensor, labels: torch.Tensor, mask_indices: torch.Tensor) -> torch.Tensor:
    """yolo_head.py:332, 346-353 for the K detections of one batch: sigmoid, pick the channel
    ``mask_indices[labels.clamp(min=0)]`` of every detection, zero masks whose channel index is < 0.
    mask_logits [K, C, M, M] fp32, labels [K] int64, mask_indices [1+nc] int64 -> [K, 1, M, M]."""
    _need_cuda(mask_logits, "mask_logits")
    if mask_logits.dim() != 4 or mask_logits.shape[2] != mask_logits.shape[3]:
        raise HdyError(f"mask_logits must be [K, C, M, M], got {tuple(mask_logits.shape)}")
    K, Cn, M, _ = mask_logits.shape
    dev = mask_logits.device
    labels = labels.to(dev, torch.int64).contiguous()
    mask_indices = mask_indices.to(dev, torch.int64).contiguous()
    if labels.shape != (K,):
        raise HdyError("labels must be [K]")
    out = torch.empty((K, 1, M, M), dtype=torch.float32, device=dev)
    if K:
        _call("hdy_mask_select", ptr(mask_logits.contiguous()), ptr(labels), ptr(mask_indices), K, Cn, M, ptr(out),
              _stream())
    return out


# ------------------------------------------------------------------------------------------------ M2
def _paste_src(masks: torch.Tensor):
    _need_cuda(masks, "masks")
    if masks.dim() == 3:
        masks = masks[:, None]
    if masks.dim() != 4 or masks.shape[2] != masks.shape[3]:
        raise HdyError(f"masks must be [k, C, M, M], got {tuple(masks.shape)}")
    return masks.contiguous()


def paste_masks_in_image(masks: torch.Tensor, boxes: torch.Tensor, img_shape, padding: int = 1) -> torch.Tensor:
    """torchvision paste_masks_in_image(masks [k,1,M,M], boxes [k,4], (H,W), padding=1) -> [k,1,H,W] fp32
    (val_nuclei.py:169-176, evaluation.py:122-123): zero-pad the mask, grow the box by (M+2p)/M about its
    centre, truncate to integers, bilinear-resize to the box, paste into a zero canvas."""
    masks = _paste_src(masks)
    k, Cn, M, _ = masks.shape
    if Cn != 1:
        raise HdyError("paste_masks_in_image takes [k,1,M,M] masks (use paste_masks_packed(channel=...) to fuse M1)")
    H, W = _hw(img_shape)
    out = torch.empty((k, 1, H, W), dtype=torch.float32, device=masks.device)
    if k:
        b = _boxes4(boxes, k)
        _call("hdy_paste_masks", ptr(masks), None, ptr(b), k, 1, M, int(padding), 0, H, W, ptr(out), _stream(),
              launches=2)
    return out


def paste_masks_packed(masks: torch.Tensor, boxes: torch.Tensor, img_shape, padding: int = 1,
                       channel: Optional[torch.Tensor] = None, apply_sigmoid: bool = False,
                       capacity_words: Optional[int] = None) -> PackedMasks:
    """M1 + M2 + M3 fused: ``paste_masks_in_image(...) > 0.5`` as box-cropped bit planes.

    masks [k, C, M, M]: probabilities, or raw logits with apply_sigmoid=True; channel [k] int32 selects the
    channel per detection (None: 0; < 0: empty mask) -- i.e. ``mask_indices[labels.clamp(min=0)]``.
    capacity_words=None sizes ``bits`` exactly (one 8-byte device->host read); pass an upper bound to stay
    asynchronous (overflow is then reported by PackedMasks.check())."""
    masks = _paste_src(masks)
    k, Cn, M, _ = masks.shape
    H, W = _hw(img_shape)
    dev = masks.device
    geom = torch.empty((k, 4), dtype=torch.int32, device=dev)
    offsets = torch.empty((k + 1,), dtype=torch.int64, device=dev)
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    b = _boxes4(boxes, k) if k else None
    if channel is not None:
        channel = channel.to(dev, torch.int32).contiguous()
    _call("hdy_paste_geometry", ptr(b), ptr(channel), k, M, int(padding), H, W, ptr(geom), ptr(offsets), _stream(),
          launches=4)
    words = int(offsets[k].item()) if capacity_words is None else int(capacity_words)
    bits = torch.empty((max(words, 1),), dtype=torch.int32, device=dev)
    if k:
        _call("hdy_paste_masks_packed", ptr(masks), ptr(channel), ptr(b), ptr(offsets), k, Cn, M, int(padding),
              int(bool(apply_sigmoid)), H, W, ptr(bits), words, ptr(status), _stream())
    return PackedMasks(geom, offsets, bits[:words], H, W, status)


# ---------------------------------------------------------------------------------- process_mask (B)
def _pm_args(protos, coef, boxes, counts):
    _need_head_tensor(protos, "protos")
    _need_cuda(coef, "masks_in")
    _need_cuda(boxes, "bboxes")
    if protos.dim() != 4 or coef.dim() != 3 or boxes.dim() != 3:
        raise HdyError("expected protos [bs,nm,mh,mw], coef [bs,max_det,nm], boxes [bs,max_det,4]")
    bs, nm, mh, mw = protos.shape
    if coef.shape[0] != bs or coef.shape[2] != nm or boxes.shape[:2] != coef.shape[:2] or boxes.shape[2] != 4:
        raise HdyError("protos / coef / boxes shapes disagree")
    if counts.shape != (bs,) or counts.dtype != torch.int32 or not counts.is_cuda:
        raise HdyError("counts must be a CUDA int32 tensor [bs]")
    return bs, nm, mh, mw, coef.shape[1]


def _pm_workspace(dev, bs: int, md: int):
    """Grow-only scratch for the two-phase path (sigmoid patches + the list of over-sized detections)."""
    nbytes = _lib.load().hdy_process_mask_workspace_bytes(bs, md)
    return _pm_scratch.get(dev, "process_mask", nbytes), nbytes


def process_mask_batch(protos: torch.Tensor, coef: torch.Tensor, boxes: torch.Tensor, counts: torch.Tensor, shape,
                       upsample: bool = False) -> torch.Tensor:
    """process_mask for a batch of tiles (struct-of-arrays, as DetectBatch holds them): protos [bs,nm,mh,mw],
    coef [bs,max_det,nm], boxes [bs,max_det,4] in image pixels, counts [bs] int32.
    Returns [bs, max_det, oh, ow] fp32 in {0,1}; slots >= counts[i] are zero."""
    bs, nm, mh, mw, md = _pm_args(protos, coef, boxes, counts)
    ih, iw = _hw(shape)
    oh, ow = (ih, iw) if upsample else (mh, mw)
    out = torch.empty((bs, md, oh, ow), dtype=torch.float32, device=protos.device)
    coef = coef.float()
    if bs and md:
        ws, wbytes = _pm_workspace(protos.device, bs, md)
        _call("hdy_process_mask", ptr(_aligned16(protos.contiguous())), _need_head_tensor(protos, "protos"),
              ptr(coef.contiguous()),
              ptr(_aligned16(boxes.contiguous())), ptr(counts), bs, md, nm, mh, mw, ih, iw, int(bool(upsample)),
              ptr(out), ptr(ws), wbytes, _stream(), launches=4)
    return out


def process_mask(protos: torch.Tensor, masks_in: torch.Tensor, bboxes: torch.Tensor, shape,
                 upsample: bool = False) -> torch.Tensor:
    """ultralytics/yolov5 v7 ``process_mask(protos [c,mh,mw], masks_in [n,c], bboxes [n,4], shape (ih,iw),
    upsample=False)`` -> [n, mh, mw] (or [n, ih, iw] with upsample) of 0/1 floats:
    sigmoid(masks_in @ protos), crop to the box scaled into proto space, optional bilinear upsample, > 0.5."""
    _need_head_tensor(protos, "protos")
    if protos.dim() != 3:
        raise HdyError("protos must be [c, mh, mw]")
    n = masks_in.shape[0]
    ih, iw = _hw(shape)
    if n == 0:
        oh, ow = (ih, iw) if upsample else tuple(protos.shape[1:])
        return protos.new_zeros((0, oh, ow), dtype=torch.float32)
    counts = torch.full((1,), n, dtype=torch.int32, device=protos.device)
    return process_mask_batch(protos[None], masks_in.float()[None], bboxes.float()[None, :, :4], counts, shape,
                              upsample)[0]


def process_mask_packed(protos: torch.Tensor, coef: torch.Tensor, boxes: torch.Tensor, counts: torch.Tensor, shape,
                        upsample: bool = False, capacity_words: Optional[int] = None,
                        row_state: Optional[torch.Tensor] = None,
                        tile_offsets: Optional[torch.Tensor] = None) -> PackedMasks:
    """Bit-packed process_mask over a batch of tiles; mask index = tile * max_det + slot (empty for slots
    >= counts[tile]).  Window coordinates are in output pixels ((ih,iw) with upsample, else (mh,mw)).
    row_state [n] uint8 + tile_offsets [bs+1] int64 (slide form): only slots whose slide row was KEPT get a mask."""
    bs, nm, mh, mw, md = _pm_args(protos, coef, boxes, counts)
    ih, iw = _hw(shape)
    dev = protos.device
    K = bs * md
    boxes = _aligned16(boxes.contiguous())
    geom = torch.empty((K, 4), dtype=torch.int32, device=dev)
    offsets = torch.empty((K + 1,), dtype=torch.int64, device=dev)
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    _call("hdy_process_mask_geometry", ptr(boxes), ptr(counts), bs, md, mh, mw, ih, iw, int(bool(upsample)),
          ptr(row_state), ptr(tile_offsets), ptr(geom), ptr(offsets), _stream(), launches=2)
    words = int(offsets[K].item()) if capacity_words is None else int(capacity_words)
    bits = torch.empty((max(words, 1),), dtype=torch.int32, device=dev)
    if K:
        ws, wbytes = _pm_workspace(dev, bs, md)
        _call("hdy_process_mask_packed", ptr(_aligned16(protos.contiguous())), _need_head_tensor(protos, "protos"),
              ptr(coef.contiguous()), ptr(boxes),
              ptr(counts), ptr(geom), ptr(offsets), bs, md, nm, mh, mw, ih, iw, int(bool(upsample)), ptr(bits), words,
              ptr(status),
              ptr(ws), wbytes, _stream(), launches=3)
    oh, ow = (ih, iw) if upsample else (mh, mw)
    return PackedMasks(geom, offsets, bits[:words], oh, ow, status)


class SlideMaskBuilder:
    """Masks of a whole slide, computed AFTER the slide-level verdicts and only for the rows Ensemble.merge keeps
    (yolo.py:197-202 gathers masks[keep]; the masks of suppressed duplicates are never materialised).  One
    PackedMasks over the slide's rows: geom[r] is the window of row r in SLIDE pixels, offsets[r] its first word in the
    slide-wide `bits`; rows that were not kept have empty windows.  Everything stays on the device; `check()` reads
    the overflow flag."""

    def __init__(self, n_rows: int, capacity_words: int, image_size, device):
        d = torch.device(device)
        self.n = int(n_rows)
        self.capacity_words = int(capacity_words)
        self.geom = torch.zeros((max(self.n, 1), 4), dtype=torch.int32, device=d)
        self.offsets = torch.zeros((self.n + 1,), dtype=torch.int64, device=d)
        self.bits = torch.empty((max(self.capacity_words, 1),), dtype=torch.int32, device=d)
        self.cursor2 = torch.zeros((2,), dtype=torch.int64, device=d)
        self.status = torch.zeros((1,), dtype=torch.int32, device=d)
        self.batches = 0
        self.H, self.W = _hw(image_size)

    def prepare(self, boxes: torch.Tensor, counts: torch.Tensor, tile_offsets: torch.Tensor, rois: torch.Tensor,
                row_state: torch.Tensor, proto_hw, shape, upsample: bool = True, lane: int = 0):
        """Windows and word offsets of the next batch (in batch order: the slide-wide word cursor advances), scattered
        to the slide rows.  Returns (geom, offsets) for ``run``; `lane` picks the scratch pair, so that the kernels of
        batch i can still read theirs while batch i + 1 is prepared (mask kernels on alternating streams)."""
        bs, md = int(boxes.shape[0]), int(boxes.shape[1])
        mh, mw = proto_hw
        ih, iw = _hw(shape)
        dev = boxes.device
        K = bs * md
        if K == 0:
            return None
        boxes = _aligned16(boxes.contiguous())
        geom = _pm_scratch.get(dev, f"slide_geom{lane}", K * 16).view(torch.int32)[:K * 4]
        offsets = _pm_scratch.get(dev, f"slide_offsets{lane}", (K + 1) * 8).view(torch.int64)[:K + 1]
        _call("hdy_process_mask_geometry", ptr(boxes), ptr(counts), bs, md, mh, mw, ih, iw, int(bool(upsample)),
              ptr(row_state), ptr(tile_offsets), ptr(geom), ptr(offsets), _stream(), launches=2)
        _call("hdy_process_mask_rows", ptr(geom), ptr(offsets), ptr(counts), ptr(tile_offsets),
              ptr(_aligned16(rois.contiguous())), bs, md, ptr(self.cursor2), self.batches & 1, ptr(self.geom),
              ptr(self.offsets), _stream())
        self.batches += 1
        return geom, offsets

    def run(self, prepared, protos: torch.Tensor, coef: torch.Tensor, boxes: torch.Tensor, counts: torch.Tensor,
            shape, upsample: bool = True) -> None:
        """The mask kernels of a prepared batch (any stream ordered after its ``prepare``)."""
        if prepared is None:
            return
        geom, offsets = prepared
        bs, nm, mh, mw, md = _pm_args(protos, coef, boxes, counts)
        ih, iw = _hw(shape)
        dev = protos.device
        boxes = _aligned16(boxes.contiguous())
        ws, wbytes = _pm_workspace(dev, bs, md)
        _call("hdy_process_mask_packed", ptr(_aligned16(protos.contiguous())), _need_head_tensor(protos, "protos"),
              ptr(coef.contiguous()), ptr(boxes),
              ptr(counts), ptr(geom), ptr(offsets), bs, md, nm, mh, mw, ih, iw, int(bool(upsample)), ptr(self.bits),
              self.capacity_words, ptr(self.status), ptr(ws), wbytes, _stream(), launches=3)

    def add_batch(self, protos: torch.Tensor, coef: torch.Tensor, boxes: torch.Tensor, counts: torch.Tensor,
                  tile_offsets: torch.Tensor, rois: torch.Tensor, row_state: torch.Tensor, shape,
                  upsample: bool = True) -> None:
        """protos [bs,nm,mh,mw] of the batch's tiles; coef / boxes / counts as DetectBatch holds them (tile
        coordinates); tile_offsets [bs+1] from the append; rois [bs,4]; row_state: verdict per slide row."""
        prep = self.prepare(boxes, counts, tile_offsets, rois, row_state, tuple(protos.shape[2:]), shape, upsample)
        self.run(prep, protos, coef, boxes, counts, shape, upsample)

    def finish(self) -> PackedMasks:
        """offsets[n] = total words.  Rows that were never live keep offset 0 / an empty window: consumers address a
        mask through geom[r] and offsets[r] only."""
        self.offsets[self.n:self.n + 1].copy_(self.cursor2[self.batches & 1:(self.batches & 1) + 1])
        return PackedMasks(self.geom[:self.n], self.offsets, self.bits, self.H, self.W, self.status)
