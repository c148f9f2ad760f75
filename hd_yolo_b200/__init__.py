"""hd_yolo_b200 -- B200-native (sm_100a) post-processing hot path of impromptuRong/hd_yolo.

Only the path from Detect/Segment head outputs to final nuclei instances lives here
(decode, filter/compact, NMS, score select, masks, tile merge).  Host code is thin Python over
the C-ABI in ``include/hd_yolo_b200.h``; there is no CPU fallback.
"""
from ._lib import HdyError, LIB_PATH, load  # noqa: F401
from .ops import (  # noqa: F401
    CapturedStep,
    DetectBatch,
    HeadSpec,
    batched_nms,
    compute_proposals,
    decode_concat,
    detect_postprocess,
    flatten_onehot_objects,
    nms,
    nms_per_image,
    non_max_suppression,
    scratch_slot,
    set_iou_compare,
)

from . import masks  # noqa: F401,E402
from .masks import (  # noqa: F401,E402
    MaskContours,
    MaskMeasurements,
    PackedMasks,
    mask_select,
    paste_masks_in_image,
    paste_masks_packed,
    process_mask,
    process_mask_batch,
    process_mask_packed,
    SlideMaskBuilder,
)

from . import slide  # noqa: F401,E402
from .slide import (  # noqa: F401,E402
    Ensemble,
    SlideAccumulator,
    clip_coords,
    ensemble_merge,
    merge_nms,
    merge_outputs,
    rescale_outputs,
    scale_coords,
    sliding_window_scanner,
    sort_keys,
    tile_cores,
)

from . import dist, hnet, io, metrics, pipeline, roi  # noqa: F401,E402
from .io import load_detections, save_detections, save_geojson  # noqa: F401,E402
from .metrics import APMeter, box_iou, match_predictions  # noqa: F401,E402
from .roi import batch_rois, compute_outputs, multiscale_roi_align, roi_align  # noqa: F401,E402
from .pipeline import SlidePostprocessor  # noqa: F401,E402

__version__ = "0.1.0"
