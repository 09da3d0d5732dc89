"""yolo_b200 -- B200-native (sm_100a) implementation of yolo-re's detection inference hot path.

Public names mirror the reference package (src/yolo/__init__.py:3-20) for the path in scope:
``YOLO`` (``from_yaml`` / ``from_config`` / ``forward`` / ``state_dict``) and ``non_max_suppression``.
"""
from ._lib import YreError, lib
from .engine import precision
from .model import BLOCKS, YOLO, ModelConfig, build_layers, parse_yaml
from .nms import PendingDetections, nms_raw, non_max_suppression, non_max_suppression_async
from .preprocess import letterbox, preprocess, scale_boxes, scale_rows
from .checkpoint import convert_upstream_state_dict, load_checkpoint
from .metrics import DetectionAccumulator, Evaluator, compute_map, match_detections
from .seg import masks_raw, process_mask, process_mask_native

__version__ = "0.2.0"
__all__ = ["YOLO", "non_max_suppression", "non_max_suppression_async", "PendingDetections", "scale_rows", "nms_raw", "precision", "YreError", "lib", "ModelConfig", "parse_yaml",
           "build_layers", "BLOCKS", "letterbox", "preprocess", "scale_boxes", "convert_upstream_state_dict", "load_checkpoint", "compute_map", "match_detections", "DetectionAccumulator", "Evaluator",
           "masks_raw", "process_mask", "process_mask_native"]
