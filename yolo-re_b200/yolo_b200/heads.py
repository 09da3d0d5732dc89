"""Detection heads (parameter containers; see blocks.py for why they look the way they do).

Reference: src/yolo/heads/detect.py:22-295, src/yolo/heads/dfl.py:14-50.  SegmentDFL: upstream YOLOv9's Proto
(models/common.py) and Segment (models/yolo.py) on top of DetectDFL."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .blocks import Conv, _EngineModule

REG_MAX = 16


def head_widths(ch0: int, nc: int) -> tuple[int, int]:
    """Tower widths (src/yolo/heads/detect.py:45-46)."""
    c2 = math.ceil(max(ch0 // 4, REG_MAX * 4, 16) / 4) * 4
    c3 = max(ch0, min(nc * 2, 128))
    return c2, c3


class DFL(nn.Module):
    """Holds the frozen arange(16) projection of the softmax-integral decode (dfl.py:29-35);
    the expectation itself is computed by K6 (dfl_decode_score)."""

    def __init__(self, num_bins: int = REG_MAX):
        super().__init__()
        self.num_bins = num_bins
        self.conv = nn.Conv2d(num_bins, 1, 1, bias=False).requires_grad_(False)
        self.conv.weight.data[:] = torch.arange(num_bins, dtype=torch.float).view(1, num_bins, 1, 1)


def _towers(chs, c_box, c_cls, nc):
    box = nn.ModuleList(nn.Sequential(Conv(ch, c_box, 3), Conv(c_box, c_box, 3, groups=4),
                                      nn.Conv2d(c_box, 4 * REG_MAX, 1, groups=4)) for ch in chs)
    cls = nn.ModuleList(nn.Sequential(Conv(ch, c_cls, 3), Conv(c_cls, c_cls, 3), nn.Conv2d(c_cls, nc, 1)) for ch in chs)
    return box, cls


def _init_tower_bias(box, cls, stride, nc):
    """detect.py:111-127: box bias 1.0, class bias log(5 / nc / (640/s)^2)."""
    for i, s in enumerate(stride.tolist()):
        box[i][-1].bias.data[:] = 1.0
        cls[i][-1].bias.data[:nc] = math.log(5 / nc / (640 / s) ** 2)


class DetectDFL(_EngineModule):
    def __init__(self, num_classes: int, in_channels: tuple[int, ...]):
        super().__init__()
        self.num_classes = num_classes
        self.num_levels = len(in_channels)
        self.reg_max = REG_MAX
        self.num_outputs = num_classes + 4 * REG_MAX
        c2, c3 = head_widths(in_channels[0], num_classes)
        self.box_convs, self.cls_convs = _towers(in_channels, c2, c3, num_classes)
        self.dfl = DFL(REG_MAX)
        self.stride = torch.zeros(self.num_levels)      # plain attribute, not a buffer (detect.py:68-70)

    def init_bias(self) -> None:
        _init_tower_bias(self.box_convs, self.cls_convs, self.stride, self.num_classes)


class DualDetectDFL(_EngineModule):
    """First half of the inputs feeds the auxiliary towers, second half the main ones (detect.py:130-205)."""

    def __init__(self, num_classes: int, in_channels: tuple[int, ...]):
        super().__init__()
        self.num_classes = num_classes
        self.num_levels = len(in_channels) // 2
        self.reg_max = REG_MAX
        self.num_outputs = num_classes + 4 * REG_MAX
        aux, main = in_channels[: self.num_levels], in_channels[self.num_levels:]
        c2, c3 = head_widths(aux[0], num_classes)
        c4, c5 = head_widths(main[0], num_classes)
        self.aux_box_convs, self.aux_cls_convs = _towers(aux, c2, c3, num_classes)
        self.main_box_convs, self.main_cls_convs = _towers(main, c4, c5, num_classes)
        self.dfl = DFL(REG_MAX)
        self.dfl2 = DFL(REG_MAX)
        self.stride = torch.zeros(self.num_levels)

    def init_bias(self) -> None:
        _init_tower_bias(self.aux_box_convs, self.aux_cls_convs, self.stride, self.num_classes)
        _init_tower_bias(self.main_box_convs, self.main_cls_convs, self.stride, self.num_classes)


class Proto(nn.Module):
    """Mask prototypes (upstream models/common.py Proto): Conv 3x3 -> nearest x2 upsample -> Conv 3x3 -> Conv 1x1."""

    def __init__(self, in_channels: int, num_protos: int = 256, num_masks: int = 32):
        super().__init__()
        self.cv1 = Conv(in_channels, num_protos, 3)
        self.cv2 = Conv(num_protos, num_protos, 3)
        self.cv3 = Conv(num_protos, num_masks, 1)


class SegmentDFL(DetectDFL):
    """DetectDFL plus upstream's instance-segmentation parts: the prototype branch on the first (stride-8) input and one
    mask-coefficient tower per level, Conv 3x3 -> Conv 3x3 -> Conv2d 1x1 (bias, no activation) with
    c4 = max(ch0 // 4, num_masks) channels (upstream models/yolo.py Segment)."""

    def __init__(self, num_classes: int, in_channels: tuple[int, ...], num_masks: int = 32, num_protos: int = 256):
        super().__init__(num_classes, in_channels)
        self.num_masks, self.num_protos = num_masks, num_protos
        self.proto = Proto(in_channels[0], num_protos, num_masks)
        c4 = max(in_channels[0] // 4, num_masks)
        self.mask_convs = nn.ModuleList(nn.Sequential(Conv(ch, c4, 3), Conv(c4, c4, 3), nn.Conv2d(c4, num_masks, 1))
                                        for ch in in_channels)
