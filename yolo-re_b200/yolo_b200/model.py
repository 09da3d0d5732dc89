"""YOLO model: the drop-in boundary of the B200 path.

Same public surface as the reference's ``yolo.model.model.YOLO`` (src/yolo/model/model.py:20-238):
``YOLO.from_yaml / from_config``, ``.layers`` (nn.ModuleDict), ``.connections``, ``.detect_inputs``,
``forward(x[B,C,H,W])`` returning ``(y[B,4+nc,A], [raw_i[B,64+nc,Hi,Wi]])`` in eval mode (dual
head: ``([y_aux, y_main], [raws_aux, raws_main])``; segmentation head, upstream YOLOv9's gelan-c-seg:
``(y, (raws, mc[B,32,A], proto[B,32,H/4,W/4]))``), ``state_dict``-compatible weights, model
returned in TRAIN mode (model.py:163), ``detect.stride`` a plain tensor attribute.

Differences by design: eval-mode forward is one replay of a pre-compiled libyre launch plan on the
current CUDA stream (engine.py) instead of the named-DAG interpreter loop (model.py:87-107).
Train-mode forward raises: in train mode the reference's BatchNorm layers normalise with BATCH statistics
(blocks/conv.py:85, nn.BatchNorm2d in training mode) while the launch plan folds the RUNNING statistics into
the weights, so handing back the plan's raw maps as the reference's train-mode output
(heads/detect.py:84-85) would be silently wrong; training itself (loss, optimizer groups, EMA) is out of
scope for this path.  Extension: ``forward`` also takes uint8 ``[B,H,W,3]`` BGR frames (cv2 layout) and fuses the
host-side conversion of scripts/detect.py:223-227 into the first convolution.
"""
from __future__ import annotations

from copy import deepcopy
from dataclasses import dataclass, field
from pathlib import Path

import torch
import torch.nn as nn
import yaml

from . import blocks as B
from .heads import DetectDFL, DualDetectDFL, SegmentDFL


@dataclass
class ModelConfig:
    """src/yolo/model/config.py:7-20."""
    num_classes: int = 80
    depth_multiplier: float = 1.0
    width_multiplier: float = 1.0
    layers: list[dict] = field(default_factory=list)


def parse_yaml(path) -> ModelConfig:
    """src/yolo/model/parser.py:19-30."""
    with open(path) as f:
        data = yaml.safe_load(f)
    m = data.get("model", {})
    return ModelConfig(m.get("num_classes", 80), m.get("depth_multiplier", 1.0), m.get("width_multiplier", 1.0),
                       data.get("layers", []))


def _scale_width(v: int, mult: float, div: int = 8) -> int:
    return v if mult == 1.0 else max(div, int(v * mult + div / 2) // div * div)      # parser.py:33-47


def _scale_depth(v: int, mult: float) -> int:
    return v if mult == 1.0 else max(1, round(v * mult))                              # parser.py:50-62


_STANDARD = {"Conv": B.Conv, "ADown": B.ADown, "RepNCSPELAN4": B.RepNCSPELAN4, "SPPELAN": B.SPPELAN}
# exported like the reference's registry (src/yolo/model/registry.py:14-26)
BLOCKS: dict[str, type[nn.Module]] = {**_STANDARD, "Concat": B.Concat, "Silence": B.Silence, "CBLinear": B.CBLinear,
                                      "CBFuse": B.CBFuse, "DetectDFL": DetectDFL, "DualDetectDFL": DualDetectDFL,
                                      "SegmentDFL": SegmentDFL, "Upsample": B.Upsample}


def build_layers(config: ModelConfig, input_channels: int = 3):
    """YAML layer list -> (ModuleDict, connections, detect_inputs); channel inference, default
    ``from`` = previous layer, width/depth multipliers -- src/yolo/model/parser.py:88-122, 250-280."""
    layers: dict[str, nn.Module] = {}
    connections: dict[str, str | list[str]] = {}
    chan = {"input": input_channels}
    prev = "input"
    detect_inputs: list[str] = []
    for raw in config.layers:
        p = deepcopy(raw)
        name, kind = p.pop("name"), p.pop("type")
        frm = p.pop("from", None) or prev
        if not isinstance(frm, (str, list)):
            raise TypeError(f"from must be str or list[str], got {type(frm)}")
        connections[name] = frm
        cin = [chan[n] for n in frm] if isinstance(frm, list) else [chan[frm]]
        if kind in ("DetectDFL", "DualDetectDFL", "SegmentDFL"):
            block, cout = BLOCKS[kind](config.num_classes, tuple(cin), **p), 0
            detect_inputs = frm if isinstance(frm, list) else [frm]
        elif kind == "Concat":
            block, cout = B.Concat(p.get("dimension", 1)), sum(cin)
        elif kind == "Silence":
            block, cout = B.Silence(), cin[0]
        elif kind == "Upsample":
            block, cout = B.Upsample(p.get("scale_factor", 2), p.get("mode", "nearest")), cin[0]
        elif kind == "CBLinear":
            outs = [_scale_width(c, config.width_multiplier) for c in p["out_channels_list"]]
            block, cout = B.CBLinear(cin[0], outs), outs[-1]
        elif kind == "CBFuse":
            block, cout = B.CBFuse(p["idx"]), cin[-1]
        elif kind in _STANDARD:
            for k in ("out_channels", "hidden_channels", "block_channels"):
                if k in p:
                    p[k] = _scale_width(p[k], config.width_multiplier)
            if "num_repeats" in p:
                p["num_repeats"] = _scale_depth(p["num_repeats"], config.depth_multiplier)
            block, cout = _STANDARD[kind](in_channels=cin[0], **p), p["out_channels"]
        else:
            raise ValueError(f"Unknown block type: {kind}")
        layers[name] = block
        chan[name] = cout
        prev = name
    return nn.ModuleDict(layers), connections, detect_inputs


class YOLO(nn.Module):
    def __init__(self, layers: nn.ModuleDict, connections: dict[str, str | list[str]], detect_inputs: list[str]):
        super().__init__()
        self.layers = layers
        self.connections = connections
        self.detect_inputs = detect_inputs
        self._stride_initialized = False
        # engine state (not part of the state_dict)
        self.precision = "bf16"          # "bf16" | "fp16" (tcgen05, fp32 accumulation) | "fp32" (FFMA validation mode)
        self.fresh_outputs = True        # False: return the plan's static output buffers (no allocation)
        self.check_weights = True        # re-fold when a parameter was modified in place
        self.use_cuda_graph = False      # with fresh_outputs=False: capture the launch list once per input buffer and replay it
        self.main_only = False           # dual-head models: True compiles the main branch only -> (y, raws) like a single head
        # None: one plan per input shape (batch size included).  N: one plan compiled for N images serves every forward of
        # 1..N images (same results as the first n images of a full run, shorter launches, one set of buffers); a larger
        # batch raises ValueError
        self.max_batch: int | None = None
        # None: every plan owns its buffers.  (H, W), with max_batch set: the plans of every input shape up to H x W take
        # their activations and static outputs from one shape arena sized for max_batch images of H x W, and share one
        # upload of the folded weights; a larger input raises ValueError.  Static outputs are then valid until the next
        # forward of any shape, and forwards must be ordered on one stream
        self.max_shape: tuple[int, int] | None = None
        self._plans: dict = {}
        self._arenas: dict = {}          # shape arenas (engine._arena)
        self._arena_weights: dict = {}   # per device: (weights version, packed weights shared by the arena plans)
        self._tta: dict = {}             # test-time augmentation: scaled-image buffers per (input shape, capacity)
        self.register_load_state_dict_post_hook(lambda m, _k: m.invalidate())

    # -- engine plumbing ------------------------------------------------------------------------
    def invalidate(self) -> None:
        """Drops the compiled launch plans (weights changed / moved).  Call it after edits the per-forward check cannot
        see: writes through ``.data`` and re-assignment of a whole ``nn.Parameter`` object.  Frees the plans' buffers, the
        shape arenas and their shared weights, and the test-time-augmentation image buffers with them."""
        self._plans.clear()
        self._arenas.clear()
        self._arena_weights.clear()
        self._tta.clear()
        self.__dict__.pop("_wt_tensors", None)

    def set_precision(self, precision: str) -> "YOLO":
        """"bf16" (default): tcgen05 convolutions on bf16 activations and weights.  "fp16": the same kernels on IEEE half
        operands -- 8x smaller rounding than bf16 at the same speed, but finite only up to +-65504: a folded conv weight
        beyond that fails the compile with YreError, activations beyond it become +-inf (they are not saturated), and
        weights below 2^-24 in magnitude become zero.  "fp32": the fp32-FMA validation engine.  Accumulation is fp32 in
        every mode; the raw head logits and y stay fp32."""
        if precision not in ("bf16", "fp16", "fp32"):
            raise ValueError("precision must be 'bf16', 'fp16' or 'fp32'")
        if precision != self.precision:
            self.precision = precision
            self.invalidate()
        return self

    def _apply(self, fn, *a, **k):
        self._plans = {}
        self._arenas, self._arena_weights = {}, {}
        self._tta = {}
        self.__dict__.pop("_wt_tensors", None)
        return super()._apply(fn, *a, **k)

    def train(self, mode: bool = True):
        if mode:
            self._plans = {}
            self._arenas, self._arena_weights = {}, {}
        return super().train(mode)

    def forward(self, x: torch.Tensor, augment: bool = False):
        """Eval-mode forward (see the module docstring).  augment=True: upstream's test-time augmentation (yolo_b200.tta),
        returning (y [B, 4+nc, A_tot], None) -- for a dual head the main head's merged y."""
        if self.training:
            raise NotImplementedError("train-mode forward is outside the B200 inference path (BatchNorm would need batch "
                                      "statistics; the launch plan folds the running ones): call .eval() -- YOLO.from_yaml "
                                      "returns the model in train mode, like the reference")
        from .engine import model_forward
        return model_forward(self, x, augment)

    # -- stride discovery ---------------------------------------------------------------------------
    def _detect_layer(self):
        for name, layer in self.layers.items():
            if isinstance(layer, (DetectDFL, DualDetectDFL)):
                return name, layer
        return None, None

    def graph_strides(self) -> dict[str, int]:
        """Down-sampling factor of every layer output.  The reference measures this with a 256x256
        dummy forward (model.py:109-163); it is a static property of the graph."""
        s = {"input": 1}
        for name, layer in self.layers.items():
            frm = self.connections[name]
            base = s[frm[-1]] if isinstance(layer, B.CBFuse) else s[frm if isinstance(frm, str) else frm[0]]
            if isinstance(layer, B.Conv):
                base *= layer.conv.stride[0]
            elif isinstance(layer, B.ADown):
                base *= 2
            elif isinstance(layer, B.Upsample):
                base //= layer.scale_factor
            s[name] = base
        return s

    def init_stride(self, input_size: int = 256) -> None:
        if self._stride_initialized:
            return
        name, detect = self._detect_layer()
        if detect is None:
            return
        frm = self.connections[name]
        if not isinstance(frm, list):
            raise ValueError("Detect head must have multiple inputs")
        if isinstance(detect, DualDetectDFL):
            frm = frm[detect.num_levels:]
        s = self.graph_strides()
        detect.stride = torch.tensor([float(s[n]) for n in frm])
        detect.init_bias()
        self._stride_initialized = True
        self.train()

    @classmethod
    def from_config(cls, config: ModelConfig, input_channels: int = 3) -> "YOLO":
        model = cls(*build_layers(config, input_channels))
        model.init_stride()
        return model

    @classmethod
    def from_yaml(cls, path: str | Path, input_channels: int = 3, num_classes: int | None = None) -> "YOLO":
        config = parse_yaml(path)
        if num_classes is not None:
            config.num_classes = num_classes
        return cls.from_config(config, input_channels)
