"""FPN level assignment + ROIAlign / ROIPool -- drop-in for ``assign_boxes_to_levels``,
``convert_boxes_to_pooler_format``, ``ROIAlign`` and ``ROIPooler`` of the reference
(python/src/models/modules/roi_poolers.py:15-331), forward and backward (gradients flow to the feature maps, as through
torchvision's roi_align / roi_pool).

The reference loops over the pyramid levels with nonzero / gather / torchvision ``roi_align`` or ``roi_pool`` /
``index_put_``; here one kernel computes every box's level (det_roi_levels) and one kernel pools all levels
(det_roi_align_levels_typed, det_roi_pool_levels).  Third-party arithmetic: torchvision.ops.roi_align / roi_pool
(un-vendored) -- the parity oracle is the installed CPU kernel.

bf16 / fp16 feature pyramids are read natively: the kernels widen each element to fp32, compute in fp32 and round the
output once to the feature dtype, bit-identical to the fp32 route on ``f.float()`` followed by ``.to(dtype)``
(torchvision's autocast rule).  Gradients accumulate in fp32 and are returned in each feature map's dtype."""
import ctypes
import math
from typing import List, Sequence, Tuple, Union

import torch

from . import _native as N
from .structures import Boxes


def _box_tensors(box_lists: Sequence) -> List[torch.Tensor]:
    return [b.tensor if isinstance(b, Boxes) else b for b in box_lists]


def convert_boxes_to_pooler_format(box_lists: Sequence) -> torch.Tensor:
    """(M,5) rows (batch index, x0, y0, x1, y1) -- reference roi_poolers.py:141-166."""
    ts = _box_tensors(box_lists)
    return torch.cat([torch.cat((torch.full_like(t[:, :1], i), t), dim=1) for i, t in enumerate(ts)], dim=0)


def assign_boxes_to_levels(box_lists: Sequence, min_level: int, max_level: int, canonical_box_size: int,
                           canonical_level: int) -> torch.Tensor:
    """int64 (M,) level offsets from ``min_level`` -- reference roi_poolers.py:103-131 (Eqn.(1) of the FPN paper)."""
    boxes = N.f32c(torch.cat(_box_tensors(box_lists), dim=0))
    N.require_cuda(boxes)
    out = torch.empty((boxes.shape[0],), dtype=torch.int64, device=boxes.device)
    if boxes.shape[0]:
        with torch.cuda.device(boxes.device):
            N.call("det_roi_levels", N.ptr(boxes), boxes.shape[0], int(min_level), int(max_level),
                   float(canonical_box_size), int(canonical_level), N.ptr(out), N.stream())
    return out


def _level_table(tensors, scales):
    lv = (N.FeatureLevel * len(tensors))()
    for i, (f, s) in enumerate(zip(tensors, scales)):
        lv[i].data, lv[i].h, lv[i].w, lv[i].spatial_scale, lv[i].reserved = f.data_ptr(), f.shape[2], f.shape[3], float(s), 0
    return lv


def _feature_route(features: Sequence[torch.Tensor]) -> Tuple[List[torch.Tensor], int]:
    """(feature maps for the kernels, DET_DTYPE_* code), for both poolers.  When every level is fp32, bf16 or fp16 alike
    the maps are read in their dtype (contiguous; the kernels widen each element to fp32 on load); anything else (mixed
    dtypes, fp64) is converted to fp32.  No detach: the returned tensors keep the autograd graph of the inputs."""
    dts = {f.dtype for f in features}
    if len(dts) == 1 and features[0].dtype in N.DTYPE_CODES:
        return [f.contiguous() for f in features], N.DTYPE_CODES[features[0].dtype]
    return [f.to(torch.float32).contiguous() for f in features], N.DTYPE_CODES[torch.float32]


def _grad_route(grad_out: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """grad_out read in its own dtype (no fp32 copy) when the kernels take it, else as fp32."""
    if grad_out.dtype in N.DTYPE_CODES:
        return grad_out.contiguous(), N.DTYPE_CODES[grad_out.dtype]
    return grad_out.contiguous().float(), N.DTYPE_CODES[torch.float32]


class _RoiAlignLevels(torch.autograd.Function):
    """forward: det_roi_align_levels_typed; backward: det_roi_align_levels_backward_typed (gradients w.r.t. the feature
    maps, accumulated in fp32 and returned in each map's dtype)."""

    @staticmethod
    def forward(ctx, boxes, batch_index, level, scales, output_size, sampling_ratio, aligned, code, *feats):
        n, c = feats[0].shape[0], feats[0].shape[1]
        m = boxes.shape[0]
        out = torch.empty((m, c, output_size[0], output_size[1]), dtype=feats[0].dtype, device=boxes.device)
        if m:
            lv = _level_table(feats, scales)
            with torch.cuda.device(boxes.device):
                N.call("det_roi_align_levels_typed", ctypes.cast(lv, ctypes.c_void_p), len(feats), n, c, N.ptr(boxes),
                       N.ptr(batch_index), N.ptr(level), m, int(output_size[0]), int(output_size[1]), int(sampling_ratio),
                       int(bool(aligned)), N.ptr(out), code, N.stream())
        ctx.save_for_backward(boxes, batch_index, level if level is not None else torch.empty(0, device=boxes.device))
        ctx.meta = (scales, output_size, sampling_ratio, aligned, [(tuple(f.shape), f.dtype) for f in feats],
                    level is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        boxes, batch_index, level = ctx.saved_tensors
        scales, output_size, sampling_ratio, aligned, shapes, has_level = ctx.meta
        grads = [torch.zeros(sh, dtype=torch.float32, device=boxes.device) for sh, _ in shapes]
        m = boxes.shape[0]
        if m:
            go, gcode = _grad_route(grad_out)
            lv = _level_table(grads, scales)
            with torch.cuda.device(boxes.device):
                N.call("det_roi_align_levels_backward_typed", ctypes.cast(lv, ctypes.c_void_p), len(grads),
                       shapes[0][0][0], shapes[0][0][1], N.ptr(boxes), N.ptr(batch_index),
                       N.ptr(level if has_level else None), m, int(output_size[0]), int(output_size[1]),
                       int(sampling_ratio), int(bool(aligned)), N.ptr(go), gcode, N.stream())
        return (None,) * 8 + tuple(g.to(dt) for g, (_, dt) in zip(grads, shapes))


class _RoiPoolLevels(torch.autograd.Function):
    """forward: det_roi_pool_levels; backward: det_roi_pool_levels_backward.  argmax is written and saved only when some
    feature map requires grad (inference passes NULL and writes no argmax bytes)."""

    @staticmethod
    def forward(ctx, boxes, batch_index, level, scales, output_size, code, *feats):
        n, c = feats[0].shape[0], feats[0].shape[1]
        m = boxes.shape[0]
        out = torch.empty((m, c, output_size[0], output_size[1]), dtype=feats[0].dtype, device=boxes.device)
        argmax = None
        if any(ctx.needs_input_grad[6:]):
            argmax = torch.empty(out.shape, dtype=torch.int32, device=boxes.device)
        if m:
            lv = _level_table(feats, scales)
            with torch.cuda.device(boxes.device):
                N.call("det_roi_pool_levels", ctypes.cast(lv, ctypes.c_void_p), len(feats), n, c, N.ptr(boxes),
                       N.ptr(batch_index), N.ptr(level), m, int(output_size[0]), int(output_size[1]), N.ptr(out),
                       N.ptr(argmax), code, N.stream())
        if argmax is not None:
            ctx.save_for_backward(batch_index, level if level is not None else torch.empty(0, device=boxes.device),
                                  argmax)
        ctx.meta = (scales, output_size, [(tuple(f.shape), f.dtype) for f in feats], level is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        batch_index, level, argmax = ctx.saved_tensors
        scales, output_size, shapes, has_level = ctx.meta
        grads = [torch.zeros(sh, dtype=torch.float32, device=grad_out.device) for sh, _ in shapes]
        m = argmax.shape[0]
        if m:
            go, gcode = _grad_route(grad_out)
            lv = _level_table(grads, scales)
            with torch.cuda.device(grad_out.device):
                N.call("det_roi_pool_levels_backward", ctypes.cast(lv, ctypes.c_void_p), len(grads), shapes[0][0][0],
                       shapes[0][0][1], N.ptr(batch_index), N.ptr(level if has_level else None), m,
                       int(output_size[0]), int(output_size[1]), N.ptr(argmax), N.ptr(go), gcode, N.stream())
        return (None,) * 6 + tuple(g.to(dt) for g, (_, dt) in zip(grads, shapes))


def _pool_inputs(features: List[torch.Tensor], boxes: torch.Tensor, batch_index: torch.Tensor):
    """the feature route, shape checks and kernel-ready boxes / batch indices shared by both poolers"""
    N.require_cuda(boxes, *features)
    feats, code = _feature_route(features)
    n, c = feats[0].shape[0], feats[0].shape[1]
    for f in feats:
        assert f.dim() == 4 and f.shape[0] == n and f.shape[1] == c, "feature maps must share batch and channels"
    return feats, code, N.f32c(boxes), batch_index.to(torch.int32).contiguous()


def _roi_align_levels(features: List[torch.Tensor], scales: Sequence[float], boxes: torch.Tensor,
                      batch_index: torch.Tensor, level, output_size: Tuple[int, int], sampling_ratio: int,
                      aligned: bool) -> torch.Tensor:
    feats, code, b, bi = _pool_inputs(features, boxes, batch_index)
    out = _RoiAlignLevels.apply(b, bi, level, tuple(float(s) for s in scales), tuple(output_size), int(sampling_ratio),
                                bool(aligned), code, *feats)
    # the result carries the feature maps' dtype like torchvision.ops.roi_align's does (fp32 route: cast back)
    return out if out.dtype == features[0].dtype else out.to(features[0].dtype)


def _roi_pool_levels(features: List[torch.Tensor], scales: Sequence[float], boxes: torch.Tensor,
                     batch_index: torch.Tensor, level, output_size: Tuple[int, int]) -> torch.Tensor:
    feats, code, b, bi = _pool_inputs(features, boxes, batch_index)
    out = _RoiPoolLevels.apply(b, bi, level, tuple(float(s) for s in scales), tuple(output_size), code, *feats)
    return out if out.dtype == features[0].dtype else out.to(features[0].dtype)


class ROIAlign:
    """reference roi_poolers.py:15-98: ``forward(input NCHW, rois (B,5))`` -> (B, C, oh, ow)."""

    def __init__(self, output_size: Tuple[int, int], spatial_scale: float, sampling_ratio: int, aligned: bool = True):
        self.output_size = (int(output_size[0]), int(output_size[1]))
        self.spatial_scale = float(spatial_scale)
        self.sampling_ratio = int(sampling_ratio)
        self.aligned = bool(aligned)

    @classmethod
    def build(cls, conf):
        return cls(conf.output_size, conf.spatial_scale, getattr(conf, "sampling_ration", getattr(conf, "sampling_ratio", 0)),
                   conf.aligned)

    def forward(self, input: torch.Tensor, rois: torch.Tensor) -> torch.Tensor:
        assert rois.dim() == 2 and rois.size(1) == 5
        r = rois.to(dtype=torch.float32)
        return _roi_align_levels([input], [self.spatial_scale], r[:, 1:5].contiguous(), r[:, 0], None, self.output_size,
                                 self.sampling_ratio, self.aligned)

    __call__ = forward

    def __repr__(self):
        return (f"ROIAlign(output_size={self.output_size}, spatial_scale={self.spatial_scale}, "
                f"sampling_ratio={self.sampling_ratio}, aligned={self.aligned})")


class ROIPooler:
    """reference roi_poolers.py:168-331: pools every box from the pyramid level its size selects."""

    def __init__(self, scales: List[float], sampling_ratio: int, output_size: Union[int, Tuple[int, int], List[int]],
                 type: str, canonical_box_size: int = 224, canonical_level: int = 4):
        if isinstance(output_size, int):
            output_size = (output_size, output_size)
        assert len(output_size) == 2 and isinstance(output_size[0], int) and isinstance(output_size[1], int)
        self.output_size = (output_size[0], output_size[1])
        if type not in ("ROIAlign", "ROIAlignV2", "ROIPool"):
            raise ValueError("Unknown pooler type: {}".format(type))
        self.type = type
        self.aligned = type == "ROIAlignV2"  # ROIAlign: legacy half-pixel-free sampling; ROIPool: not used
        self.scales = [float(s) for s in scales]
        self.sampling_ratio = int(sampling_ratio)
        min_level, max_level = -(math.log2(scales[0])), -(math.log2(scales[-1]))
        assert math.isclose(min_level, int(min_level)) and math.isclose(max_level, int(max_level)), \
            "Featuremap stride is not power of 2!"
        self.min_level, self.max_level = int(min_level), int(max_level)
        assert len(scales) == self.max_level - self.min_level + 1, \
            "[ROIPooler] Sizes of input featuremaps do not form a pyramid!"
        assert 0 <= self.min_level <= self.max_level
        assert canonical_box_size > 0
        self.canonical_level, self.canonical_box_size = canonical_level, canonical_box_size

    @classmethod
    def build(cls, conf, scales: List[float]):
        return cls(scales=scales, output_size=conf.output_size, sampling_ratio=conf.sampling_ratio, type=conf.type,
                   canonical_box_size=conf.canonical_box_size, canonical_level=conf.canonical_level)

    def forward(self, x: List[torch.Tensor], box_lists: List[Boxes]) -> torch.Tensor:
        nl = len(self.scales)
        assert isinstance(x, list) and isinstance(box_lists, list), "Arguments to pooler must be lists"
        assert len(x) == nl, f"unequal value, num_level_assignments={nl}, but x is list of {len(x)} Tensors"
        assert len(box_lists) == x[0].size(0), \
            f"unequal value, x[0] batch dim 0 is {x[0].size(0)}, but box_list has length {len(box_lists)}"
        if len(box_lists) == 0:
            return torch.zeros((0, x[0].shape[1]) + self.output_size, device=x[0].device, dtype=x[0].dtype)
        ts = _box_tensors(box_lists)
        boxes = N.f32c(torch.cat(ts, dim=0))
        batch_index = torch.cat([torch.full((t.shape[0],), i, dtype=torch.int32, device=boxes.device)
                                 for i, t in enumerate(ts)])
        level = None
        if nl > 1:
            level = assign_boxes_to_levels(ts, self.min_level, self.max_level, self.canonical_box_size,
                                           self.canonical_level)
        if self.type == "ROIPool":
            return _roi_pool_levels(x, self.scales, boxes, batch_index, level, self.output_size)
        return _roi_align_levels(x, self.scales, boxes, batch_index, level, self.output_size, self.sampling_ratio,
                                 self.aligned)

    __call__ = forward
