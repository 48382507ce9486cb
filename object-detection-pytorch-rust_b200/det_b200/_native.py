"""ctypes binding of libdet_b200.so (the C ABI declared in include/det_b200.h).

There is deliberately NO fallback: if the shared library is missing it is built with nvcc, and if that fails the
import raises.  Every op of the package goes through :func:`call`, which raises on a non-zero status.
"""
import ctypes
import os
import sys

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_lib", "libdet_b200.so")

c_p = ctypes.c_void_p
c_i = ctypes.c_int
c_l = ctypes.c_int64
c_f = ctypes.c_float
c_d = ctypes.c_double
c_u64 = ctypes.c_uint64

# name -> (restype, argtypes); must list every DET_API symbol of include/det_b200.h
PROTOTYPES = {
    "det_abi_version": (c_i, []),
    "det_last_error": (ctypes.c_char_p, []),
    "det_sm_count": (c_i, []),
    "det_pairwise_overlap": (c_i, [c_p, c_l, c_p, c_l, c_i, c_p, c_p]),
    "det_matched_iou": (c_i, [c_p, c_p, c_l, c_p, c_p]),
    "det_apply_deltas": (c_i, [c_p, c_p, c_l, c_i, c_f, c_f, c_f, c_f, c_f, c_p, c_p]),
    "det_apply_deltas_backward": (c_i, [c_p, c_p, c_p, c_l, c_i, c_f, c_f, c_f, c_f, c_f, c_p, c_p, c_p]),
    "det_get_deltas": (c_i, [c_p, c_p, c_l, c_f, c_f, c_f, c_f, c_p, c_p, c_p]),
    "det_grid_anchors": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p]),
    "det_rpn_decode_level": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_f, c_p, c_f, c_f, c_f, c_f, c_f, c_p, c_p,
                                   c_l, c_l, c_p]),
    "det_rpn_decode": (c_i, [c_p, c_i, c_i, c_i, c_f, c_f, c_f, c_f, c_f, c_f, c_p, c_p, c_l, c_p]),
    "det_rpn_decode_typed": (c_i, [c_p, c_i, c_i, c_i, c_f, c_f, c_f, c_f, c_f, c_f, c_p, c_p, c_l, c_i, c_p]),
    "det_nms_workspace_bytes": (c_l, [c_i, c_l]),
    "det_nms_batched": (c_i, [c_p, c_p, c_p, c_p, c_i, c_l, c_d, c_i, c_l, c_p, c_p, c_p, c_l, c_p]),
    "det_rpn_proposals_workspace_bytes": (c_l, [c_i, c_l]),
    "det_rpn_proposals": (c_i, [c_p, c_p, c_i, c_l, c_p, c_i, c_p, c_d, c_l, c_l, c_f, c_p, c_p, c_p, c_p, c_p, c_l,
                                c_p]),
    "det_yolo_decode_nms": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_i, c_f, c_d, c_i, c_p, c_p, c_p, c_l,
                                  c_p, c_p, c_p, c_p, c_p]),
    "det_yolo_decode_nms_i32": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_i, c_f, c_d, c_i, c_p, c_p, c_p, c_l,
                                      c_p, c_p, c_p, c_p, c_p]),
    "det_yolo_decode_nms_typed": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_i, c_f, c_d, c_i, c_p, c_p,
                                        c_p, c_l, c_p, c_i, c_p, c_p, c_p, c_p]),
    "det_dense_decode_level": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_p, c_p, c_p, c_l, c_l, c_p]),
    "det_dense_decode": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_l, c_p]),
    "det_dense_decode_typed": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_l, c_i, c_p]),
    "det_dense_detect_workspace_bytes": (c_l, [c_i, c_l]),
    "det_dense_detect_counter_bytes": (c_l, [c_i]),
    "det_dense_detect": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_f, c_d, c_i, c_i, c_l, c_l, c_p, c_p, c_p, c_p, c_p, c_p,
                               c_p, c_l, c_p]),
    "det_dense_detect_typed": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_f, c_d, c_i, c_i, c_l, c_l, c_p, c_p, c_p, c_p, c_p,
                                     c_p, c_p, c_l, c_i, c_p]),
    "det_threshold_compact": (c_i, [c_p, c_p, c_p, c_i, c_l, c_f, c_l, c_p, c_p, c_p, c_p, c_p, c_p]),
    "det_gather_detections": (c_i, [c_p, c_p, c_i, c_l, c_p, c_p, c_p, c_p, c_l, c_p, c_p, c_p, c_p, c_p]),
    "det_peer_sums_publish": (c_i, [c_p, c_i, c_i, c_i, c_p, c_i, c_i, ctypes.c_uint32, c_p]),
    "det_peer_sums_collect": (c_i, [c_p, c_i, c_i, c_p, c_i, c_i, ctypes.c_uint32, c_l, c_p, c_p]),
    "det_peer_sums_exchange": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p, c_i, ctypes.c_uint32, ctypes.c_uint32, c_l, c_p, c_p]),
    "det_peer_sums_exchange_dev": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p, c_i, c_p, ctypes.c_uint32, c_l, c_p, c_p]),
    "det_yolo_loss_peer": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_f, c_f, c_p, c_p,
                                 c_p, c_p, c_p, c_p]),
    "det_roi_levels": (c_i, [c_p, c_l, c_i, c_i, c_f, c_i, c_p, c_p]),
    "det_roi_align_levels": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_i, c_i, c_p, c_p]),
    "det_roi_align_levels_backward": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_i, c_i, c_p, c_p]),
    "det_roi_align_levels_typed": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_i, c_i, c_p, c_i, c_p]),
    "det_roi_align_levels_backward_typed": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_i, c_i, c_p, c_i,
                                                  c_p]),
    "det_roi_pool_levels": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_p, c_p, c_i, c_p]),
    "det_roi_pool_levels_backward": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_l, c_i, c_i, c_p, c_p, c_i, c_p]),
    "det_roi_detect_workspace_bytes": (c_l, [c_i, c_l]),
    "det_roi_detect_counter_bytes": (c_l, [c_i]),
    "det_roi_detect_typed": (c_i, [c_p, c_p, c_i, c_p, c_p, c_i, c_l, c_i, c_i, c_p, c_f, c_f, c_f, c_f, c_f, c_f, c_d,
                                   c_i, c_i, c_l, c_l, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_l, c_p]),
    "det_roi_decode_dense_typed": (c_i, [c_p, c_p, c_i, c_p, c_p, c_i, c_l, c_i, c_i, c_p, c_f, c_f, c_f, c_f, c_f, c_i,
                                         c_i, c_p, c_p, c_p]),
    "det_fast_rcnn_loss_typed": (c_i, [c_p, c_p, c_i, c_p, c_p, c_p, c_l, c_i, c_i, c_f, c_f, c_f, c_f, c_f, c_i, c_f,
                                       c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p]),
    "det_roi_sample_workspace_bytes": (c_l, [c_i, c_l, c_l]),
    "det_roi_sample_proposals": (c_i, [c_p, c_p, c_i, c_l, c_p, c_p, c_p, c_l, c_i, c_p, c_p, c_i, c_i, c_i, c_d, c_i,
                                       c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_l, c_p]),
    "det_match_workspace_bytes": (c_l, [c_i, c_l, c_l]),
    "det_match_anchors": (c_i, [c_p, c_p, c_i, c_l, c_p, c_l, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_l, c_p]),
    "det_match_grid_workspace_bytes": (c_l, [c_i, c_l, c_p, c_i]),
    "det_match_grid": (c_i, [c_p, c_p, c_i, c_l, c_p, c_l, c_p, c_i, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p,
                             c_i, c_p, c_l, c_p]),
    "det_subsample_labels_grid": (c_i, [c_p, c_i, c_l, c_i, c_d, c_u64, c_p, c_p, c_i, c_p, c_p, c_i, c_p]),
    "det_rpn_loss_sampled": (c_i, [c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                   c_i, c_l, c_f, c_f, c_f, c_f, c_f, c_i, c_f, c_f, c_f, c_p, c_p, c_p, c_p]),
    "det_assign_sampled_workspace_bytes": (c_l, [c_i, c_l, c_i]),
    "det_assign_sampled": (c_i, [c_p, c_p, c_i, c_l, c_p, c_l, c_p, c_i, c_i, c_p, c_p, c_i, c_i, c_i, c_d, c_u64, c_p, c_p,
                                 c_p, c_p, c_i, c_p, c_l, c_p]),
    "det_match_quality": (c_i, [c_p, c_l, c_l, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_l, c_p]),
    "det_subsample_labels": (c_i, [c_p, c_i, c_l, c_i, c_d, c_u64, c_p]),
    "det_rpn_loss": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_l, c_f, c_f, c_f, c_f, c_f, c_i, c_f, c_f, c_f,
                           c_p, c_p, c_p, c_p, c_p, c_p]),
    "det_yolo_loss": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_f, c_f, c_f, c_p, c_p,
                            c_p, c_p, c_p]),
}



class DenseLevel(ctypes.Structure):
    """det_dense_level_t of include/det_b200.h"""
    _fields_ = [("head", c_p), ("anchors_wh", c_p), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
                ("stride", ctypes.c_int32), ("reserved", ctypes.c_int32), ("out_offset", c_l)]


class RpnLevel(ctypes.Structure):
    """det_rpn_level_t of include/det_b200.h"""
    _fields_ = [("objectness", c_p), ("deltas", c_p), ("cell_anchors", c_p), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
                ("stride", ctypes.c_int32), ("reserved", ctypes.c_int32), ("out_offset", c_l)]


class AnchorLevel(ctypes.Structure):
    """det_anchor_level_t of include/det_b200.h"""
    _fields_ = [("h", ctypes.c_int32), ("w", ctypes.c_int32), ("stride", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("first_row", c_l)]


class HeadLevel(ctypes.Structure):
    """det_head_level_t of include/det_b200.h"""
    _fields_ = [("objectness", c_p), ("deltas", c_p), ("grad_objectness", c_p), ("grad_deltas", c_p),
                ("h", ctypes.c_int32), ("w", ctypes.c_int32)]


class PeerCtx(ctypes.Structure):
    """det_peer_ctx_t of include/det_b200.h"""
    _fields_ = [("peers_dev", c_p), ("out", c_p), ("error_flag", c_p), ("done_counter", c_p), ("timeout_ns", c_l),
                ("width", ctypes.c_int32), ("rank", ctypes.c_int32), ("world", ctypes.c_int32), ("slots", ctypes.c_int32),
                ("stamp", ctypes.c_uint32), ("lag", ctypes.c_uint32), ("stamp_counter", c_p)]


class FeatureLevel(ctypes.Structure):
    """det_feature_level_t of include/det_b200.h"""
    _fields_ = [("data", c_p), ("h", ctypes.c_int32), ("w", ctypes.c_int32), ("spatial_scale", c_f),
                ("reserved", ctypes.c_int32)]


_lib = None


def _build():
    """object-detection-pytorch-rust_b200/build.py: a no-op when the in-tree .so matches the hash of the sources."""
    sys.path.insert(0, os.path.dirname(_HERE))
    try:
        import build as _b
        _b.build()
    finally:
        sys.path.pop(0)


def lib():
    """Load the shared library, (re)building it first when it is missing or STALE: build.needs_build() compares the hash
    of csrc/ + include/ + the nvcc flags with the one recorded next to the .so, so an edited kernel can never run
    against an old binary.  Raises if the library cannot be produced -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    try:
        _build()
    except Exception as e:  # noqa: BLE001
        raise ImportError(
            f"det_b200: native library {_LIB_PATH} is missing or stale and could not be built ({e}). "
            "There is no CPU or PyTorch fallback for this package.") from e
    handle = ctypes.CDLL(_LIB_PATH)
    handle.det_abi_version.restype = c_i
    if handle.det_abi_version() != 3:
        raise ImportError("det_b200: ABI version mismatch")
    _lib = handle
    return _lib


_bound = {}


def fn(name):
    """Typed entry point `name`; AttributeError if the library does not export it (never a silent fallback)."""
    f = _bound.get(name)
    if f is None:
        f = getattr(lib(), name)
        f.restype, f.argtypes = PROTOTYPES[name]
        _bound[name] = f
    return f


def missing_symbols():
    """Names declared in include/det_b200.h (== PROTOTYPES) that the loaded library does not export."""
    return [n for n in PROTOTYPES if not hasattr(lib(), n)]


class DetError(RuntimeError):
    pass


def call(name, *args):
    rc = fn(name)(*args)
    if rc != 0:
        msg = fn("det_last_error")().decode("utf-8", "replace")
        raise DetError(f"{name} failed with status {rc}: {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("det_b200 runs on CUDA tensors only (there is no CPU fallback); got a "
                               f"{t.device.type} tensor")


_accumulators = {}


def accumulators(device) -> torch.Tensor:
    """The 16-float scratch the loss kernels accumulate into (include/det_b200.h: zero before the first call, re-armed by
    every launch): one per (device, stream), created once -- no per-step memset."""
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    t = _accumulators.get(key)
    if t is None:
        t = torch.zeros((16,), dtype=torch.float32, device=device)
        _accumulators[key] = t
    return t


def f32c(t):
    """contiguous fp32 view/copy (the reference forces boxes to fp32, structures/boxes.py:21), 16-byte aligned as the
    box kernels require: a view can be contiguous and still start inside a row, e.g. rois[:, 1:5] of a single roi."""
    t = t.detach().to(torch.float32).contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


# DET_DTYPE_* of include/det_b200.h: head element types the decode kernels read natively (widened to fp32 on load)
DTYPE_CODES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def heads_c(tensors):
    """(list of head tensors, DET_DTYPE_* code) for the *_typed entry points.  When every tensor is fp32, bf16 or fp16
    and they all share that dtype, each is kept in it -- contiguous and 16-byte aligned, copied only where it is not --
    so a 16-bit head is read as it is (no fp32 copy; the result is bit-identical to the fp32 path on h.float()).
    Anything else (fp64, mixed dtypes) goes through f32c, code 0."""
    tensors = list(tensors)
    dts = {t.dtype for t in tensors}
    if len(dts) != 1 or next(iter(dts)) not in DTYPE_CODES:
        return [f32c(t) for t in tensors], 0
    out = []
    for t in tensors:
        t = t.detach().contiguous()
        out.append(t if t.data_ptr() % 16 == 0 else t.clone())
    return out, DTYPE_CODES[tensors[0].dtype]
