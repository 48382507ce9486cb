"""NMS -- drop-in for ``batched_nms`` (reference python/src/utils.py:96-119) and the torchvision ``nms`` it wraps,
plus the batch-of-images form the kernels are built for.  Arithmetic: det_nms_batched (csrc/nms*.cu*)."""
from typing import Optional, Tuple

import torch

from . import _native as N

MODE_AUTO, MODE_PER_CATEGORY, MODE_OFFSET_TRICK = 0, 1, 2
MAX_BOXES_PER_IMAGE = 131071
MAX_CATEGORY = 32766


def nms_workspace_bytes(n: int, m: int) -> int:
    """Bytes of scratch det_nms_batched needs for n images of at most m boxes (det_nms_workspace_bytes)."""
    return int(N.fn("det_nms_workspace_bytes")(int(n), int(m)))


def nms_images(boxes: torch.Tensor, scores: torch.Tensor, categories: Optional[torch.Tensor],
               counts: Optional[torch.Tensor], iou_threshold: float, max_out: Optional[int] = None,
               mode: int = MODE_AUTO, workspace: Optional[torch.Tensor] = None,
               out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Whole-batch NMS.  boxes (N,M,4), scores (N,M), categories (N,M) int64 or None, counts (N) int32 or None.
    Returns (keep (N,max_out) int64 padded, keep_counts (N) int32); no host synchronisation.
    workspace (uint8, >= nms_workspace_bytes(N, M)) and out = (keep, keep_counts) let a serving loop run without any
    per-call allocation."""
    N.require_cuda(boxes, scores, categories, counts)
    assert boxes.dim() == 3 and boxes.shape[-1] == 4
    n, m = boxes.shape[0], boxes.shape[1]
    b, s = N.f32c(boxes), N.f32c(scores)
    c = None if categories is None else categories.detach().to(torch.int64).contiguous()
    k = None if counts is None else counts.detach().to(torch.int32).contiguous()
    max_out = m if max_out is None else int(max_out)
    if out is None:
        keep = torch.empty((n, max_out), dtype=torch.int64, device=b.device)
        keep_counts = torch.empty((n,), dtype=torch.int32, device=b.device)
    else:
        keep, keep_counts = out
        assert keep.shape == (n, max_out) and keep.dtype == torch.int64 and keep.is_contiguous()
        assert keep_counts.shape == (n,) and keep_counts.dtype == torch.int32
    if n == 0:
        return keep, keep_counts
    wsb = N.fn("det_nms_workspace_bytes")(n, m)
    ws = workspace
    if ws is None or ws.numel() < wsb or ws.dtype != torch.uint8 or ws.device != b.device:
        ws = torch.empty((wsb,), dtype=torch.uint8, device=b.device)
    with torch.cuda.device(b.device):
        N.call("det_nms_batched", N.ptr(b), N.ptr(s), N.ptr(c), N.ptr(k), n, m, float(iou_threshold), int(mode),
               max_out, N.ptr(keep), N.ptr(keep_counts), N.ptr(ws), wsb, N.stream())
    return keep, keep_counts


# ---- the candidate-list detectors (det_dense_detect, det_roi_detect): padded output, workspace, exact unfused route

class DenseDetectWorkspace:
    """Scratch memory of det_dense_detect that is used for nothing else: the per-image candidate counters at its head are
    zeroed once here and every call leaves them zero, so ``detect_thresholded(..., workspace=this)`` is exactly two
    launches (no memset node).  One object per stream of calls in flight."""

    def __init__(self, n: int, cand_cap: int, device):
        self.n, self.cand_cap, self.device = int(n), int(cand_cap), self._norm(device)
        nbytes = N.fn("det_dense_detect_workspace_bytes")(self.n, self.cand_cap)
        self.buf = torch.empty((nbytes,), dtype=torch.uint8, device=self.device)
        self.buf[:N.fn("det_dense_detect_counter_bytes")(self.n)].zero_()

    @staticmethod
    def _norm(device) -> torch.device:
        d = torch.device(device)
        return torch.device("cuda", torch.cuda.current_device()) if d.type == "cuda" and d.index is None else d

    def claim(self, n: int, cand_cap: int, device) -> torch.Tensor:
        if (n, cand_cap) != (self.n, self.cand_cap) or self._norm(device) != self.device:
            raise ValueError(f"DenseDetectWorkspace was built for n={self.n}, cand_cap={self.cand_cap} on {self.device}")
        return self.buf


def detection_buffers(n: int, max_det: int, device) -> dict:
    """The padded detection dict: idx (n,max_det) int64, boxes (n,max_det,4), scores (n,max_det), classes (n,max_det)
    int64, count (n) int32, overflow (1) int32."""
    return {"idx": torch.empty((n, max_det), dtype=torch.int64, device=device),
            "boxes": torch.empty((n, max_det, 4), dtype=torch.float32, device=device),
            "scores": torch.empty((n, max_det), dtype=torch.float32, device=device),
            "classes": torch.empty((n, max_det), dtype=torch.int64, device=device),
            "count": torch.empty((n,), dtype=torch.int32, device=device),
            "overflow": torch.empty((1,), dtype=torch.int32, device=device)}


def detect_workspace(workspace, n: int, cand_cap: int, device) -> Tuple[torch.Tensor, int, int]:
    """(buffer, nbytes, gate bit 1) for the `workspace` argument of a candidate-list detector: a DenseDetectWorkspace is
    claimed (its counters are zero: gate bit 1 set, no memset node); any other buffer is used as it is unless it is None
    or smaller than det_dense_detect_workspace_bytes(n, cand_cap), in which case a fresh one is allocated."""
    wsb = N.fn("det_dense_detect_workspace_bytes")(n, cand_cap)
    if isinstance(workspace, DenseDetectWorkspace):
        return workspace.claim(n, cand_cap, device), wsb, 2
    if workspace is None or workspace.numel() < wsb:
        workspace = torch.empty((wsb,), dtype=torch.uint8, device=device)
    return workspace, wsb, 0


def detect_unfused(boxes: torch.Tensor, scores: torch.Tensor, classes: Optional[torch.Tensor], score_thresh: float,
                   iou_thresh: float, max_det: int, mode: int = MODE_AUTO) -> dict:
    """The exact route of the candidate-list detectors for any candidate count (up to MAX_BOXES_PER_IMAGE per image):
    boxes (n,R,4), scores (n,R), classes (n,R) int64 or None -> det_threshold_compact (score > score_thresh, in row
    order) -> det_nms_batched -> det_gather_detections.  Returns the padded detection dict with overflow 0; idx is the
    row in [0, R).  Library kernels only, no host synchronisation."""
    n, R = scores.shape
    dev = scores.device
    cap = max(int(R), 1)
    out = detection_buffers(n, max_det, dev)
    out["overflow"].zero_()
    if n == 0 or R == 0:
        out["count"].zero_()
        return out
    rows = torch.empty((n, cap), dtype=torch.int64, device=dev)
    cb = torch.empty((n, cap, 4), dtype=torch.float32, device=dev)
    cs = torch.empty((n, cap), dtype=torch.float32, device=dev)
    cc = torch.empty((n, cap), dtype=torch.int64, device=dev)
    counts = torch.empty((n,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        N.call("det_threshold_compact", N.ptr(boxes), N.ptr(scores), N.ptr(classes), n, R, float(score_thresh), cap,
               N.ptr(rows), N.ptr(cb), N.ptr(cs), N.ptr(cc), N.ptr(counts), N.stream())
    keep, out["count"] = nms_images(cb, cs, cc, counts, iou_thresh, max_det, mode)
    with torch.cuda.device(dev):
        N.call("det_gather_detections", N.ptr(keep), N.ptr(out["count"]), n, max_det, N.ptr(rows), N.ptr(cb),
               N.ptr(cs), N.ptr(cc), cap, N.ptr(out["idx"]), N.ptr(out["boxes"]), N.ptr(out["scores"]),
               N.ptr(out["classes"]), N.stream())
    return out


def batched_nms(boxes: torch.Tensor, scores: torch.Tensor, idxs: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    """Same contract as the reference: int64 kept indices by descending score (python/src/utils.py:96)."""
    assert boxes.shape[-1] == 4
    if boxes.shape[0] == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    keep, cnt = nms_images(boxes[None], scores[None], idxs[None], None, iou_threshold)
    k = int(cnt.item())
    if k < 0:
        raise ValueError(f"batched_nms: category ids must lie in [0, {MAX_CATEGORY}]")
    return keep[0, :k]


def nms(boxes: torch.Tensor, scores: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    """torchvision.ops.nms contract (single category)."""
    if boxes.shape[0] == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    keep, cnt = nms_images(boxes[None], scores[None], None, None, iou_threshold, mode=MODE_PER_CATEGORY)
    return keep[0, :int(cnt.item())]
