"""TEST INFRASTRUCTURE ONLY -- CPU/GPU oracle of the second-stage (Fast R-CNN box predictor) inference that
det_roi_detect_typed / det_b200.FastRCNNOutputs implement.

The reference never wrote the ROI predictor (SURVEY.md section 0), so this is the repository's own specification after
detectron2's fast_rcnn_inference_single_image -- "parity unpinned by reference".  It builds on the CPU oracle of
``oracle/ref_torch.py`` (greedy NMS in C, the reference's batched_nms branch rule, stable descending order).
"""
from __future__ import annotations

from typing import Sequence, Tuple

import torch

from oracle.ref_torch import DEFAULT_SCALE_CLAMP, batched_nms, nms, stable_desc_order


def softmax_rows_sequential(logits: torch.Tensor) -> torch.Tensor:
    """Row softmax in a fixed operation order: m = max (NaN-propagating), e = exp(x - m), s = e[:, 0] + e[:, 1] + ...
    summed left to right, p = e / s.  det_roi_detect sums in the same order, so its probabilities are bit-comparable
    (torch.softmax's reduction order is unspecified).  Every step is elementwise or a column loop, so the result does
    not depend on the device the tensors live on."""
    x = logits.float()
    m = x.max(dim=1, keepdim=True).values if x.shape[0] else x[:, :1]
    e = torch.exp(x - m)
    s = e[:, 0]
    for c in range(1, e.shape[1]):
        s = s + e[:, c]
    return e / s[:, None]


def _batched_nms_mode(boxes: torch.Tensor, scores: torch.Tensor, idxs: torch.Tensor, iou_threshold: float,
                      mode: int) -> torch.Tensor:
    """batched_nms with det_nms_batched's `mode`: 0 the reference's branch rule (batched_nms above), 1 always
    per category, 2 always torchvision's coordinate-offset trick."""
    if mode == 0 or boxes.numel() == 0:
        return batched_nms(boxes, scores, idxs, iou_threshold)
    boxes = boxes.float()
    if mode == 2:
        span = boxes.max() + torch.tensor(1).to(boxes)
        return nms(boxes + (idxs.to(boxes) * span)[:, None], scores, iou_threshold)
    hit = torch.zeros_like(scores, dtype=torch.bool)
    for c in torch.unique(idxs):
        members = torch.nonzero(idxs == c, as_tuple=True)[0]
        hit[members[nms(boxes[members], scores[members], iou_threshold)]] = True
    kept = torch.nonzero(hit, as_tuple=True)[0]
    return kept[stable_desc_order(scores[kept])]


def fast_rcnn_decode_single_image(logits: torch.Tensor, deltas: torch.Tensor, proposals: torch.Tensor,
                                  image_hw: Tuple[int, int], weights: Sequence[float] = (10.0, 10.0, 5.0, 5.0),
                                  scale_clamp: float = DEFAULT_SCALE_CLAMP):
    """Steps 1-4 of fast_rcnn_inference_single_image for one image of P proposals and K classes: logits (P, K+1),
    deltas (P, K*4) or (P, 4) (class-agnostic), proposals (P, 4).  Returns (probs (P, K+1), boxes (P, K, 4) clipped,
    valid (P,) bool).  Elementwise only: on a CUDA tensor every step is one IEEE fp32 torch kernel, the kernel's
    arithmetic (exp included), so the values can be compared bit for bit."""
    P, K = logits.shape[0], logits.shape[1] - 1
    probs = softmax_rows_sequential(logits)
    # apply_deltas above, with the weights as tensors on the same device: torch turns a CUDA tensor divided by a Python
    # scalar into a multiplication by its reciprocal, which is not the IEEE quotient
    d = deltas.float().reshape(P, deltas.shape[1] // 4, 4)
    bx = proposals.float()
    wt = torch.tensor(list(weights), dtype=torch.float32, device=d.device)
    w = (bx[:, 2] - bx[:, 0])[:, None]
    h = (bx[:, 3] - bx[:, 1])[:, None]
    cx = bx[:, 0:1] + 0.5 * w
    cy = bx[:, 1:2] + 0.5 * h
    dx, dy = d[..., 0] / wt[0], d[..., 1] / wt[1]
    dw = torch.clamp(d[..., 2] / wt[2], max=scale_clamp)
    dh = torch.clamp(d[..., 3] / wt[3], max=scale_clamp)
    pcx, pcy = dx * w + cx, dy * h + cy
    pw, ph = torch.exp(dw) * w, torch.exp(dh) * h
    boxes = torch.stack((pcx - 0.5 * pw, pcy - 0.5 * ph, pcx + 0.5 * pw, pcy + 0.5 * ph), dim=-1)
    valid = torch.isfinite(boxes).flatten(1).all(1) & torch.isfinite(probs).all(1)
    h, w = image_hw
    lim = torch.tensor([w, h, w, h], dtype=torch.float32, device=boxes.device)
    # Boxes.clip (x to [0, w], y to [0, h]) as comparisons: the same result on every device, signed zeros included
    boxes = torch.where(boxes < 0, torch.zeros((), dtype=torch.float32, device=boxes.device), boxes)
    boxes = torch.where(boxes > lim, lim, boxes)
    return probs, boxes.expand(P, K, 4), valid


def fast_rcnn_select_single_image(probs: torch.Tensor, boxes: torch.Tensor, valid: torch.Tensor, score_thresh: float,
                                  nms_thresh: float, topk: int, mode: int = 0):
    """Steps 5-7 on the output of fast_rcnn_decode_single_image (CPU tensors): candidates (i, c), c < K, of valid rows
    with probs[i, c] > score_thresh in row-major order (torch.nonzero, which decides ties), keep =
    batched_nms(box, score, c, nms_thresh)[:topk] (all when topk < 0).  Returns (flat ids i*K + c, boxes, scores,
    classes) by descending score, ties by lower flat id."""
    K = probs.shape[1] - 1
    fg = probs[:, :K]
    pi, ci = torch.nonzero((fg > score_thresh) & valid[:, None], as_tuple=True)
    cb, cs = boxes[pi, ci], fg[pi, ci]
    keep = _batched_nms_mode(cb, cs, ci, nms_thresh, mode)
    if topk >= 0:
        keep = keep[:topk]
    return (pi * K + ci)[keep], cb[keep], cs[keep], ci[keep]


def fast_rcnn_inference_single_image(logits: torch.Tensor, deltas: torch.Tensor, proposals: torch.Tensor,
                                     image_hw: Tuple[int, int], weights: Sequence[float] = (10.0, 10.0, 5.0, 5.0),
                                     scale_clamp: float = DEFAULT_SCALE_CLAMP, score_thresh: float = 0.05,
                                     nms_thresh: float = 0.5, topk: int = 100, mode: int = 0):
    """detectron2's fast_rcnn_inference_single_image on one image, in its order:
      1. probs = softmax(logits) (softmax_rows_sequential: the row sum in column order);
      2. boxes = apply_deltas(deltas, proposals), k = K (or 1 for class-agnostic (P, 4) deltas);
      3. a row is valid iff all its boxes and all its K+1 probabilities are finite; invalid rows are dropped;
      4. every box clipped to (h, w) as Boxes.clip;
      5. candidates (i, c), c < K (background column dropped), probs[i, c] > score_thresh, row-major order;
      6. keep = batched_nms(box, score, c, nms_thresh) (`mode` as in det_nms_batched), then [:topk] when topk >= 0;
      7. (flat id i*K + c, box, score, class) by descending score, ties by lower flat id.
    Deviation from detectron2: i is the proposal's index among the image's ORIGINAL rows; detectron2 returns indices
    into the rows left after step 3, which differ whenever a row is invalid.
    Steps 1-4 run on the tensors' device (see fast_rcnn_decode_single_image), 5-7 on the CPU."""
    probs, boxes, valid = fast_rcnn_decode_single_image(logits, deltas, proposals, image_hw, weights, scale_clamp)
    return fast_rcnn_select_single_image(probs.cpu(), boxes.cpu(), valid.cpu(), score_thresh, nms_thresh, topk, mode)
