"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the post-backbone detection hot path.

A from-scratch CPU restatement (torch CPU tensors + the C greedy-NMS in ``nms_ref.c``)
of the reference's algorithm for every function on the hot path.  It exists to *check*
the CUDA path: only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import it.  The product package
(``det_b200``) never imports anything from ``oracle/``.

Pinning: the reference ships no tests / golden vectors (SURVEY.md section 4), so this
restatement is pinned against the *unmodified reference functions executed in the build
container* (``oracle/ref_loader.py``): ``tests/test_oracle_vs_reference.py`` runs them
side by side when ``/root/reference`` is present, and ``tests/golden/*.npz`` (made by
``tests/golden/make_golden.py`` from the reference) pin it everywhere else.

Third-party arithmetic on the path that is NOT under ``/root/reference``:
  * torchvision.ops.nms / batched_nms (reference call sites ``python/src/utils.py:110,115``;
    no version pinned by the reference; 0.26.0 installed).  Greedy NMS is restated in C
    (``oracle/nms_ref.c``) and in :func:`batched_nms` below; it is pinned against the
    installed ``torch.ops.torchvision.nms`` CPU kernel by ``tests/test_oracle_nms.py``.
  * fvcore.nn.smooth_l1_loss / giou_loss (``box_regression.py:4``; absent, unpinned):
    restated from fvcore's published definitions.  The default config is beta=0 => L1.

Deliberate, documented deviation: the reference uses *unstable* descending sorts
(``python/src/models/utils.py:56`` ``logits_i.sort(descending=True)``; torchvision's
``_batched_nms_vanilla`` final sort; ``python/src/utils.py:118`` ``argsort``) whose order
among exactly-tied scores is an artefact of introsort on CPU.  The oracle (and the CUDA
path) define ties as "lower index first" (stable).  With distinct scores both agree
bit-for-bit.

The YOLO-grid functions at the bottom (``yolo_*``) have NO reference implementation
(SURVEY.md section 8 row a15): they are this repository's own specification --
"parity unpinned by reference".
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build_c_oracle(force: bool = False) -> str:
    """Compile oracle/nms_ref.c -> oracle/libnms_ref.so (gcc, -O2, no fast-math, no FMA contraction)."""
    src = os.path.join(_HERE, "nms_ref.c")
    out = os.path.join(_HERE, "libnms_ref.so")
    if force or not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                               "-o", out, src, "-lm"])
    return out


def _lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build_c_oracle())
        _LIB.oracle_nms_f32.restype = ctypes.c_int64
        _LIB.oracle_nms_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                        ctypes.c_double, ctypes.c_void_p]
    return _LIB


# --------------------------------------------------------------------------------------
# structures/boxes.py
# --------------------------------------------------------------------------------------
def box_area(b: torch.Tensor) -> torch.Tensor:
    """(x2-x1)*(y2-y1) in fp32 -- reference Boxes.area, python/src/structures/boxes.py:43-51."""
    return (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])


def pairwise_intersection(b1: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """[N,M] intersection areas -- reference python/src/structures/boxes.py:173-190.
    Same fp32 operation order: (min(hi) - max(lo)) clamped at 0, then w*h."""
    iw = (torch.minimum(b1[:, None, 2], b2[None, :, 2]) - torch.maximum(b1[:, None, 0], b2[None, :, 0])).clamp_(min=0)
    ih = (torch.minimum(b1[:, None, 3], b2[None, :, 3]) - torch.maximum(b1[:, None, 1], b2[None, :, 1])).clamp_(min=0)
    return iw * ih


def pairwise_iou(b1: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """[N,M] IoU; exactly 0 where inter<=0 -- reference python/src/structures/boxes.py:193-214."""
    a1, a2 = box_area(b1), box_area(b2)
    inter = pairwise_intersection(b1, b2)
    return torch.where(inter > 0, inter / (a1[:, None] + a2[None, :] - inter), torch.zeros((), dtype=inter.dtype))


def pairwise_ioa(b1: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """[N,M] intersection over area(b2) -- reference python/src/structures/boxes.py:217-232."""
    inter = pairwise_intersection(b1, b2)
    return torch.where(inter > 0, inter / box_area(b2)[None, :], torch.zeros((), dtype=inter.dtype))


def matched_boxlist_iou(b1: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """[N] diagonal IoU, no empty-box guard (0/0 -> NaN) -- reference boxes.py:235-258."""
    assert b1.shape[0] == b2.shape[0]
    iw = (torch.minimum(b1[:, 2], b2[:, 2]) - torch.maximum(b1[:, 0], b2[:, 0])).clamp(min=0)
    ih = (torch.minimum(b1[:, 3], b2[:, 3]) - torch.maximum(b1[:, 1], b2[:, 1])).clamp(min=0)
    inter = iw * ih
    return inter / (box_area(b1) + box_area(b2) - inter)


def clip_boxes_(b: torch.Tensor, size_hw: Tuple[int, int]) -> None:
    """In-place clamp x to [0,w], y to [0,h]; asserts finite -- reference boxes.py:53-65."""
    assert torch.isfinite(b).all(), "Box tensor contains infinite or NaN!"
    h, w = size_hw
    b[:, 0::2].clamp_(min=0, max=w)
    b[:, 1::2].clamp_(min=0, max=h)


def nonempty(b: torch.Tensor, threshold: float = 0.0) -> torch.Tensor:
    """(w > thr) & (h > thr) -- reference boxes.py:67-80."""
    return ((b[:, 2] - b[:, 0]) > threshold) & ((b[:, 3] - b[:, 1]) > threshold)


# --------------------------------------------------------------------------------------
# models/components/box_regression.py
# --------------------------------------------------------------------------------------
DEFAULT_SCALE_CLAMP = math.log(1000.0 / 16)  # reference python/src/config/rpn.py:10


def apply_deltas(deltas: torch.Tensor, boxes: torch.Tensor,
                 weights: Sequence[float] = (1.0, 1.0, 1.0, 1.0),
                 scale_clamp: float = DEFAULT_SCALE_CLAMP) -> torch.Tensor:
    """(M,k*4),(M,4)->(M,k*4) -- reference Box2BoxTransform.apply_deltas, box_regression.py:75-115."""
    d = deltas.float().reshape(deltas.shape[0], -1, 4)
    bx = boxes.to(torch.float32)
    w = (bx[:, 2] - bx[:, 0])[:, None]
    h = (bx[:, 3] - bx[:, 1])[:, None]
    cx = bx[:, 0:1] + 0.5 * w
    cy = bx[:, 1:2] + 0.5 * h
    wx, wy, ww, wh = weights
    dx, dy = d[..., 0] / wx, d[..., 1] / wy
    dw = torch.clamp(d[..., 2] / ww, max=scale_clamp)
    dh = torch.clamp(d[..., 3] / wh, max=scale_clamp)
    pcx, pcy = dx * w + cx, dy * h + cy
    pw, ph = torch.exp(dw) * w, torch.exp(dh) * h
    out = torch.stack((pcx - 0.5 * pw, pcy - 0.5 * ph, pcx + 0.5 * pw, pcy + 0.5 * ph), dim=-1)
    return out.reshape(deltas.shape)


def get_deltas(src: torch.Tensor, tgt: torch.Tensor,
               weights: Sequence[float] = (1.0, 1.0, 1.0, 1.0)) -> torch.Tensor:
    """(M,4),(M,4)->(M,4) regression targets -- reference Box2BoxTransform.get_deltas, box_regression.py:33-73."""
    sw, sh = src[:, 2] - src[:, 0], src[:, 3] - src[:, 1]
    scx, scy = src[:, 0] + 0.5 * sw, src[:, 1] + 0.5 * sh
    tw, th = tgt[:, 2] - tgt[:, 0], tgt[:, 3] - tgt[:, 1]
    tcx, tcy = tgt[:, 0] + 0.5 * tw, tgt[:, 1] + 0.5 * th
    wx, wy, ww, wh = weights
    out = torch.stack((wx * (tcx - scx) / sw, wy * (tcy - scy) / sh,
                       ww * torch.log(tw / sw), wh * torch.log(th / sh)), dim=1)
    assert bool((sw > 0).all()), "Input boxes to Box2BoxTransform are not valid!"
    return out


def smooth_l1_sum(x: torch.Tensor, y: torch.Tensor, beta: float) -> torch.Tensor:
    """fvcore.nn.smooth_l1_loss(reduction='sum') restated (third-party, unpinned; see module docstring)."""
    n = torch.abs(x - y)
    if beta < 1e-5:
        return n.sum()
    return torch.where(n < beta, 0.5 * n ** 2 / beta, n - 0.5 * beta).sum()


def giou_sum(p: torch.Tensor, g: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """fvcore.nn.giou_loss(reduction='sum') restated (third-party, unpinned)."""
    x1, y1, x2, y2 = p.unbind(-1)
    X1, Y1, X2, Y2 = g.unbind(-1)
    ix1, iy1 = torch.max(x1, X1), torch.max(y1, Y1)
    ix2, iy2 = torch.min(x2, X2), torch.min(y2, Y2)
    overlap = (iy2 > iy1) & (ix2 > ix1)
    inter = torch.where(overlap, (ix2 - ix1) * (iy2 - iy1), torch.zeros_like(x1))
    union = (x2 - x1) * (y2 - y1) + (X2 - X1) * (Y2 - Y1) - inter
    iou = inter / (union + eps)
    hull = (torch.max(x2, X2) - torch.min(x1, X1)) * (torch.max(y2, Y2) - torch.min(y1, Y1))
    return (1 - (iou - (hull - union) / (hull + eps))).sum()


def dense_box_regression_loss(anchors: torch.Tensor, pred_deltas: torch.Tensor,
                              gt_boxes: torch.Tensor, fg_mask: torch.Tensor,
                              weights=(1.0, 1.0, 1.0, 1.0), scale_clamp=DEFAULT_SCALE_CLAMP,
                              box_reg_loss_type: str = "smooth_l1", smooth_l1_beta: float = 0.0) -> torch.Tensor:
    """anchors (R,4), pred_deltas (N,R,4), gt_boxes (N,R,4), fg_mask (N,R) bool ->
    summed localisation loss -- reference _dense_box_regression_loss, box_regression.py:128-168."""
    if box_reg_loss_type == "smooth_l1":
        tgt = torch.stack([get_deltas(anchors, g, weights) for g in gt_boxes])
        return smooth_l1_sum(pred_deltas[fg_mask], tgt[fg_mask], smooth_l1_beta)
    if box_reg_loss_type == "giou":
        pb = torch.stack([apply_deltas(d, anchors, weights, scale_clamp) for d in pred_deltas])
        return giou_sum(pb[fg_mask], gt_boxes[fg_mask])
    raise ValueError(f"Invalid dense box regression loss type '{box_reg_loss_type}'")


# --------------------------------------------------------------------------------------
# models/modules/anchor_generators.py
# --------------------------------------------------------------------------------------
def cell_anchors(sizes: Sequence[float], aspect_ratios: Sequence[float]) -> torch.Tensor:
    """(len(sizes)*len(ratios),4) XYXY anchors centred on 0; python double math then .float()
    -- reference generate_cell_anchors, anchor_generators.py:181-210 (+ .float() at :132)."""
    rows = []
    for s in sizes:
        for r in aspect_ratios:
            w = math.sqrt((s ** 2.0) / r)
            h = r * w
            rows.append([-w / 2.0, -h / 2.0, w / 2.0, h / 2.0])
    return torch.tensor(rows).float()


def grid_anchors(grid_sizes: Sequence[Tuple[int, int]], strides: Sequence[int],
                 cells: Sequence[torch.Tensor], offset: float = 0.0) -> List[torch.Tensor]:
    """Per level (Hi*Wi*A,4), order (h,w,a) -- reference _grid_anchors/_create_grid_offsets,
    anchor_generators.py:31-56,158-179."""
    out = []
    for (gh, gw), s, base in zip(grid_sizes, strides, cells):
        xs = torch.arange(offset * s, gw * s, step=s, dtype=torch.float32)
        ys = torch.arange(offset * s, gh * s, step=s, dtype=torch.float32)
        sy = ys[:, None].expand(len(ys), len(xs)).reshape(-1)
        sx = xs[None, :].expand(len(ys), len(xs)).reshape(-1)
        shifts = torch.stack((sx, sy, sx, sy), dim=1)
        out.append((shifts[:, None, :] + base[None, :, :]).reshape(-1, 4))
    return out


# --------------------------------------------------------------------------------------
# models/components/matcher.py
# --------------------------------------------------------------------------------------
def match(quality: torch.Tensor, thresholds: Sequence[float], labels: Sequence[int],
          allow_low_quality_matches: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """(G,R) quality -> (int64[R] matched gt, int8[R] label) -- reference Matcher.__call__ and
    set_low_quality_matches_, matcher.py:53-120.  Bucket rule low <= v < high; ties in the
    column max go to the lowest gt index; low-quality promotion marks every column equal to
    its row's max (including the all-zero-row quirk)."""
    assert quality.dim() == 2
    bounds = [-float("inf")] + list(thresholds) + [float("inf")]
    assert len(labels) == len(bounds) - 1
    R = quality.shape[1]
    if quality.numel() == 0:
        return (torch.zeros(R, dtype=torch.int64), torch.full((R,), labels[0], dtype=torch.int8))
    assert bool(torch.all(quality >= 0))
    vals, idx = quality.max(dim=0)
    lab = torch.ones(R, dtype=torch.int8)
    for l, lo, hi in zip(labels, bounds[:-1], bounds[1:]):
        lab[(vals >= lo) & (vals < hi)] = l
    if allow_low_quality_matches:
        best = quality.max(dim=1).values
        lab[(quality == best[:, None]).any(dim=0)] = 1
    return idx, lab


# --------------------------------------------------------------------------------------
# utils.py : subsample_labels, batched_nms (+ torchvision nms restated)
# --------------------------------------------------------------------------------------
def subsample_counts(num_pos_avail: int, num_neg_avail: int, num_samples: int,
                     positive_fraction: float) -> Tuple[int, int]:
    """min(#pos, int(S*f)), min(#neg, S - num_pos) -- reference python/src/utils.py:64-69."""
    num_pos = min(num_pos_avail, int(num_samples * positive_fraction))
    num_neg = min(num_neg_avail, num_samples - num_pos)
    return num_pos, num_neg


def subsample_labels(labels: torch.Tensor, num_samples: int, positive_fraction: float,
                     bg_label: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Random fg/bg index sample with torch.randperm (global RNG) -- reference python/src/utils.py:34-76."""
    pos = torch.nonzero((labels != -1) & (labels != bg_label), as_tuple=True)[0]
    neg = torch.nonzero(labels == bg_label, as_tuple=True)[0]
    num_pos, num_neg = subsample_counts(pos.numel(), neg.numel(), num_samples, positive_fraction)
    p1 = torch.randperm(pos.numel())[:num_pos]
    p2 = torch.randperm(neg.numel())[:num_neg]
    return pos[p1], neg[p2]


def rpn_subsample_(label: torch.Tensor, batch_size_per_image: int, positive_fraction: float) -> torch.Tensor:
    """fill(-1) then scatter 1 / 0 at the sampled indices -- reference rpn.py:108-130."""
    pos, neg = subsample_labels(label, batch_size_per_image, positive_fraction, 0)
    label.fill_(-1)
    label[pos] = 1
    label[neg] = 0
    return label


def nms(boxes: torch.Tensor, scores: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    """Greedy NMS, C restatement of torchvision's CPU kernel (stable descending score order,
    fp32 IoU = inter/(a_i + a_j - inter), suppressed iff IoU > threshold compared in double)."""
    b = boxes.detach().to(torch.float32).contiguous()
    s = scores.detach().to(torch.float32).contiguous()
    n = b.shape[0]
    keep = torch.empty(n, dtype=torch.int64)
    if n == 0:
        return keep
    k = _lib().oracle_nms_f32(b.data_ptr(), s.data_ptr(), n, float(iou_threshold), keep.data_ptr())
    return keep[:k].clone()


def stable_desc_order(scores: torch.Tensor) -> torch.Tensor:
    return torch.sort(scores, descending=True, stable=True)[1]


def batched_nms(boxes: torch.Tensor, scores: torch.Tensor, idxs: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    """Category-partitioned NMS, kept indices by descending score -- reference python/src/utils.py:96-119
    on top of torchvision.ops.boxes.batched_nms (CPU rule: numel<=4000 -> coordinate-offset trick in fp32,
    else per-category; reference's own per-id loop at len>=40000 gives the same kept set)."""
    assert boxes.shape[-1] == 4
    boxes = boxes.float()
    if boxes.numel() == 0:
        return torch.empty((0,), dtype=torch.int64)
    if boxes.shape[0] < 40000 and boxes.numel() <= 4000:
        span = boxes.max() + torch.tensor(1).to(boxes)
        shifted = boxes + (idxs.to(boxes) * span)[:, None]
        return nms(shifted, scores, iou_threshold)
    hit = torch.zeros_like(scores, dtype=torch.bool)
    for c in torch.unique(idxs):
        members = torch.nonzero(idxs == c, as_tuple=True)[0]
        hit[members[nms(boxes[members], scores[members], iou_threshold)]] = True
    kept = torch.nonzero(hit, as_tuple=True)[0]
    return kept[stable_desc_order(scores[kept])]


# --------------------------------------------------------------------------------------
# models/utils.py : find_top_rpn_proposals
# --------------------------------------------------------------------------------------
def find_top_rpn_proposals(proposals: List[torch.Tensor], logits: List[torch.Tensor],
                           image_sizes: List[Tuple[int, int]], nms_thresh: float, pre_nms_topk: int,
                           post_nms_topk: int, min_box_size: float, training: bool
                           ) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """Per level top-k -> per image {finite filter, clip, small-box filter, per-level NMS, top-k}.
    Returns [(boxes[K,4], logits[K])] per image -- reference models/utils.py:9-109."""
    n_img = len(image_sizes)
    sel_boxes, sel_scores, sel_level = [], [], []
    for lvl, (p, s) in enumerate(zip(proposals, logits)):
        k = min(s.shape[1], pre_nms_topk)
        order = torch.sort(s, dim=1, descending=True, stable=True)[1][:, :k]
        sel_scores.append(torch.gather(s, 1, order))
        sel_boxes.append(torch.gather(p, 1, order[:, :, None].expand(-1, -1, 4)))
        sel_level.append(torch.full((k,), lvl, dtype=torch.int64))
    all_scores, all_boxes, all_level = torch.cat(sel_scores, 1), torch.cat(sel_boxes, 1), torch.cat(sel_level, 0)
    out = []
    for i in range(n_img):
        b, s, l = all_boxes[i].clone(), all_scores[i], all_level
        ok = torch.isfinite(b).all(dim=1) & torch.isfinite(s)
        if not bool(ok.all()):
            if training:
                raise FloatingPointError("Predicted boxes or scores contain Inf/NaN. Training has diverged.")
            b, s, l = b[ok], s[ok], l[ok]
        clip_boxes_(b, image_sizes[i])
        big = nonempty(b, min_box_size)
        b, s, l = b[big], s[big], l[big]
        keep = batched_nms(b, s, l, nms_thresh)[:post_nms_topk]
        out.append((b[keep], s[keep]))
    return out


# --------------------------------------------------------------------------------------
# models/rpn.py : decode, label_and_sample_anchors, losses
# --------------------------------------------------------------------------------------
def head_to_hwa(objectness: torch.Tensor, deltas: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(N,A,H,W)->(N,HWA); (N,A*4,H,W)->(N,HWA,4): the layout change the reference *intends* at
    rpn.py:270-284 (commented detectron2 form at :272,:278-280; the einops line at :282 is broken)."""
    n, a, h, w = objectness.shape
    obj = objectness.permute(0, 2, 3, 1).reshape(n, -1)
    dl = deltas.view(n, a, 4, h, w).permute(0, 3, 4, 1, 2).reshape(n, -1, 4)
    return obj, dl


def decode_proposals(anchors: List[torch.Tensor], pred_deltas: List[torch.Tensor],
                     weights=(1.0, 1.0, 1.0, 1.0), scale_clamp=DEFAULT_SCALE_CLAMP) -> List[torch.Tensor]:
    """Per level (N,HiWiA,4) proposals -- reference _decode_proposals, rpn.py:330-348."""
    out = []
    for a, d in zip(anchors, pred_deltas):
        n = d.shape[0]
        rep = a[None].expand(n, -1, -1).reshape(-1, 4)
        out.append(apply_deltas(d.reshape(-1, 4), rep, weights, scale_clamp).view(n, -1, 4))
    return out


def label_anchors(anchors: torch.Tensor, gt_boxes: List[torch.Tensor],
                  thresholds=(0.3, 0.7), labels=(0, -1, 1), allow_low_quality=True
                  ) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
    """The deterministic half of reference label_and_sample_anchors (rpn.py:132-185): per image
    IoU -> Matcher, *before* the random subsample.  Returns (labels int8[R], matched idx int64[R])."""
    labs, idxs = [], []
    for g in gt_boxes:
        q = pairwise_iou(g, anchors)
        i, l = match(q, list(thresholds), list(labels), allow_low_quality)
        labs.append(l)
        idxs.append(i)
    return labs, idxs


def label_and_sample_anchors(anchors: torch.Tensor, gt_boxes: List[torch.Tensor],
                             batch_size_per_image=256, positive_fraction=0.5,
                             thresholds=(0.3, 0.7), labels=(0, -1, 1), allow_low_quality=True):
    """Full reference label_and_sample_anchors (rpn.py:132-185) incl. torch.randperm subsample."""
    labs, idxs = label_anchors(anchors, gt_boxes, thresholds, labels, allow_low_quality)
    out_l, out_b = [], []
    for g, l, i in zip(gt_boxes, labs, idxs):
        l = rpn_subsample_(l, batch_size_per_image, positive_fraction)
        out_b.append(torch.zeros_like(anchors) if len(g) == 0 else g[i])
        out_l.append(l)
    return out_l, out_b


def rpn_losses(anchors: torch.Tensor, pred_logits: torch.Tensor, gt_labels: torch.Tensor,
               pred_deltas: torch.Tensor, gt_boxes: torch.Tensor, batch_size_per_image=256,
               weights=(1.0, 1.0, 1.0, 1.0), scale_clamp=DEFAULT_SCALE_CLAMP,
               box_reg_loss_type="smooth_l1", smooth_l1_beta=0.0, loss_weight=(1.0, 1.0)):
    """anchors (R,4), logits (N,R), labels (N,R) int8, deltas (N,R,4), matched gt (N,R,4) ->
    {"cls_loss","loc_loss"} -- reference losses, rpn.py:187-244."""
    n = gt_labels.shape[0]
    pos = gt_labels == 1
    loc = dense_box_regression_loss(anchors, pred_deltas, gt_boxes, pos, weights, scale_clamp,
                                    box_reg_loss_type, smooth_l1_beta)
    valid = gt_labels >= 0
    # targets in the logits' dtype: with fp32 targets, BCE-with-logits computes a float64 run in fp32
    obj = F.binary_cross_entropy_with_logits(pred_logits[valid], gt_labels[valid].to(pred_logits.dtype), reduction="sum")
    norm = batch_size_per_image * n
    return {"cls_loss": obj / norm * loss_weight[0], "loc_loss": loc / norm * loss_weight[1],
            "num_pos": int(pos.sum()), "num_neg": int((gt_labels == 0).sum())}


# --------------------------------------------------------------------------------------
# models/roi.py : label_and_sample_proposals ("next" tier, SURVEY.md section 8f rank 1)
# --------------------------------------------------------------------------------------
GT_LOGIT = math.log((1.0 - 1e-10) / (1 - (1.0 - 1e-10)))  # reference models/utils.py:147


def roi_label_proposals(proposal_boxes: torch.Tensor, gt_boxes: torch.Tensor, gt_classes: torch.Tensor,
                        num_classes: int, thresholds=(0.5,), labels=(0, 1), allow_low_quality=False,
                        append_gt=True):
    """Deterministic half of reference ROIHeads.label_and_sample_proposals (roi.py:107-193):
    optional GT append -> IoU -> Matcher -> class labels (bg=num_classes, ignore=-1; roi.py:84-95)."""
    if append_gt:
        proposal_boxes = torch.cat([proposal_boxes, gt_boxes], dim=0)
    q = pairwise_iou(gt_boxes, proposal_boxes)
    midx, mlab = match(q, list(thresholds), list(labels), allow_low_quality)
    if gt_classes.numel() > 0:
        cls = gt_classes[midx].clone()
        cls[mlab == 0] = num_classes
        cls[mlab == -1] = -1
    else:
        cls = torch.zeros_like(midx) + num_classes
    return proposal_boxes, midx, mlab, cls


# --------------------------------------------------------------------------------------
# YOLO-grid superset (NO reference implementation -- this repository's own specification)
# --------------------------------------------------------------------------------------
def yolo_decode(head: torch.Tensor, num_boxes: int, num_classes: int, image_hw: Tuple[int, int],
                priors: torch.Tensor, scale_clamp: float = DEFAULT_SCALE_CLAMP, clip: bool = True):
    """head (N,S,S,B*5+C) channels-last: per cell B x (tx,ty,tw,th,tconf) then C class logits.
        cx=(sigmoid(tx)+col)*stride_x  cy=(sigmoid(ty)+row)*stride_y
        w =exp(min(tw,clamp))*prior_w[b]   h=exp(min(th,clamp))*prior_h[b]
        box=(cx-0.5w, cy-0.5h, cx+0.5w, cy+0.5h), clamped to [0,W]x[0,H] when clip;   conf=sigmoid(tconf)
        score[b,c]=conf[b]*sigmoid(class_logit[c])
    Returns boxes (N,S*S*B,4), conf (N,S*S*B), scores (N,S*S*B,C); predictor order (row,col,b)."""
    n, s1, s2, ch = head.shape
    B, C = num_boxes, num_classes
    assert ch == B * 5 + C
    H, W = image_hw
    sx, sy = W / s2, H / s1
    t = head[..., :B * 5].reshape(n, s1, s2, B, 5).float()
    col = torch.arange(s2, dtype=torch.float32).view(1, 1, s2, 1)
    row = torch.arange(s1, dtype=torch.float32).view(1, s1, 1, 1)
    cx = (torch.sigmoid(t[..., 0]) + col) * sx
    cy = (torch.sigmoid(t[..., 1]) + row) * sy
    w = torch.exp(torch.clamp(t[..., 2], max=scale_clamp)) * priors[:, 0].view(1, 1, 1, B)
    h = torch.exp(torch.clamp(t[..., 3], max=scale_clamp)) * priors[:, 1].view(1, 1, 1, B)
    boxes = torch.stack((cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h), dim=-1).reshape(n, -1, 4)
    if clip:
        boxes[..., 0::2].clamp_(min=0, max=W)
        boxes[..., 1::2].clamp_(min=0, max=H)
    conf = torch.sigmoid(t[..., 4])
    pcls = torch.sigmoid(head[..., B * 5:].float())
    scores = (conf[..., None] * pcls[:, :, :, None, :]).reshape(n, -1, C)
    return boxes, conf.reshape(n, -1), scores


def yolo_select_nms(boxes: torch.Tensor, scores: torch.Tensor, score_thresh: float, iou_thresh: float,
                    max_det: Optional[int] = None):
    """One image: candidates = (predictor,class) pairs with score > thresh in row-major order,
    then the reference's batched_nms with category = class.  Returns (flat ids = pred*C+cls, boxes,
    scores, classes) of kept detections, by descending score."""
    C = scores.shape[1]
    pi, ci = torch.nonzero(scores > score_thresh, as_tuple=True)
    cb, cs = boxes[pi], scores[pi, ci]
    keep = batched_nms(cb, cs, ci, iou_thresh)
    if max_det is not None:
        keep = keep[:max_det]
    return (pi[keep] * C + ci[keep]), cb[keep], cs[keep], ci[keep]


def dense_decode(head: torch.Tensor, num_anchors: int, num_classes: int, stride: int, anchors_wh: torch.Tensor,
                 scale_clamp: float = DEFAULT_SCALE_CLAMP):
    """Dense anchor head of one level in the conv layout (N, A*(5+C), H, W) (own specification):
        cx=(sigmoid(tx)+col)*stride  cy=(sigmoid(ty)+row)*stride  w=exp(min(tw,clamp))*aw  h=exp(min(th,clamp))*ah
        class = argmax_c logit_c (first maximum), score = sigmoid(tobj) * sigmoid(max logit)
    Returns boxes (N,HWA,4), score (N,HWA), class (N,HWA) int64, order (h,w,a)."""
    n, _, H, W = head.shape
    A, C = num_anchors, num_classes
    t = head.view(n, A, 5 + C, H, W).float()
    col = torch.arange(W, dtype=torch.float32).view(1, 1, 1, W)
    row = torch.arange(H, dtype=torch.float32).view(1, 1, H, 1)
    cx = (torch.sigmoid(t[:, :, 0]) + col) * float(stride)
    cy = (torch.sigmoid(t[:, :, 1]) + row) * float(stride)
    w = torch.exp(torch.clamp(t[:, :, 2], max=scale_clamp)) * anchors_wh[:, 0].view(1, A, 1, 1)
    h = torch.exp(torch.clamp(t[:, :, 3], max=scale_clamp)) * anchors_wh[:, 1].view(1, A, 1, 1)
    boxes = torch.stack((cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h), dim=-1)  # N,A,H,W,4
    obj = torch.sigmoid(t[:, :, 4])
    if C > 0:
        cmax, cidx = t[:, :, 5:].max(dim=2)
        score = obj * torch.sigmoid(cmax)
    else:
        cidx = torch.zeros_like(obj, dtype=torch.int64)
        score = obj * 1.0
    boxes = boxes.permute(0, 2, 3, 1, 4).reshape(n, -1, 4)
    return boxes, score.permute(0, 2, 3, 1).reshape(n, -1), cidx.permute(0, 2, 3, 1).reshape(n, -1)


def dense_select_nms(boxes: torch.Tensor, scores: torch.Tensor, classes: torch.Tensor, score_thresh: float,
                     iou_thresh: float, max_det: Optional[int] = None):
    """Inference selection of ONE image of a dense anchor head (own specification; the NMS is the reference's
    batched_nms, python/src/utils.py:96-119): candidates = rows with score > score_thresh in row order,
    keep = batched_nms(...)[:max_det].  Returns (rows int64, boxes, scores, classes) by descending score."""
    cand = torch.nonzero(scores > score_thresh, as_tuple=True)[0]
    cb, cs, cc = boxes[cand], scores[cand], classes[cand]
    keep = batched_nms(cb, cs, cc, iou_thresh)
    if max_det is not None:
        keep = keep[:max_det]
    return cand[keep], cb[keep], cs[keep], cc[keep]


def yolo_grid_anchors(S: int, image_hw: Tuple[int, int], priors: torch.Tensor) -> torch.Tensor:
    """Prior boxes of the S*S*B predictors (cell-centred), order (row,col,b); used for IoU target assignment."""
    H, W = image_hw
    sx, sy = W / S, H / S
    cx = ((torch.arange(S, dtype=torch.float32) + 0.5) * sx).view(1, S, 1).expand(S, S, priors.shape[0])
    cy = ((torch.arange(S, dtype=torch.float32) + 0.5) * sy).view(S, 1, 1).expand(S, S, priors.shape[0])
    pw = priors[:, 0].view(1, 1, -1).expand(S, S, -1)
    ph = priors[:, 1].view(1, 1, -1).expand(S, S, -1)
    return torch.stack((cx - 0.5 * pw, cy - 0.5 * ph, cx + 0.5 * pw, cy + 0.5 * ph), dim=-1).reshape(-1, 4)


def yolo_loss(head: torch.Tensor, labels: torch.Tensor, matched: torch.Tensor, gt_boxes: List[torch.Tensor],
              gt_classes: List[torch.Tensor], num_boxes: int, num_classes: int, image_hw: Tuple[int, int],
              priors: torch.Tensor, lambda_coord: float = 5.0, lambda_noobj: float = 0.5,
              normalizer: Optional[float] = None):
    """YOLO-style fused loss (own spec).  labels (N,P) int8 in {-1,0,1}, matched (N,P) int64, P=S*S*B.
       positives: loc += (sig(tx)-x*)^2 + (sig(ty)-y*)^2 + (tw-log(gw/pw))^2 + (th-log(gh/ph))^2
                  cls += sum_c BCEWithLogits(class_logit_c, [c==gt_class])
       label>=0 : obj += (1 if pos else lambda_noobj) * BCEWithLogits(tconf, label)
       result = {loc*lambda_coord/norm, obj/norm, cls/norm}, norm defaults to N."""
    n, S, _, ch = head.shape
    B, C = num_boxes, num_classes
    H, W = image_hw
    sx, sy = W / S, H / S
    norm = float(n if normalizer is None else normalizer)
    t = head[..., :B * 5].reshape(n, S * S, B, 5).reshape(n, S * S * B, 5)
    cl = head[..., B * 5:].reshape(n, S * S, C)
    loc = head.new_zeros(())
    obj = head.new_zeros(())
    cls = head.new_zeros(())
    for i in range(n):
        lab = labels[i]
        valid = lab >= 0
        # weights and BCE targets in the head's dtype, so that a float64 run is float64 throughout
        wgt = torch.where(lab == 1, torch.ones((), dtype=head.dtype), torch.full((), lambda_noobj, dtype=head.dtype))
        obj = obj + (wgt[valid] * F.binary_cross_entropy_with_logits(
            t[i, valid, 4], lab[valid].to(head.dtype), reduction="none")).sum()
        p = torch.nonzero(lab == 1, as_tuple=True)[0]
        if p.numel() == 0:
            continue
        g = gt_boxes[i][matched[i, p]]
        gc = gt_classes[i][matched[i, p]]
        cell = p // B
        b = p % B
        rowi, coli = (cell // S).float(), (cell % S).float()
        gw, gh = g[:, 2] - g[:, 0], g[:, 3] - g[:, 1]
        xs = (g[:, 0] + 0.5 * gw) / sx - coli
        ys = (g[:, 1] + 0.5 * gh) / sy - rowi
        tw_t, th_t = torch.log(gw / priors[b, 0]), torch.log(gh / priors[b, 1])
        tp = t[i, p]
        loc = loc + ((torch.sigmoid(tp[:, 0]) - xs) ** 2 + (torch.sigmoid(tp[:, 1]) - ys) ** 2
                     + (tp[:, 2] - tw_t) ** 2 + (tp[:, 3] - th_t) ** 2).sum()
        onehot = F.one_hot(gc, C).to(head.dtype)
        cls = cls + F.binary_cross_entropy_with_logits(cl[i, cell], onehot, reduction="sum")
    return {"loc_loss": loc * lambda_coord / norm, "obj_loss": obj / norm, "cls_loss": cls / norm}
