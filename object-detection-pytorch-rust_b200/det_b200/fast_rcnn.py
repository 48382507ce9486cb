"""Second-stage (Fast R-CNN box predictor) inference -- what detectron2's ``FastRCNNOutputLayers.inference`` /
``fast_rcnn_inference`` do with the box head's ``class_logits (M, K+1)`` and ``proposal_deltas (M, K*4)``: softmax,
class-specific decode, clip, score threshold, per-class NMS and top-k, for the whole batch in two launches
(det_roi_detect_typed, csrc/roi_detect.cu) instead of a Python loop with a host sync per image.

Specification: tests/fast_rcnn_oracle.py fast_rcnn_inference_single_image (detectron2's fast_rcnn_inference_single_image).
One deviation: the kept proposal index of a detection counts the image's ORIGINAL rows; detectron2 counts the rows
left after dropping those with a non-finite box or score, which differs only when such a row exists.

Training: ``FastRCNNOutputs.losses`` is detectron2's ``FastRCNNOutputLayers.losses`` (softmax cross-entropy and
smooth-L1 / GIoU box regression on the gt class's deltas, plus ``_log_classification_stats``), forward and backward in
one kernel (det_fast_rcnn_loss_typed, csrc/fast_rcnn_loss.cu); specification tests/fast_rcnn_loss_oracle.py."""
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch

from . import _native as N
from .box_regression import Box2BoxTransform
from .nms import MODE_AUTO, detect_unfused, detect_workspace, detection_buffers
from .structures import Boxes, Instances

ROI_HEAD_WEIGHTS = (10.0, 10.0, 5.0, 5.0)  # detectron2's ROI_BOX_HEAD.BBOX_REG_WEIGHTS default


def _packed_offsets(lengths: Sequence[int], device) -> torch.Tensor:
    off = [0]
    for n in lengths:
        off.append(off[-1] + int(n))
    return torch.tensor(off, dtype=torch.int32).to(device)


def _sizes_tensor(image_shapes: Sequence[Tuple[int, int]], device) -> torch.Tensor:
    return torch.tensor([[int(h), int(w)] for h, w in image_shapes], dtype=torch.int32).reshape(-1, 2).to(device)


def _select_dense(rows, cols, code, proposals, offsets, sizes, n, p_max, K, agnostic, decoded, weights, scale_clamp,
                  score_thresh, nms_thresh, max_det, mode):
    """The exact route for any candidate count: det_roi_decode_dense_typed -> nms.detect_unfused on the (n, p_max * K)
    rows with classes = flat % K.  Library kernels only, no host sync.  max_det < 0: every kept detection
    (max_det = p_max * K)."""
    dev = rows.device
    R = p_max * K
    max_det = max(R, 1) if max_det < 0 else max_det
    scores = torch.empty((n, R), dtype=torch.float32, device=dev)
    boxes = torch.empty((n, R, 4), dtype=torch.float32, device=dev)
    if n and R:
        with torch.cuda.device(dev):
            N.call("det_roi_decode_dense_typed", N.ptr(rows), N.ptr(cols), code, N.ptr(proposals), N.ptr(offsets), n,
                   rows.shape[0], K, int(agnostic), N.ptr(sizes), *weights, scale_clamp, int(decoded), p_max,
                   N.ptr(scores), N.ptr(boxes), N.stream())
    classes = torch.arange(K, dtype=torch.int64, device=dev).repeat(n * p_max).view(n, R)
    return detect_unfused(boxes, scores, classes, score_thresh, nms_thresh, max_det, mode)


def _instances(out, image_shapes, K):
    """Per-image Instances (pred_boxes, scores, pred_classes) and kept proposal indices from the padded result."""
    counts = out["count"].tolist()
    results, kept = [], []
    for i, shape in enumerate(image_shapes):
        k = counts[i]
        inst = Instances(tuple(shape))
        inst.pred_boxes = Boxes(out["boxes"][i, :k])
        inst.scores = out["scores"][i, :k]
        inst.pred_classes = out["classes"][i, :k]
        results.append(inst)
        kept.append(out["idx"][i, :k] // K)
    return results, kept


class _FastRCNNLoss(torch.autograd.Function):
    """det_fast_rcnn_loss_typed behind autograd.  Forward: one launch that reduces the sums (no gradient stores).
    Backward: the same kernel with the upstream gradients read on the device, writing grad_logits / grad_deltas in the
    inputs' dtype.  Everything the backward launch reads goes through save_for_backward, so an in-place change of the
    labels or boxes between forward and backward trips autograd's version check."""

    @staticmethod
    def forward(ctx, owner, class_logits, deltas, proposal_boxes, gt_classes, gt_boxes):
        (lg, dl), code = N.heads_c([class_logits, deltas])
        sums = owner._run_loss(lg, dl, code, proposal_boxes, gt_classes, gt_boxes, None, None, None)
        ctx.owner, ctx.code = owner, code
        ctx.save_for_backward(lg, dl, proposal_boxes, gt_classes, gt_boxes)
        return sums

    @staticmethod
    def backward(ctx, grad_sums):
        lg, dl, props, gtc, gtb = ctx.saved_tensors
        up = grad_sums[:2].contiguous().float()
        gl, gd = torch.empty_like(lg), torch.empty_like(dl)
        ctx.owner._run_loss(lg, dl, ctx.code, props, gtc, gtb, up, gl, gd)
        return None, gl, gd, None, None, None


class FastRCNNOutputs:
    """detectron2's FastRCNNOutputLayers on the box head's outputs: inference, and the training losses.

    num_classes K foreground classes (the logits carry K+1 columns, background last); box2box_transform defaults to the
    ROI heads' weights (10, 10, 5, 5); topk_per_image < 0 keeps every detection.  cand_cap (<= 4096) bounds the
    per-image candidate list of the fused path; mode is det_nms_batched's NMS branch rule.  box_reg_loss_type
    ("smooth_l1" or "giou"), smooth_l1_beta and loss_weight (a float for both losses, or a dict keyed "loss_cls" /
    "loss_box_reg", 1.0 for a missing key) configure the losses as in detectron2."""

    def __init__(self, num_classes: int, box2box_transform: Optional[Box2BoxTransform] = None,
                 score_thresh: float = 0.05, nms_thresh: float = 0.5, topk_per_image: int = 100,
                 class_agnostic: bool = False, cand_cap: int = 4096, mode: int = MODE_AUTO, *,
                 box_reg_loss_type: str = "smooth_l1", smooth_l1_beta: float = 0.0,
                 loss_weight: Union[float, Dict[str, float]] = 1.0):
        self.num_classes = int(num_classes)
        self.box2box_transform = box2box_transform if box2box_transform is not None else Box2BoxTransform(ROI_HEAD_WEIGHTS)
        self.score_thresh, self.nms_thresh = float(score_thresh), float(nms_thresh)
        self.topk_per_image = int(topk_per_image)
        self.class_agnostic = bool(class_agnostic)
        self.cand_cap = int(cand_cap)
        self.mode = int(mode)
        if not 1 <= self.cand_cap <= 4096:
            raise ValueError("cand_cap must lie in [1, 4096]")
        self.box_reg_loss_type = box_reg_loss_type
        self.smooth_l1_beta = float(smooth_l1_beta)
        if not isinstance(loss_weight, dict):
            loss_weight = {"loss_cls": loss_weight, "loss_box_reg": loss_weight}
        self.loss_weight = loss_weight
        self.last_sums = None

    def _check_rows(self, class_logits, deltas, proposal_boxes):
        K = self.num_classes
        M = class_logits.shape[0]
        if class_logits.shape != (M, K + 1):
            raise ValueError(f"class_logits must be (M, {K + 1}), got {tuple(class_logits.shape)}")
        want = (M, 4) if self.class_agnostic else (M, 4 * K)
        if deltas.shape != want or proposal_boxes.shape != (M, 4):
            raise ValueError(f"deltas must be {want} and proposals (M, 4), got {tuple(deltas.shape)}, "
                             f"{tuple(proposal_boxes.shape)}")

    def _prepare(self, class_logits, deltas, proposal_boxes):
        self._check_rows(class_logits, deltas, proposal_boxes)
        (lg, dl), code = N.heads_c([class_logits, deltas])
        return lg, dl, code, N.f32c(proposal_boxes)

    def inference_batched(self, class_logits: torch.Tensor, deltas: torch.Tensor, proposal_boxes: torch.Tensor,
                          row_offsets: torch.Tensor, image_sizes: torch.Tensor, out: Optional[dict] = None,
                          workspace=None, check: bool = True) -> dict:
        """The whole batch, rows packed as the box head sees them: class_logits (M, K+1), deltas (M, K*4) or (M, 4)
        (fp32, or bf16 / fp16 read as they are: bit-identical to the call on .float()), proposal_boxes (M, 4),
        row_offsets (N+1) int32 (image b owns rows [row_offsets[b], row_offsets[b+1])), image_sizes (N, 2) int32 (h, w),
        all on the GPU.  Returns a dict of padded tensors: idx (N, D) int64 = i*K + c with i the proposal's row in its
        image, boxes (N, D, 4), scores (N, D), classes (N, D) int64, count (N) int32 -- entries past count undefined --
        and overflow (1) int32.  D = topk_per_image, or cand_cap when topk_per_image < 0.

        check=False: no host synchronisation; an image with more than cand_cap candidates has count -1 and overflow is
        set.  check=True (one 4-byte read-back): such a batch is redone on the exact unfused route (then, with
        topk_per_image < 0, D = the largest image's row count * K).  With workspace = a DenseDetectWorkspace(N, cand_cap)
        -- the same layout -- the call is exactly two launches and can be captured in a CUDA graph."""
        N.require_cuda(class_logits, deltas, proposal_boxes, row_offsets, image_sizes)
        dev = class_logits.device
        K = self.num_classes
        n = row_offsets.numel() - 1
        lg, dl, code, props = self._prepare(class_logits, deltas, proposal_boxes)
        offsets = row_offsets.detach().to(torch.int32).contiguous()
        sizes = image_sizes.detach().to(torch.int32).contiguous()
        max_det = self.topk_per_image if self.topk_per_image >= 0 else self.cand_cap
        if out is None:
            out = detection_buffers(n, max_det, dev)
        if n == 0:
            return out
        workspace, wsb, gate = detect_workspace(workspace, n, self.cand_cap, dev)
        w = self.box2box_transform
        with torch.cuda.device(dev):
            N.call("det_roi_detect_typed", N.ptr(lg), N.ptr(dl), code, N.ptr(props), N.ptr(offsets), n, lg.shape[0], K,
                   int(self.class_agnostic), N.ptr(sizes), *w.weights, w.scale_clamp, self.score_thresh,
                   self.nms_thresh, self.mode, gate, self.cand_cap, max_det, N.ptr(out["idx"]), N.ptr(out["boxes"]),
                   N.ptr(out["scores"]), N.ptr(out["classes"]), N.ptr(out["count"]), N.ptr(out["overflow"]),
                   N.ptr(workspace), wsb, N.stream())
        if check and int(out["overflow"].item()) != 0:
            p_max = int((offsets[1:] - offsets[:-1]).max())
            return _select_dense(lg, dl, code, props, offsets, sizes, n, p_max, K, self.class_agnostic, False,
                                 w.weights, w.scale_clamp, self.score_thresh, self.nms_thresh, self.topk_per_image,
                                 self.mode)
        return out

    def inference(self, predictions: Tuple[torch.Tensor, torch.Tensor], proposals: List[Instances]):
        """detectron2's FastRCNNOutputLayers.inference: predictions = (class_logits, proposal_deltas) over the
        concatenated proposals of the images, proposals = per-image Instances with proposal_boxes.  Returns
        (List[Instances] with pred_boxes, scores, pred_classes; List[Tensor] kept proposal indices)."""
        class_logits, deltas = predictions
        dev = class_logits.device
        boxes = [p.proposal_boxes.tensor if isinstance(p.proposal_boxes, Boxes) else p.proposal_boxes for p in proposals]
        shapes = [tuple(p.image_size) for p in proposals]
        pb = boxes[0] if len(boxes) == 1 else torch.cat(boxes, 0)
        out = self.inference_batched(class_logits, deltas, pb, _packed_offsets([len(b) for b in boxes], dev),
                                     _sizes_tensor(shapes, dev), check=True)
        return _instances(out, shapes, self.num_classes)

    # ------------------------------------------------------------------ training losses
    def _loss_scales(self, m):
        """(loss_type, w_cls / max(m, 1), w_loc / max(m, 1)): detectron2 averages both losses over all m rows."""
        if self.box_reg_loss_type not in ("smooth_l1", "giou"):
            raise ValueError(f"Invalid bbox reg loss type '{self.box_reg_loss_type}'")
        norm = float(max(m, 1))
        return (0 if self.box_reg_loss_type == "smooth_l1" else 1), \
            float(self.loss_weight.get("loss_cls", 1.0)) / norm, float(self.loss_weight.get("loss_box_reg", 1.0)) / norm

    def _run_loss(self, lg, dl, code, props, gt_classes, gt_boxes, upstream, grad_logits, grad_deltas):
        """One det_fast_rcnn_loss_typed launch: returns sums (8) = [loss_cls, loss_box_reg, num_fg, num_accurate,
        fg_num_accurate, num_false_negative, num_bad_labels, 0], the losses already weighted and normalised."""
        m = lg.shape[0]
        loss_type, s_cls, s_loc = self._loss_scales(m)
        w = self.box2box_transform
        dev = lg.device
        with torch.cuda.device(dev):
            sums = torch.empty((8,), dtype=torch.float32, device=dev)
            N.call("det_fast_rcnn_loss_typed", N.ptr(lg), N.ptr(dl), code, N.ptr(props), N.ptr(gt_classes),
                   N.ptr(gt_boxes), m, self.num_classes, int(self.class_agnostic), *w.weights, w.scale_clamp,
                   loss_type, self.smooth_l1_beta, s_cls, s_loc, N.ptr(upstream), N.ptr(N.accumulators(dev)),
                   N.ptr(sums), N.ptr(grad_logits), N.ptr(grad_deltas), N.stream())
        return sums

    def losses_batched(self, class_logits: torch.Tensor, deltas: torch.Tensor, proposal_boxes: torch.Tensor,
                       gt_classes: torch.Tensor, gt_boxes: torch.Tensor, with_grads: bool = False) -> dict:
        """detectron2's FastRCNNOutputLayers.losses on the M rows the box head saw, packed over the batch:
        class_logits (M, K+1), deltas (M, K*4) or (M, 4) (fp32, or bf16 / fp16 read as they are), proposal_boxes and
        gt_boxes (M, 4) (a row without gt carries its proposal box), gt_classes (M,) int64 in [0, K], K = background.

        Returns {"loss_cls", "loss_box_reg", "sums"}: device scalars autograd-connected to class_logits and deltas
        (backward is one more launch, gradients in the inputs' dtype), and the 8-float sums vector of
        det_fast_rcnn_loss_typed with detectron2's classification statistics in [2:6].  with_grads=True: one fused
        forward + backward launch that adds grad_logits / grad_deltas (d(loss_cls + loss_box_reg)/d(input), detached).
        No host synchronisation either way, so the call can be captured in a CUDA graph."""
        N.require_cuda(class_logits, deltas, proposal_boxes, gt_classes, gt_boxes)
        self._check_rows(class_logits, deltas, proposal_boxes)
        m = class_logits.shape[0]
        if gt_classes.shape != (m,) or gt_boxes.shape != (m, 4):
            raise ValueError(f"gt_classes must be ({m},) and gt_boxes ({m}, 4), got {tuple(gt_classes.shape)}, "
                             f"{tuple(gt_boxes.shape)}")
        self._loss_scales(m)  # an unknown loss type raises before anything is launched
        props, gtb = N.f32c(proposal_boxes), N.f32c(gt_boxes)
        gtc = gt_classes.detach().to(torch.int64).contiguous()
        if with_grads:
            (lg, dl), code = N.heads_c([class_logits, deltas])
            gl, gd = torch.empty_like(lg), torch.empty_like(dl)
            sums = self._run_loss(lg, dl, code, props, gtc, gtb, None, gl, gd)
        else:
            sums = _FastRCNNLoss.apply(self, class_logits, deltas, props, gtc, gtb)
        out = {"loss_cls": sums[0], "loss_box_reg": sums[1], "sums": sums}
        if with_grads:
            out["grad_logits"], out["grad_deltas"] = gl, gd
        return out

    def losses(self, predictions: Tuple[torch.Tensor, torch.Tensor], proposals: List[Instances]) -> Dict[str, torch.Tensor]:
        """detectron2's FastRCNNOutputLayers.losses: predictions = (class_logits, proposal_deltas) over the sampled
        proposals of the images, proposals = per-image Instances with proposal_boxes, gt_classes and, where the image
        has gt, gt_boxes.  Returns {"loss_cls", "loss_box_reg"}; the device sums vector (classification statistics
        included) stays in self.last_sums for logging, read back only when the caller wants it."""
        class_logits, deltas = predictions
        dev = class_logits.device
        box = lambda b: b.tensor if isinstance(b, Boxes) else b
        if len(proposals):
            pb = torch.cat([box(p.proposal_boxes) for p in proposals], 0)
            gtc = torch.cat([p.gt_classes for p in proposals], 0)
            gtb = torch.cat([box(p.gt_boxes if p.has("gt_boxes") else p.proposal_boxes) for p in proposals], 0)
        else:
            pb = gtb = torch.empty((0, 4), dtype=torch.float32, device=dev)
            gtc = torch.empty((0,), dtype=torch.int64, device=dev)
        res = self.losses_batched(class_logits, deltas, pb, gtc, gtb)
        self.last_sums = res["sums"].detach()
        return {"loss_cls": res["loss_cls"], "loss_box_reg": res["loss_box_reg"]}


def fast_rcnn_inference(boxes: List[torch.Tensor], scores: List[torch.Tensor], image_shapes: List[Tuple[int, int]],
                        score_thresh: float, nms_thresh: float, topk_per_image: int, mode: int = MODE_AUTO):
    """detectron2's fast_rcnn_inference over boxes and probabilities the caller already computed: per image boxes
    (R_i, K*4) or (R_i, 4) (class-agnostic) and scores (R_i, K+1).  Rows with a non-finite box or score are dropped,
    boxes are clipped, candidates are score > score_thresh, then per-class NMS and top-k (topk_per_image < 0: all).
    Runs on the library's unfused route (det_roi_decode_dense_typed on decoded rows -> det_threshold_compact ->
    det_nms_batched -> det_gather_detections); limit: the largest R_i * K <= 131071.  Returns (List[Instances],
    List[Tensor] kept row indices of the ORIGINAL rows)."""
    N.require_cuda(*boxes, *scores)
    if len(scores) == 0:
        return [], []
    dev = scores[0].device
    K = scores[0].shape[1] - 1
    agnostic = boxes[0].shape[1] == 4 and K != 1
    rows = scores[0] if len(scores) == 1 else torch.cat(scores, 0)
    cols = boxes[0] if len(boxes) == 1 else torch.cat(boxes, 0)
    (sc, bx), code = N.heads_c([rows, cols])
    n = len(scores)
    p_max = max(int(s.shape[0]) for s in scores)
    out = _select_dense(sc, bx, code, None, _packed_offsets([s.shape[0] for s in scores], dev),
                        _sizes_tensor(image_shapes, dev), n, p_max, K, agnostic, True, (1.0, 1.0, 1.0, 1.0), 0.0,
                        score_thresh, nms_thresh, int(topk_per_image), mode)
    return _instances(out, image_shapes, K)
