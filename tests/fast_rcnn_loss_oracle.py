"""Specification of the second-stage training losses: detectron2 v0.6 FastRCNNOutputLayers.losses (softmax
cross-entropy + box_reg_loss) and _log_classification_stats, restated in fp32 torch autograd on top of oracle/ref_torch
(get_deltas, apply_deltas, smooth_l1_sum, giou_sum).  One deviation, the library's: a label outside [0, K] (detectron2
device-asserts on it) contributes to neither loss and has zero gradients; M stays the denominator.

Runs on whatever device its inputs are on: CPU for the parity tests, CUDA for the end-to-end graph."""
import torch
import torch.nn.functional as F

from oracle.ref_torch import DEFAULT_SCALE_CLAMP, apply_deltas, get_deltas, giou_sum, smooth_l1_sum


def fast_rcnn_losses(logits, deltas, proposals, gt_classes, gt_boxes, num_classes, loss_type="smooth_l1", beta=0.0,
                     weights=(10.0, 10.0, 5.0, 5.0), scale_clamp=DEFAULT_SCALE_CLAMP, loss_weight=1.0):
    """-> {"loss_cls", "loss_box_reg"} (autograd-connected to logits and deltas) and the statistics
    {"num_fg", "num_accurate", "fg_num_accurate", "num_false_negative", "num_bad_labels"} as Python ints."""
    K = num_classes
    M = logits.shape[0]
    gt = gt_classes.long()
    lw = loss_weight if isinstance(loss_weight, dict) else {"loss_cls": loss_weight, "loss_box_reg": loss_weight}
    valid = (gt >= 0) & (gt <= K)
    fg = (gt >= 0) & (gt < K)
    if M == 0:
        loss_cls = logits.sum() * 0.0  # detectron2's cross_entropy on an empty batch
    else:
        ce = F.cross_entropy(logits, torch.where(valid, gt, torch.zeros_like(gt)), reduction="none")
        loss_cls = torch.where(valid, ce, torch.zeros_like(ce)).sum() / M
    fg_inds = fg.nonzero().squeeze(1)
    if deltas.shape[1] == 4:  # class-agnostic (detectron2's test: one box's worth of deltas per row)
        d = deltas[fg_inds]
    else:
        d = deltas.view(M, K, 4)[fg_inds, gt[fg_inds]]
    p, g = proposals[fg_inds], gt_boxes[fg_inds]
    if loss_type == "smooth_l1":
        box = smooth_l1_sum(d, get_deltas(p, g, weights), beta)
    elif loss_type == "giou":
        box = giou_sum(apply_deltas(d, p, weights, scale_clamp), g) if len(fg_inds) else d.sum() * 0.0
    else:
        raise ValueError(loss_type)
    loss_box = box / max(M, 1)
    pred = logits.detach().argmax(dim=1) if M else gt
    stats = {"num_fg": int(fg.sum()), "num_accurate": int((pred == gt).sum()),
             "fg_num_accurate": int((pred[fg] == gt[fg]).sum()), "num_false_negative": int((pred[fg] == K).sum()),
             "num_bad_labels": int((~valid).sum())}
    return {"loss_cls": loss_cls * lw.get("loss_cls", 1.0), "loss_box_reg": loss_box * lw.get("loss_box_reg", 1.0)}, stats
