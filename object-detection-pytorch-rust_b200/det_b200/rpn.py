"""RPN hot path -- drop-in for the post-head methods of ``RegionProposalNetwork``
(reference python/src/models/rpn.py:17-357): layout change + decode, label_and_sample_anchors, losses,
predict_proposals.  The conv head itself is out of scope (SURVEY.md section 2 row 12): ``forward`` takes the head's
NCHW outputs.  Two API levels:
  * the reference's own signatures (lists of per-level / per-image tensors, ``Boxes``, ``Instances``);
  * batched zero-synchronisation forms (``decode_heads``, ``assign``, ``fused_losses``) the former are built on.
"""
import math
from typing import Dict, List, Optional, Sequence, Tuple, Union

import ctypes

import torch

from . import _native as N
from .anchors import AnchorGenerator
from .box_regression import Box2BoxTransform, _DEFAULT_SCALE_CLAMP
from .matcher import Matcher, subsample_labels_
from .proposals import find_top_rpn_proposals, rpn_proposals_batched
from .structures import Boxes, Instances


class Assignment:
    """Result of the batched target assignment: labels (N,R) int8, matched (N,R) int64 indices into each image's own
    gt boxes, the packed gt table (sum_G,4) and its int32 offsets (N+1).  After a grid assignment with sampling it
    also carries the per-image sample lists (N,S) int32 (anchor row | label << 24) + counts (N) int32 that the sampled
    loss (det_rpn_loss_sampled) works from.  A sample-list-only assignment (assign_sampled) has labels = matched = None
    and sample_gt (N,S) int32 = the matched gt index of every sample instead."""

    def __init__(self, labels, matched, gt_table, gt_offsets, samples=None, sample_count=None, sample_gt=None):
        self.labels, self.matched, self.gt_table, self.gt_offsets = labels, matched, gt_table, gt_offsets
        self.samples, self.sample_count, self.sample_gt = samples, sample_count, sample_gt


class _FusedRPNLoss(torch.autograd.Function):
    """Forward: one pass that reduces the BCE / L1 sums (no gradient stores).  Backward: the same kernel with the
    upstream gradients read on the device, writing grad_logits / grad_deltas.  `fused_losses(..., with_grads=True)`
    is the single-launch fwd+bwd form used when the caller drives backward by hand.

    Everything the backward launch reads -- anchors and the four Assignment tensors -- is an explicit argument and
    goes through save_for_backward: two forwards before one backward (gradient accumulation, multi-scale batches)
    each keep their own anchors, and an in-place change of the labels between forward and backward (e.g. a later
    subsample_labels_) trips autograd's version check instead of silently encoding against the wrong targets."""

    @staticmethod
    def forward(ctx, logits, deltas, anchors, labels, matched, gt_table, gt_offsets, owner, n_norm):
        asg = Assignment(labels, matched, gt_table, gt_offsets)
        sums = owner._run_loss(anchors, logits, deltas, asg, n_norm, None, None, None)
        ctx.owner, ctx.n_norm = owner, n_norm
        ctx.save_for_backward(logits, deltas, anchors, labels, matched, gt_table, gt_offsets)
        return sums

    @staticmethod
    def backward(ctx, grad_sums):
        logits, deltas, anchors, labels, matched, gt_table, gt_offsets = ctx.saved_tensors
        up = grad_sums[:2].contiguous().float()
        gl = torch.empty_like(logits)
        gd = torch.empty_like(deltas)
        ctx.owner._run_loss(anchors, logits, deltas, Assignment(labels, matched, gt_table, gt_offsets), ctx.n_norm, up,
                            gl, gd)
        return gl, gd, None, None, None, None, None, None, None


class _SampledRPNLoss(torch.autograd.Function):
    """det_rpn_loss_sampled behind autograd: forward reduces the sums from the NCHW head tensors, backward re-launches
    the kernel with the upstream gradients read on the device and scatters into zero-initialised NCHW gradients."""

    @staticmethod
    def forward(ctx, owner, n_norm, nl, anchors, matched, sample_gt, gt_table, gt_offsets, samples, sample_count, *heads):
        obj = [h.contiguous() for h in heads[:nl]]
        dlt = [h.contiguous() for h in heads[nl:]]
        asg = Assignment(None, matched, gt_table, gt_offsets, samples, sample_count, sample_gt)
        sums = owner._run_sampled(anchors, obj, dlt, asg, n_norm, None, None)
        ctx.owner, ctx.n_norm, ctx.nl = owner, n_norm, nl
        ctx.save_for_backward(anchors, matched, sample_gt, gt_table, gt_offsets, samples, sample_count, *obj, *dlt)
        return sums

    @staticmethod
    def backward(ctx, grad_sums):
        anchors, matched, sample_gt, gt_table, gt_offsets, samples, sample_count = ctx.saved_tensors[:7]
        heads = ctx.saved_tensors[7:]
        obj, dlt = list(heads[:ctx.nl]), list(heads[ctx.nl:])
        up = grad_sums[:2].contiguous().float()
        g_obj, g_dlt = [torch.zeros_like(o) for o in obj], [torch.zeros_like(d) for d in dlt]
        asg = Assignment(None, matched, gt_table, gt_offsets, samples, sample_count, sample_gt)
        ctx.owner._run_sampled(anchors, obj, dlt, asg, ctx.n_norm, up, (g_obj, g_dlt))
        return (None,) * 10 + tuple(g_obj) + tuple(g_dlt)


class RegionProposalNetwork:
    def __init__(self, strides: Sequence[int], anchor_sizes=((32,), (64,), (128,), (256,), (512,)),
                 aspect_ratios=((0.5, 1.0, 2.0),), anchor_offset: float = 0.0,
                 iou_thresholds=(0.3, 0.7), iou_labels=(0, -1, 1), allow_low_quality_matches: bool = True,
                 box2box_weights=(1.0, 1.0, 1.0, 1.0), scale_clamp: float = _DEFAULT_SCALE_CLAMP,
                 batch_size_per_image: int = 256, positive_fraction: float = 0.5,
                 pre_nms_topk: Tuple[int, int] = (12000, 6000), post_nms_topk: Tuple[int, int] = (2000, 1000),
                 nms_thresh: float = 0.7, min_box_size: float = 0.0, loss_weight=(1.0, 1.0),
                 box_reg_loss_type: str = "smooth_l1", smooth_l1_beta: float = 0.0, head=None):
        """Defaults = reference python/src/config/rpn.py:113-130 (pre/post_nms_topk are indexed by `training`)."""
        self.anchor_generator = AnchorGenerator(list(strides), anchor_sizes, aspect_ratios, anchor_offset)
        self.anchor_matcher = Matcher(list(iou_thresholds), list(iou_labels), allow_low_quality_matches)
        self.box2box_transform = Box2BoxTransform(box2box_weights, scale_clamp)
        self.batch_size_per_image = batch_size_per_image
        self.positive_fraction = positive_fraction
        self.pre_nms_topk = pre_nms_topk
        self.post_nms_topk = post_nms_topk
        self.nms_thresh = nms_thresh
        self.min_box_size = float(min_box_size)
        self.loss_weight = loss_weight
        self.box_reg_loss_type = box_reg_loss_type
        self.smooth_l1_beta = smooth_l1_beta
        self.head = head
        self.training = False
        self._sample_seed = 0
        self._anchor_cache = {}

    @classmethod
    def build(cls, conf, input_shapes):
        strides = [input_shapes[f].stride for f in conf.in_features]
        return cls(strides, conf.anchor_generator.sizes, conf.anchor_generator.aspect_ratios,
                   conf.anchor_generator.offset, conf.anchor_matcher.thresholds, conf.anchor_matcher.labels,
                   conf.anchor_matcher.allow_low_quality_matches, conf.box2box_transform.weights,
                   conf.box2box_transform.scale_clamp, conf.batch_size_per_image, conf.positive_fraction,
                   conf.pre_nms_topk, conf.post_nms_topk, conf.nms_thresh, conf.min_box_size, conf.loss_weight,
                   conf.box_reg_loss_type, conf.smooth_l1_beta)

    def train(self, mode: bool = True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)

    # ------------------------------------------------------------------ decode
    def decode_heads(self, pred_objectness: List[torch.Tensor], pred_deltas: List[torch.Tensor]):
        """Conv-layout head outputs, per level (N,A,Hi,Wi) and (N,A*4,Hi,Wi) -> logits (N,R), proposals (N,R,4) with all
        levels concatenated in (level,h,w,a) order; anchors are synthesised in the kernel (rpn.py:270-284 + :330-348).
        bf16 / fp16 heads (objectness and deltas of every level one dtype) are read as they are: bit-identical to the
        fp32 heads h.float()."""
        N.require_cuda(*pred_objectness, *pred_deltas)
        dev = pred_objectness[0].device
        n = pred_objectness[0].shape[0]
        cells = self.anchor_generator.device_cell_anchors(dev)
        sizes = [o.shape[1] * o.shape[2] * o.shape[3] for o in pred_objectness]
        R = sum(sizes)
        logits = torch.empty((n, R), dtype=torch.float32, device=dev)
        boxes = torch.empty((n, R, 4), dtype=torch.float32, device=dev)
        w = self.box2box_transform.weights
        nl = len(pred_objectness)
        hcs, code = N.heads_c(list(pred_objectness) + list(pred_deltas))
        ocs, dcs = hcs[:nl], hcs[nl:]
        na = ocs[0].shape[1]
        if all(o.shape[1] == na for o in ocs):  # one launch for the whole pyramid (det_rpn_decode)
            lv = (N.RpnLevel * len(ocs))()
            off = 0
            for i, (oc, dc, cell, stride, sz) in enumerate(zip(ocs, dcs, cells, self.anchor_generator.strides, sizes)):
                assert dc.shape[1] == na * 4 and na == cell.shape[0]
                lv[i].objectness, lv[i].deltas, lv[i].cell_anchors = oc.data_ptr(), dc.data_ptr(), cell.data_ptr()
                lv[i].h, lv[i].w, lv[i].stride, lv[i].reserved, lv[i].out_offset = oc.shape[2], oc.shape[3], int(stride), 0, off
                off += sz
            with torch.cuda.device(dev):
                N.call("det_rpn_decode_typed", ctypes.cast(lv, ctypes.c_void_p), len(ocs), n, na,
                       float(self.anchor_generator.offset), *w, self.box2box_transform.scale_clamp, N.ptr(logits),
                       N.ptr(boxes), R, code, N.stream())
            return logits, boxes, sizes
        off = 0
        with torch.cuda.device(dev):
            for oc, dc, cell, stride, sz in zip(ocs, dcs, cells, self.anchor_generator.strides, sizes):
                a, h, wd = oc.shape[1], oc.shape[2], oc.shape[3]
                assert dc.shape[1] == a * 4 and a == cell.shape[0]
                lv = N.RpnLevel(oc.data_ptr(), dc.data_ptr(), cell.data_ptr(), h, wd, int(stride), 0, off)
                N.call("det_rpn_decode_typed", ctypes.byref(lv), 1, n, a, float(self.anchor_generator.offset), *w,
                       self.box2box_transform.scale_clamp, N.ptr(logits), N.ptr(boxes), R, code, N.stream())
                off += sz
        return logits, boxes, sizes

    def _decode_proposals(self, anchors: List[Boxes], pred_anchor_deltas: List[torch.Tensor]) -> List[torch.Tensor]:
        """Reference signature (rpn.py:330): per level (N,HiWiA,4) deltas + anchors -> (N,HiWiA,4) proposals."""
        out = []
        for a, d in zip(anchors, pred_anchor_deltas):
            n = d.shape[0]
            at = a.tensor if isinstance(a, Boxes) else a
            rep = at.unsqueeze(0).expand(n, -1, -1).reshape(-1, 4)
            out.append(self.box2box_transform.apply_deltas(d.reshape(-1, 4), rep).view(n, -1, 4))
        return out

    # ------------------------------------------------------------------ assignment
    def assign(self, anchors: torch.Tensor, gt_boxes: List[torch.Tensor], sample: bool = True,
               seed: Optional[int] = None, grid=None) -> Assignment:
        """Batched IoU -> Matcher -> (optional) device fg/bg subsample; no (G,R) matrix, no per-image loop.
        grid = AnchorGenerator.grid_layout(feature sizes) when `anchors` is that generator's table: one-pass grid
        matcher + O(samples) subsample, and the Assignment carries the sample lists for `sampled_losses`."""
        gts = [g.tensor if isinstance(g, Boxes) else g for g in gt_boxes]
        use_grid = grid is not None
        res = self.anchor_matcher.match_boxes(gts, anchors, grid=grid, with_stats=use_grid and sample)
        if use_grid and sample:
            matched, labels, stats, table, offsets = res
        else:
            (matched, labels, table, offsets), stats = res, None
        samples = counts = None
        if sample:
            if seed is None:
                self._sample_seed += 1
                seed = self._sample_seed
            if stats is not None:
                _, samples, counts = subsample_labels_(labels, self.batch_size_per_image, self.positive_fraction, seed,
                                                       stats=stats, return_samples=True)
            else:
                subsample_labels_(labels, self.batch_size_per_image, self.positive_fraction, seed)
        return Assignment(labels, matched, table, offsets, samples, counts)

    def assign_sampled(self, anchors: torch.Tensor, gt_table: torch.Tensor, gt_offsets: torch.Tensor, n: int, grid,
                       seed: Optional[int] = None) -> Assignment:
        """label_and_sample_anchors reduced to what the losses read (det_assign_sampled): the sampled anchors of every
        image, their labels and matched gt -- nothing is computed or written for the other anchors.  gt_table (sum_G,4)
        + int32 gt_offsets (n+1) as in Matcher.match_packed; grid = AnchorGenerator.grid_layout(...)."""
        N.require_cuda(anchors, gt_table, gt_offsets)
        from .matcher import _rule_arrays, grid_supported
        m = self.anchor_matcher
        r, sum_g = anchors.shape[0], gt_table.shape[0]
        assert grid is not None and grid_supported(grid, r) and m.labels[0] in (0, -1) and r < (1 << 24)
        if seed is None:
            self._sample_seed += 1
            seed = self._sample_seed
        dev = anchors.device
        levels, a = grid
        lv = (N.AnchorLevel * len(levels))()
        row = 0
        for i, (h, w, stride) in enumerate(levels):
            lv[i].h, lv[i].w, lv[i].stride, lv[i].reserved, lv[i].first_row = int(h), int(w), int(stride), 0, row
            row += int(h) * int(w) * a
        cap = max(int(self.batch_size_per_image), 1)
        thr, lab = _rule_arrays(m._inner, m.labels)
        with torch.cuda.device(dev):
            samples = torch.empty((n, cap), dtype=torch.int32, device=dev)
            sample_gt = torch.empty((n, cap), dtype=torch.int32, device=dev)
            counts = torch.empty((n,), dtype=torch.int32, device=dev)
            scratch = torch.empty((n, r), dtype=torch.int8, device=dev)  # only written for images with dense positives
            wsb = N.fn("det_assign_sampled_workspace_bytes")(n, sum_g, 1024)
            ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)
            N.call("det_assign_sampled", N.ptr(gt_table), N.ptr(gt_offsets), n, sum_g, N.ptr(anchors), r,
                   ctypes.cast(lv, ctypes.c_void_p), len(levels), int(a), thr, lab, len(m._inner),
                   int(m.allow_low_quality_matches), int(self.batch_size_per_image), float(self.positive_fraction),
                   int(seed) & 0xFFFFFFFFFFFFFFFF, N.ptr(scratch), N.ptr(samples), N.ptr(sample_gt), N.ptr(counts), cap,
                   N.ptr(ws), wsb, N.stream())
        return Assignment(None, None, gt_table, gt_offsets, samples, counts, sample_gt)

    @staticmethod
    def _grid_of(level_tensors) -> Optional[tuple]:
        """(levels, a) if every per-level anchor tensor carries AnchorGenerator's layout tag, else None."""
        tags = [getattr(t, "_det_grid", None) for t in level_tensors]
        if any(t is None for t in tags) or len({t[3] for t in tags}) != 1:
            return None
        if any(t[0] * t[1] * t[3] != x.shape[0] for t, x in zip(tags, level_tensors)):
            return None
        return [(t[0], t[1], t[2]) for t in tags], tags[0][3]

    @torch.no_grad()
    def label_and_sample_anchors(self, anchors: List[Boxes], gt_instances: List[Instances]):
        """Reference signature (rpn.py:132): -> (list of int8[R] labels, list of (R,4) matched gt boxes)."""
        level_tensors = [a.tensor if isinstance(a, Boxes) else a for a in anchors]
        at = level_tensors[0] if len(level_tensors) == 1 else torch.cat(level_tensors, 0)
        gt_boxes = [x.gt_boxes for x in gt_instances]
        asg = self.assign(at, gt_boxes, sample=True, grid=self._grid_of(level_tensors))
        gt_labels, matched_gt = [], []
        for i, g in enumerate(gt_boxes):
            gt_labels.append(asg.labels[i])
            gt_t = g.tensor if isinstance(g, Boxes) else g
            matched_gt.append(torch.zeros_like(at) if len(gt_t) == 0 else gt_t[asg.matched[i]])
        return gt_labels, matched_gt

    # ------------------------------------------------------------------ losses
    def _loss_scales(self, n_norm):
        """(loss_type, w_cls / norm, w_loc / norm) with norm = batch_size_per_image * N_global (rpn.py:238-243)."""
        if self.box_reg_loss_type not in ("smooth_l1", "giou"):
            raise ValueError(f"Invalid dense box regression loss type '{self.box_reg_loss_type}'")
        norm = float(self.batch_size_per_image * n_norm)
        lw = self.loss_weight
        w_cls = float(getattr(lw, "cls_loss", lw[0] if isinstance(lw, (tuple, list)) else 1.0))
        w_loc = float(getattr(lw, "loc_loss", lw[1] if isinstance(lw, (tuple, list)) else 1.0))
        return (0 if self.box_reg_loss_type == "smooth_l1" else 1), w_cls / norm, w_loc / norm

    def _run_loss(self, anchors, logits, deltas, asg: Assignment, n_norm, upstream, grad_logits, grad_deltas):
        """One launch of the dense fused kernel: returns sums (8) = [cls_loss, loc_loss, #pos, #neg, 0...] already
        weighted and normalised (the kernel's last CTA does it: no memset before, no scaling op after)."""
        n, r = logits.shape
        dev = logits.device
        loss_type, s_cls, s_loc = self._loss_scales(n_norm)
        w = self.box2box_transform.weights
        with torch.cuda.device(dev):
            sums = torch.empty((8,), dtype=torch.float32, device=dev)
            N.call("det_rpn_loss", N.ptr(logits), N.ptr(deltas), N.ptr(asg.labels), N.ptr(asg.matched),
                   N.ptr(asg.gt_table), N.ptr(asg.gt_offsets), N.ptr(anchors), n, r, *w,
                   self.box2box_transform.scale_clamp, loss_type, float(self.smooth_l1_beta), s_cls, s_loc,
                   N.ptr(upstream), N.ptr(N.accumulators(dev)), N.ptr(sums), N.ptr(grad_logits), N.ptr(grad_deltas),
                   N.stream())
        return sums

    # ------------------------------------------------------------------ sampled losses on the conv-layout head
    def _run_sampled(self, anchors, obj, dlt, asg: Assignment, n_norm, upstream, grads, clear=None):
        """det_rpn_loss_sampled on per-level NCHW head tensors (obj[l] (N,A,H,W), dlt[l] (N,A*4,H,W)) -- or, with
        dlt.dim() == 3, on flat (N,R) / (N,R,4) tensors.  grads = (list of grad_obj, list of grad_dlt) buffers the
        kernel scatters into (None: forward only); clear = (samples, counts) of the previous step for persistent
        buffers.  Returns sums (8) like _run_loss."""
        assert asg.samples is not None, "sampled losses need an Assignment from assign(..., grid=...) with sampling"
        flat = isinstance(obj, torch.Tensor)
        dev = (obj if flat else obj[0]).device
        n = (obj if flat else obj[0]).shape[0]
        r = anchors.shape[0]
        loss_type, s_cls, s_loc = self._loss_scales(n_norm)
        w = self.box2box_transform.weights
        cs, cc = (None, None) if clear is None else clear
        with torch.cuda.device(dev):
            sums = torch.empty((8,), dtype=torch.float32, device=dev)
            if flat:
                lv, nl, a = None, 0, 1
                ptrs = (N.ptr(obj), N.ptr(dlt), N.ptr(grads[0] if grads else None), N.ptr(grads[1] if grads else None))
            else:
                a = obj[0].shape[1]
                lv = (N.HeadLevel * len(obj))()
                for i, (o, d) in enumerate(zip(obj, dlt)):
                    assert o.shape[1] == a and d.shape[1] == 4 * a and o.is_contiguous() and d.is_contiguous()
                    lv[i].objectness, lv[i].deltas = o.data_ptr(), d.data_ptr()
                    lv[i].grad_objectness = grads[0][i].data_ptr() if grads else None
                    lv[i].grad_deltas = grads[1][i].data_ptr() if grads else None
                    lv[i].h, lv[i].w = o.shape[2], o.shape[3]
                nl = len(obj)
                ptrs = (None, None, None, None)
                lv = ctypes.cast(lv, ctypes.c_void_p)
            N.call("det_rpn_loss_sampled", lv, nl, a, *ptrs, N.ptr(asg.samples), N.ptr(asg.sample_count),
                   asg.samples.shape[1], N.ptr(cs), N.ptr(cc), N.ptr(asg.matched), N.ptr(asg.sample_gt), N.ptr(asg.gt_table),
                   N.ptr(asg.gt_offsets), N.ptr(anchors), n, r, *w, self.box2box_transform.scale_clamp, loss_type,
                   float(self.smooth_l1_beta), s_cls, s_loc, N.ptr(upstream), N.ptr(N.accumulators(dev)), N.ptr(sums),
                   N.stream())
        return sums

    def sampled_losses(self, anchors: torch.Tensor, pred_objectness: List[torch.Tensor], pred_deltas: List[torch.Tensor],
                       asg: Assignment, num_images_global: Optional[int] = None, grad_buffers=None,
                       clear_previous=None):
        """The RPN losses straight from the head convolutions' NCHW outputs (per level (N,A,Hi,Wi) / (N,A*4,Hi,Wi)), on
        the sampled anchors only: no layout change (rpn.py:270-284), no dense label sweep, O(samples) traffic.

        Default: autograd-connected {"cls_loss", "loc_loss", ...}; backward re-launches the kernel, which scatters the
        gradients into zero-initialised NCHW tensors (exactly what the head convolutions' backward takes).
        grad_buffers=(list grad_obj, list grad_dlt): fused forward+backward in ONE launch into caller-owned buffers --
        zeroed by the caller, or persistent with clear_previous=(samples, counts) of the step that last wrote them."""
        N.require_cuda(anchors, *pred_objectness, *pred_deltas)
        at = N.f32c(anchors)
        n_norm = pred_objectness[0].shape[0] if num_images_global is None else int(num_images_global)
        if grad_buffers is not None:
            obj = [o.detach().contiguous() for o in pred_objectness]
            dlt = [d.detach().contiguous() for d in pred_deltas]
            sums = self._run_sampled(at, obj, dlt, asg, n_norm, None, grad_buffers, clear_previous)
        else:
            nl = len(pred_objectness)
            sums = _SampledRPNLoss.apply(self, n_norm, nl, at, asg.matched, asg.sample_gt, asg.gt_table, asg.gt_offsets,
                                         asg.samples, asg.sample_count, *pred_objectness, *pred_deltas)
        return {"cls_loss": sums[0], "loc_loss": sums[1], "num_pos_anchors": sums[2].detach(),
                "num_neg_anchors": sums[3].detach(), "sums": sums}

    def fused_losses(self, anchors: torch.Tensor, logits: torch.Tensor, deltas: torch.Tensor, asg: Assignment,
                     num_images_global: Optional[int] = None, with_grads: bool = False):
        """logits (N,R), deltas (N,R,4).  Returns {"cls_loss","loc_loss","num_pos_anchors","num_neg_anchors"} (device
        scalars, autograd-connected to logits/deltas) -- or, with_grads=True, additionally grad_logits/grad_deltas from
        the SAME launch (fused forward+backward, detached).  `num_images_global` = batch size over all data-parallel
        ranks (normaliser = batch_size_per_image * that, rpn.py:238)."""
        N.require_cuda(anchors, logits, deltas)
        at = N.f32c(anchors)
        # the loss kernel reads fp32: a 16-bit head (forward(training) sends those here) is converted, autograd-connected
        lg, dl = logits.float().contiguous(), deltas.float().contiguous()
        n_norm = lg.shape[0] if num_images_global is None else int(num_images_global)
        if with_grads:
            gl, gd = torch.empty_like(lg), torch.empty_like(dl)
            sums = self._run_loss(at, lg.detach(), dl.detach(), asg, n_norm, None, gl, gd)
        else:
            sums = _FusedRPNLoss.apply(lg, dl, at, asg.labels, asg.matched, asg.gt_table, asg.gt_offsets, self, n_norm)
        out = {"cls_loss": sums[0], "loc_loss": sums[1], "num_pos_anchors": sums[2].detach(),
               "num_neg_anchors": sums[3].detach(), "sums": sums}
        if with_grads:
            out["grad_logits"], out["grad_deltas"] = gl, gd
        return out

    def losses(self, anchors: List[Boxes], pred_objectness_logits: List[torch.Tensor], gt_labels: List[torch.Tensor],
               pred_anchor_deltas: List[torch.Tensor], gt_boxes: List[torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Reference signature (rpn.py:187): per-level logits (N,HiWiA) / deltas (N,HiWiA,4), per-image labels int8[R]
        and matched gt boxes (R,4) -> {"cls_loss", "loc_loss"}."""
        at = Boxes.cat(anchors).tensor
        labels = torch.stack(gt_labels).contiguous()
        n, r = labels.shape
        logits = pred_objectness_logits[0] if len(pred_objectness_logits) == 1 else torch.cat(pred_objectness_logits, 1)
        deltas = pred_anchor_deltas[0] if len(pred_anchor_deltas) == 1 else torch.cat(pred_anchor_deltas, 1)
        table = N.f32c(torch.stack(gt_boxes).reshape(-1, 4))      # matched boxes as an (N*R,4) table ...
        matched = torch.arange(r, device=at.device, dtype=torch.int64).repeat(n, 1)  # ... indexed by the anchor id
        offsets = (torch.arange(n + 1, device=at.device, dtype=torch.int64) * r).to(torch.int32)
        res = self.fused_losses(at, logits, deltas, Assignment(labels, matched, table, offsets))
        return {"cls_loss": res["cls_loss"], "loc_loss": res["loc_loss"]}

    # ------------------------------------------------------------------ proposals
    def predict_proposals(self, anchors: List[Boxes], pred_objectness_logits: List[torch.Tensor],
                          pred_anchor_deltas: List[torch.Tensor], image_sizes: List[Tuple[int, int]]):
        """Reference signature (rpn.py:299)."""
        with torch.no_grad():
            props = self._decode_proposals(anchors, pred_anchor_deltas)
            return find_top_rpn_proposals(props, pred_objectness_logits, image_sizes, self.nms_thresh,
                                          self.pre_nms_topk[self.training], self.post_nms_topk[self.training],
                                          self.min_box_size, self.training)

    @torch.no_grad()
    def proposals_from_heads(self, pred_objectness: List[torch.Tensor], pred_deltas: List[torch.Tensor],
                             image_sizes: torch.Tensor):
        """Zero-synchronisation inference path: conv-layout heads -> padded proposals (N,K,4), logits (N,K), counts (N)."""
        logits, boxes, sizes = self.decode_heads(pred_objectness, pred_deltas)
        return rpn_proposals_batched(boxes, logits, sizes, image_sizes, self.nms_thresh,
                                     self.pre_nms_topk[self.training], self.post_nms_topk[self.training],
                                     self.min_box_size)

    def _cached_anchors(self, feats_hw, device):
        """Per-level anchors + their concatenation for these feature sizes: a pure function of the shapes
        (anchor_generators.py:212-225 recomputes them every forward), so they are generated once per shape."""
        key = (tuple(feats_hw), str(device))
        hit = self._anchor_cache.get(key)
        if hit is None:
            if len(self._anchor_cache) > 16:
                self._anchor_cache.clear()
            levels = self.anchor_generator.grid_anchors(feats_hw, device)
            hit = (levels, levels[0] if len(levels) == 1 else torch.cat(levels, 0))
            self._anchor_cache[key] = hit
        return hit

    def forward(self, images, features: Dict[str, torch.Tensor] = None, gt_instances: Optional[List[Instances]] = None,
                head_outputs=None):
        """`forward` of the reference (rpn.py:246) from the head outputs: (objectness list, deltas list) in the conv
        layout, either passed as `head_outputs` or produced by the optional `head` callable from `features`."""
        if head_outputs is None:
            assert self.head is not None, "pass head_outputs=(objectness, deltas) or construct with head=..."
            head_outputs = self.head(features)
        obj, dlt = head_outputs
        image_sizes = images.image_sizes if hasattr(images, "image_sizes") else images
        feats_hw = [tuple(int(v) for v in o.shape[-2:]) for o in obj]
        anchors, anchors_cat = self._cached_anchors(feats_hw, obj[0].device)
        losses = {}
        if self.training:
            # grid matcher -> O(samples) subsample -> sampled loss reading the NCHW head in place: the reference's
            # layout change (rpn.py:270-284) is never materialised and only library kernels of this package launch
            assert gt_instances is not None, "RPN requires gt_instances in training!"
            at = anchors_cat
            grid = self.anchor_generator.grid_layout(feats_hw)
            from .matcher import grid_supported
            if (grid is not None and grid_supported(grid, at.shape[0]) and self.anchor_matcher.labels[0] in (0, -1)
                    and all(o.dtype == torch.float32 for o in obj)):
                gts = [x.gt_boxes.tensor if isinstance(x.gt_boxes, Boxes) else x.gt_boxes for x in gt_instances]
                table, offsets = self.anchor_matcher.pack_gt(gts, at.device)
                asg = self.assign_sampled(at, table, offsets, len(gts), grid)
                res = self.sampled_losses(at, list(obj), list(dlt), asg)
            else:  # levels with different anchor counts: generic matcher + dense loss on re-laid-out tensors
                n = obj[0].shape[0]
                logits = [o.permute(0, 2, 3, 1).reshape(n, -1) for o in obj]
                deltas = [d.view(n, -1, 4, d.shape[-2], d.shape[-1]).permute(0, 3, 4, 1, 2).reshape(n, -1, 4) for d in dlt]
                asg = self.assign(at, [x.gt_boxes for x in gt_instances])
                res = self.fused_losses(at, torch.cat(logits, 1), torch.cat(deltas, 1), asg)
            losses = {"cls_loss": res["cls_loss"], "loc_loss": res["loc_loss"]}
        sizes = torch.tensor([[int(h), int(w)] for h, w in image_sizes], dtype=torch.int32).to(obj[0].device)
        ob, os_, cnt, flag = self.proposals_from_heads(obj, dlt, sizes)
        counts = cnt.tolist()
        if self.training and int(flag.item()):
            raise FloatingPointError("Predicted boxes or scores contain Inf/NaN. Training has diverged.")
        proposals = []
        for i, sz in enumerate(image_sizes):
            inst = Instances(tuple(sz))
            inst.proposal_boxes = Boxes(ob[i, :counts[i]])
            inst.objectness_logits = os_[i, :counts[i]]
            proposals.append(inst)
        return proposals, losses

    __call__ = forward


def _dense_box_regression_loss(anchors: List[Boxes], box2box_transform: Box2BoxTransform,
                               pred_anchor_deltas: List[torch.Tensor], gt_boxes: List[torch.Tensor],
                               fg_mask: torch.Tensor, box_reg_loss_type="smooth_l1", smooth_l1_beta=0.0):
    """Reference signature (components/box_regression.py:128): summed localisation loss over fg_mask."""
    if box_reg_loss_type not in ("smooth_l1", "giou"):
        raise ValueError(f"Invalid dense box regression loss type '{box_reg_loss_type}'")
    rpn = RegionProposalNetwork([1], box2box_weights=box2box_transform.weights,
                                scale_clamp=box2box_transform.scale_clamp, batch_size_per_image=1,
                                box_reg_loss_type=box_reg_loss_type, smooth_l1_beta=smooth_l1_beta)
    at = type(anchors[0]).cat(anchors).tensor
    n, r = fg_mask.shape
    deltas = pred_anchor_deltas[0] if len(pred_anchor_deltas) == 1 else torch.cat(pred_anchor_deltas, 1)
    labels = torch.where(fg_mask, 1, -1).to(torch.int8).contiguous()
    table = N.f32c(torch.stack(gt_boxes).reshape(-1, 4))
    matched = torch.arange(r, device=at.device, dtype=torch.int64).repeat(n, 1)
    offsets = (torch.arange(n + 1, device=at.device, dtype=torch.int64) * r).to(torch.int32)
    logits = torch.zeros((n, r), dtype=torch.float32, device=at.device)
    res = rpn.fused_losses(at, logits, deltas, Assignment(labels, matched, table, offsets), num_images_global=1)
    return res["loc_loss"]
