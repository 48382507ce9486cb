"""ROI-head side of target assignment -- drop-in for the matching / sampling half of the reference's ``ROIHeads``
(python/src/models/roi.py:15-193) and for ``subsample_labels`` (python/src/utils.py:34-76).

The IoU + Matcher arithmetic runs in the fused device kernels (det_match_anchors: no (G, P) matrix is materialised);
the fg/bg subsample keeps the reference's two ``torch.randperm`` calls so that, under the same torch seed, the sampled
indices are the reference's (SURVEY.md section 8 row a11); the class-label convention is the reference's:
background = ``num_classes``, ignored = -1 (roi.py:84-95)."""
from typing import Dict, List, Optional, Tuple

import torch

from . import _native as N
from .matcher import Matcher, _rule_arrays
from .proposals import add_ground_truth_to_proposals
from .structures import Boxes, Instances


def subsample_labels(labels: torch.Tensor, num_samples: int, positive_fraction: float,
                     bg_label: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Indices of up to ``num_samples`` random elements of ``labels``: at most ``int(num_samples * positive_fraction)``
    positives (neither -1 nor ``bg_label``), the rest background -- same contract, counts and RNG consumption as
    reference python/src/utils.py:34-76."""
    positive = torch.nonzero((labels != -1) & (labels != bg_label), as_tuple=True)[0]
    negative = torch.nonzero(labels == bg_label, as_tuple=True)[0]
    num_pos = min(positive.numel(), int(num_samples * positive_fraction))
    num_neg = min(negative.numel(), num_samples - num_pos)
    pick_pos = torch.randperm(positive.numel(), device=positive.device)[:num_pos]
    pick_neg = torch.randperm(negative.numel(), device=negative.device)[:num_neg]
    return positive[pick_pos], negative[pick_neg]


class ROIHeads:
    """Matching / sampling logic of the reference's ROIHeads (roi.py:15-193); the per-region heads themselves are out
    of scope (the reference never wrote them)."""

    def __init__(self, num_classes: int, batch_size_per_image: int, positive_fraction: float,
                 proposal_matcher: Matcher, proposal_append_gt: bool = True):
        self.num_classes = int(num_classes)
        self.batch_size_per_image = int(batch_size_per_image)
        self.positive_fraction = float(positive_fraction)
        self.proposal_matcher = proposal_matcher
        self.proposal_append_gt = bool(proposal_append_gt)
        self.last_num_fg_samples: Optional[float] = None  # what the reference logs (roi.py:189-191)
        self.last_num_bg_samples: Optional[float] = None
        self._ws_cache = {}  # sample_proposals_batched's workspace per (device, stream)

    @classmethod
    def build(cls, conf):
        return cls(num_classes=conf.num_classes, batch_size_per_image=conf.batch_size_per_image,
                   positive_fraction=conf.positive_fraction, proposal_matcher=Matcher.build(conf.proposal_matcher),
                   proposal_append_gt=conf.proposal_append_gt)

    def label_proposals(self, proposal_boxes: torch.Tensor, gt_boxes: torch.Tensor,
                        gt_classes: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Deterministic half for one image: (matched gt index int64[P], matcher label int8[P], class label int64[P])
        with background = num_classes and ignored = -1 (roi.py:157-160 + :84-95)."""
        matched, labels, _, _ = self.proposal_matcher.match_boxes([gt_boxes.reshape(-1, 4)], proposal_boxes)
        matched, labels = matched[0], labels[0]
        if gt_classes.numel() > 0:
            cls = gt_classes.to(torch.int64)[matched]
            cls = torch.where(labels == 0, torch.full_like(cls, self.num_classes), cls)
            cls = torch.where(labels == -1, torch.full_like(cls, -1), cls)
        else:
            cls = torch.zeros_like(matched) + self.num_classes
        return matched, labels, cls

    def _sample_proposals(self, matched_idxs: torch.Tensor, matched_labels: torch.Tensor,
                          gt_classes: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """reference roi.py:68-105: class labels from the matching, then the fg/bg subsample."""
        if gt_classes.numel() > 0:
            cls = gt_classes.to(torch.int64)[matched_idxs]
            cls[matched_labels == 0] = self.num_classes
            cls[matched_labels == -1] = -1
        else:
            cls = torch.zeros_like(matched_idxs) + self.num_classes
        fg, bg = subsample_labels(cls, self.batch_size_per_image, self.positive_fraction, self.num_classes)
        sampled = torch.cat([fg, bg], dim=0)
        return sampled, cls[sampled]

    @staticmethod
    def sample_workspace(n: int, p_stride: int, sum_g: int, device) -> torch.Tensor:
        """Zeroed workspace of det_roi_sample_proposals for these sizes (or any smaller ones): every call leaves it zero,
        so one made before a graph capture serves every replay without a memset.  One per stream of calls in flight."""
        nbytes = N.fn("det_roi_sample_workspace_bytes")(int(n), int(p_stride), int(sum_g))
        return torch.zeros((max(nbytes, 16),), dtype=torch.uint8, device=device)

    def _workspace(self, n, p_stride, sum_g, device) -> torch.Tensor:
        """A cached sample_workspace per (device, stream), grown when a call needs more."""
        key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
        need = N.fn("det_roi_sample_workspace_bytes")(int(n), int(p_stride), int(sum_g))
        ws = self._ws_cache.get(key)
        if ws is None or ws.numel() < need:
            ws = self.sample_workspace(n, p_stride, sum_g, device)
            self._ws_cache[key] = ws
        return ws

    @torch.no_grad()
    def sample_proposals_batched(self, proposal_boxes: torch.Tensor, proposal_counts: torch.Tensor,
                                 gt_table: torch.Tensor, gt_offsets: torch.Tensor, gt_classes: torch.Tensor,
                                 seed: torch.Tensor, out: Optional[Dict[str, torch.Tensor]] = None,
                                 workspace: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """Gt append, matching, class labels and the fg/bg subsample of label_and_sample_proposals for the whole batch
        (det_roi_sample_proposals: two launches, no host synchronisation, CUDA-graph capturable).

        proposal_boxes (N, P, 4) with image b's first proposal_counts[b] rows valid (rpn_proposals_batched /
        proposals_from_heads output; rows past the count are never read); gt_table (sum_G, 4) + int32 gt_offsets (N+1)
        from Matcher.pack_gt; gt_classes (sum_G) int64; seed: device int64 (1,) read by the kernel -- advance it (e.g.
        ``seed.add_(1)`` in the captured graph) to draw new samples.  Same counts and distribution as the reference's
        subsample_labels; the samples are the per-candidate hash keys' smallest, not torch.randperm's.

        Returns a dict of padded (N, S) rows, S = batch_size_per_image, foreground rows first, then background, each in
        candidate order (the proposals, then the appended gt boxes): ``boxes`` (N,S,4), ``gt_classes`` int64,
        ``gt_boxes`` (N,S,4), ``matched`` int32 (index into the image's gt, -1 without gt), ``src`` int32 (candidate
        index); ``count`` / ``num_fg`` (N) int32 and ``underfull`` (1) int32 (1 iff some image has count < S).  Rows
        past the count: src = gt_classes = matched = -1, zero boxes.  ``out``: a previous result to write into.
        ``workspace``: a sample_workspace large enough for these sizes (default: one cached per stream)."""
        N.require_cuda(proposal_boxes, proposal_counts, gt_table, gt_offsets, gt_classes, seed)
        dev = proposal_boxes.device
        pb = N.f32c(proposal_boxes.reshape(proposal_boxes.shape[0], -1, 4))
        n, p_stride = pb.shape[0], pb.shape[1]
        gt = N.f32c(gt_table.reshape(-1, 4))
        sum_g = gt.shape[0]
        counts = proposal_counts.to(torch.int32).contiguous()
        offsets = gt_offsets.to(torch.int32).contiguous()
        classes = gt_classes.to(torch.int64).contiguous()
        assert seed.dtype == torch.int64 and seed.numel() == 1
        S = self.batch_size_per_image
        if out is None:
            out = {"boxes": torch.empty((n, S, 4), dtype=torch.float32, device=dev),
                   "gt_classes": torch.empty((n, S), dtype=torch.int64, device=dev),
                   "gt_boxes": torch.empty((n, S, 4), dtype=torch.float32, device=dev),
                   "matched": torch.empty((n, S), dtype=torch.int32, device=dev),
                   "src": torch.empty((n, S), dtype=torch.int32, device=dev),
                   "count": torch.empty((n,), dtype=torch.int32, device=dev),
                   "num_fg": torch.empty((n,), dtype=torch.int32, device=dev),
                   "underfull": torch.empty((1,), dtype=torch.int32, device=dev)}
        if workspace is None:
            workspace = self._workspace(n, p_stride, sum_g, dev)
        m = self.proposal_matcher
        thr, lab = _rule_arrays(m._inner, m.labels)
        with torch.cuda.device(dev):
            N.call("det_roi_sample_proposals", N.ptr(pb) if p_stride else None, N.ptr(counts), n, p_stride,
                   N.ptr(gt) if sum_g else None, N.ptr(offsets), N.ptr(classes) if sum_g else None, sum_g,
                   self.num_classes, thr, lab, len(m._inner), int(m.allow_low_quality_matches), S,
                   self.positive_fraction, int(self.proposal_append_gt), N.ptr(seed), N.ptr(out["boxes"]),
                   N.ptr(out["gt_classes"]), N.ptr(out["gt_boxes"]), N.ptr(out["matched"]), N.ptr(out["src"]),
                   N.ptr(out["count"]), N.ptr(out["num_fg"]), N.ptr(out["underfull"]), N.ptr(workspace),
                   workspace.numel(), N.stream())
        return out

    @torch.no_grad()
    def label_and_sample_proposals_batched(self, proposals: List[Instances], targets: List[Instances],
                                           seed: Optional[int] = None) -> List[Instances]:
        """label_and_sample_proposals on sample_proposals_batched: the same fields -- every proposal field gathered
        after add_ground_truth_to_proposals, gt_classes, and every gt_* target field of the matched gt for images with
        gt -- with foreground rows first, then background, each in candidate order.  One device-to-host read (the
        counts) for the whole batch.  seed=None draws one integer from torch's default CPU generator, so
        torch.manual_seed makes the call reproducible."""
        if not proposals:
            return []
        if seed is None:
            seed = int(torch.randint(-(1 << 63), (1 << 63) - 1, (1,), dtype=torch.int64))
        boxes = [p.proposal_boxes.tensor if isinstance(p.proposal_boxes, Boxes) else p.proposal_boxes
                 for p in proposals]
        gt_boxes = [t.gt_boxes.tensor if isinstance(t.gt_boxes, Boxes) else t.gt_boxes for t in targets]
        dev = boxes[0].device
        n, p_stride = len(boxes), max(int(b.shape[0]) for b in boxes)
        padded = torch.zeros((n, p_stride, 4), dtype=torch.float32, device=dev)
        for i, b in enumerate(boxes):
            padded[i, :b.shape[0]] = b
        counts = torch.tensor([int(b.shape[0]) for b in boxes], dtype=torch.int32).to(dev, non_blocking=True)
        table, offsets = Matcher.pack_gt(gt_boxes, dev)
        classes = (torch.cat([t.gt_classes.reshape(-1) for t in targets]).to(dev, torch.int64) if targets
                   else torch.zeros((0,), dtype=torch.int64, device=dev))
        seed_t = torch.tensor([seed], dtype=torch.int64).to(dev, non_blocking=True)
        res = self.sample_proposals_batched(padded, counts, table, offsets, classes, seed_t)
        if self.proposal_append_gt:
            proposals = add_ground_truth_to_proposals([t.gt_boxes for t in targets], proposals)
        cnt, nfg = torch.stack([res["count"], res["num_fg"]]).cpu().tolist()  # the one read-back
        out = []
        for i, (props, tgt) in enumerate(zip(proposals, targets)):
            src = res["src"][i, :cnt[i]].long()
            props = props[src]
            props.gt_classes = res["gt_classes"][i, :cnt[i]]
            if len(tgt) > 0:
                rows = res["matched"][i, :cnt[i]].long()
                for name, value in tgt.get_fields().items():
                    if name.startswith("gt_") and not props.has(name):
                        props.set(name, value[rows])
            out.append(props)
        self.last_num_fg_samples = sum(nfg) / n
        self.last_num_bg_samples = sum(c - f for c, f in zip(cnt, nfg)) / n
        return out

    @torch.no_grad()
    def label_and_sample_proposals(self, proposals: List[Instances], targets: List[Instances]) -> List[Instances]:
        """reference roi.py:107-193: optional gt append, per image IoU -> Matcher -> sample, copy the gt_* fields of
        the matched targets onto the sampled proposals."""
        gt_boxes = [t.gt_boxes for t in targets]
        if self.proposal_append_gt:
            proposals = add_ground_truth_to_proposals(gt_boxes, proposals)
        out, num_fg, num_bg = [], [], []
        for props, tgt in zip(proposals, targets):
            has_gt = len(tgt) > 0
            gtb = tgt.gt_boxes.tensor if isinstance(tgt.gt_boxes, Boxes) else tgt.gt_boxes
            pb = props.proposal_boxes.tensor if isinstance(props.proposal_boxes, Boxes) else props.proposal_boxes
            matched, labels, _, _ = self.proposal_matcher.match_boxes([gtb.reshape(-1, 4)], pb)
            sampled, cls = self._sample_proposals(matched[0], labels[0], tgt.gt_classes)
            props = props[sampled]
            props.gt_classes = cls
            if has_gt:
                sampled_targets = matched[0][sampled]
                for name, value in tgt.get_fields().items():
                    if name.startswith("gt_") and not props.has(name):
                        props.set(name, value[sampled_targets])
            num_bg.append(int((cls == self.num_classes).sum()))
            num_fg.append(cls.numel() - num_bg[-1])
            out.append(props)
        if out:
            self.last_num_fg_samples = sum(num_fg) / len(num_fg)
            self.last_num_bg_samples = sum(num_bg) / len(num_bg)
        return out
