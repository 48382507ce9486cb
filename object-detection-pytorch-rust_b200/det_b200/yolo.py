"""YOLO-style grid / dense anchor heads: decode + score threshold + per-class NMS.

The reference has no such head (SURVEY.md section 8 row a15); the specification is this repository's own
(oracle/ref_torch.py: yolo_decode, yolo_select_nms, dense_decode) -- parity is pinned by that oracle only.
Arithmetic: det_yolo_decode_nms (csrc/yolo.cu), det_dense_decode / det_dense_detect (csrc/dense_decode.cu) +
det_nms_batched.
"""
import ctypes
import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _native as N
from .matcher import Matcher
from .nms import nms_images, MODE_AUTO, detect_unfused, detect_workspace, detection_buffers

_DEFAULT_SCALE_CLAMP = math.log(1000.0 / 16)


class YoloGridHead:
    """S x S x (B*5+C) channels-last grid head (YOLOv1 geometry, sigmoid/exp parameterisation)."""

    def __init__(self, grid: int = 7, num_boxes: int = 2, num_classes: int = 20, image_size: Tuple[int, int] = (448, 448),
                 priors: Optional[Sequence[Sequence[float]]] = None, scale_clamp: float = _DEFAULT_SCALE_CLAMP,
                 clip: bool = True):
        self.S, self.B, self.C = int(grid), int(num_boxes), int(num_classes)
        self.image_size = (int(image_size[0]), int(image_size[1]))
        if priors is None:  # one cell and three cells wide, square
            cw, chh = self.image_size[1] / self.S, self.image_size[0] / self.S
            priors = [[cw * (1 + 2 * i), chh * (1 + 2 * i)] for i in range(self.B)]
        self.priors = torch.tensor(priors, dtype=torch.float32).reshape(self.B, 2)
        self.scale_clamp = float(scale_clamp)
        self.clip = bool(clip)
        self._dev_priors = {}

    @property
    def num_predictors(self) -> int:
        return self.S * self.S * self.B

    def priors_on(self, device) -> torch.Tensor:
        k = str(device)
        if k not in self._dev_priors:
            self._dev_priors[k] = self.priors.to(device).contiguous()
        return self._dev_priors[k]

    def detect(self, head: torch.Tensor, score_thresh: float = 0.25, iou_thresh: float = 0.5,
               max_det: Optional[int] = None, return_dense: bool = False, mode: int = MODE_AUTO, out=None,
               index_dtype: torch.dtype = torch.int64):
        """head (N,S,S,B*5+C) -> dict(flat (N,K) int64 = predictor*C+class, boxes (N,K,4), scores (N,K),
        count (N) int32) with K = max_det padding, by descending score; one launch, no host synchronisation.
        With return_dense the decoded boxes/conf/scores of every predictor are written too.
        `out` may carry a dict returned by an earlier call with the same shapes to reuse its buffers.
        index_dtype=torch.int32 writes the same `flat` values as 32-bit integers (det_yolo_decode_nms_i32).
        A bf16 / fp16 head is read as it is (det_yolo_decode_nms_typed): the results are bit-identical to head.float()."""
        N.require_cuda(head)
        (h,), code = N.heads_c([head])
        n = h.shape[0]
        assert tuple(h.shape[1:]) == (self.S, self.S, self.B * 5 + self.C), h.shape
        P, C = self.num_predictors, self.C
        max_det = P * C if max_det is None else int(max_det)
        dev = h.device
        if out is None:
            out = {"flat": torch.empty((n, max_det), dtype=index_dtype, device=dev),
                   "boxes": torch.empty((n, max_det, 4), dtype=torch.float32, device=dev),
                   "scores": torch.empty((n, max_det), dtype=torch.float32, device=dev),
                   "count": torch.empty((n,), dtype=torch.int32, device=dev), "num_classes": C}
            if return_dense:
                out.update(dense_boxes=torch.empty((n, P, 4), dtype=torch.float32, device=dev),
                           dense_conf=torch.empty((n, P), dtype=torch.float32, device=dev),
                           dense_scores=torch.empty((n, P, C), dtype=torch.float32, device=dev))
        assert out["flat"].dtype in (torch.int64, torch.int32)
        if n:
            with torch.cuda.device(dev):
                N.call("det_yolo_decode_nms_typed", N.ptr(h), code, n, self.S, self.B, C, self.image_size[0],
                       self.image_size[1], N.ptr(self.priors_on(dev)), self.scale_clamp, int(self.clip),
                       float(score_thresh), float(iou_thresh), int(mode), N.ptr(out.get("dense_boxes")),
                       N.ptr(out.get("dense_conf")), N.ptr(out.get("dense_scores")), max_det, N.ptr(out["flat"]),
                       out["flat"].element_size(), N.ptr(out["boxes"]), N.ptr(out["scores"]), N.ptr(out["count"]),
                       N.stream())
        return out

    def decode(self, head: torch.Tensor):
        """Dense decode only: boxes (N,P,4), conf (N,P), scores (N,P,C)."""
        r = self.detect(head, score_thresh=float("inf"), max_det=1, return_dense=True)
        return r["dense_boxes"], r["dense_conf"], r["dense_scores"]


class YoloHostPipeline:
    """Serving loop for host-resident head tensors: `depth` slots, each with pinned host input / output buffers, device
    buffers, its own stream and a CUDA graph [H2D copy -> det_yolo_decode_nms -> D2H copy].  Slots run on different
    streams, so the upload of batch i+1, the kernel of batch i and the download of batch i-1 overlap (separate copy
    engines per direction).  The producer writes a batch into ``input(slot)`` (pinned), calls ``launch(slot)`` and
    later ``wait(slot)`` -> dict of pinned host views (flat, boxes, scores, count).  No per-step allocation.
    input_dtype torch.bfloat16 / torch.float16: the host and device inputs are 16-bit and the kernel reads them as they
    are -- half the upload bytes, results bit-identical to the fp32 head holding the same values."""

    def __init__(self, head: "YoloGridHead", batch: int, score_thresh: float = 0.25, iou_thresh: float = 0.5,
                 max_det: int = 300, depth: int = 3, device=None, mode: int = MODE_AUTO, use_graph: bool = True,
                 index_dtype: torch.dtype = torch.int64, input_dtype: torch.dtype = torch.float32):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.head, self.batch, self.depth, self.device = head, int(batch), int(depth), dev
        self.args = (float(score_thresh), float(iou_thresh), int(max_det), int(mode))
        shape = (self.batch, head.S, head.S, head.B * 5 + head.C)
        k = int(max_det)
        assert index_dtype in (torch.int64, torch.int32)
        assert input_dtype in N.DTYPE_CODES, f"input_dtype must be one of {list(N.DTYPE_CODES)}"
        self.index_dtype = index_dtype  # int32: the same indices, 4 bytes less per detection on the PCIe download
        isz = 8 if index_dtype == torch.int64 else 4
        # one output blob per slot so the download is a single copy: [flat i64/i32 | boxes f32x4 | scores f32 | count i32]
        self._sizes = (self.batch * k * isz, self.batch * k * 16, self.batch * k * 4, self.batch * 4)
        nbytes = sum(self._sizes)
        self.h_in = [torch.empty(shape, dtype=input_dtype).pin_memory() for _ in range(depth)]
        self.d_in = [torch.empty(shape, dtype=input_dtype, device=dev) for _ in range(depth)]
        self.d_blob = [torch.empty((nbytes,), dtype=torch.uint8, device=dev) for _ in range(depth)]
        self.h_blob = [torch.empty((nbytes,), dtype=torch.uint8).pin_memory() for _ in range(depth)]
        self.d_out = [self._views(b, k) for b in self.d_blob]
        self.h_out = [self._views(b, k) for b in self.h_blob]
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(depth)]
        self.done = [torch.cuda.Event() for _ in range(depth)]
        self.graphs = [None] * depth
        self.h2d_bytes = self.h_in[0].numel() * self.h_in[0].element_size()
        self.d2h_bytes = nbytes
        if use_graph:
            for s in range(depth):
                with torch.cuda.stream(self.streams[s]):
                    self._enqueue(s)  # warm-up outside capture (function attributes, lazy init)
                self.streams[s].synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.streams[s]):
                    self._enqueue(s)
                self.graphs[s] = g

    def _views(self, blob, k):
        o0, o1, o2, o3 = 0, self._sizes[0], self._sizes[0] + self._sizes[1], self._sizes[0] + self._sizes[1] + self._sizes[2]
        return {"flat": blob[o0:o1].view(self.index_dtype).view(self.batch, k),
                "boxes": blob[o1:o2].view(torch.float32).view(self.batch, k, 4),
                "scores": blob[o2:o3].view(torch.float32).view(self.batch, k),
                "count": blob[o3:].view(torch.int32).view(self.batch), "num_classes": self.head.C}

    def _enqueue(self, s):
        thr, iou, k, mode = self.args
        self.d_in[s].copy_(self.h_in[s], non_blocking=True)
        self.head.detect(self.d_in[s], thr, iou, max_det=k, mode=mode, out=self.d_out[s])
        self.h_blob[s].copy_(self.d_blob[s], non_blocking=True)

    def input(self, slot: int) -> torch.Tensor:
        return self.h_in[slot]

    def launch(self, slot: int) -> None:
        st = self.streams[slot]
        if self.graphs[slot] is not None:
            with torch.cuda.stream(st):
                self.graphs[slot].replay()
        else:
            with torch.cuda.stream(st):
                self._enqueue(slot)
        self.done[slot].record(st)

    def wait(self, slot: int):
        self.done[slot].synchronize()
        return self.h_out[slot]

    def run(self, host_head: torch.Tensor):
        """Convenience: one batch through slot 0, synchronously."""
        self.h_in[0].copy_(host_head)
        self.launch(0)
        return self.wait(0)


class _FusedYoloLoss(torch.autograd.Function):
    """Everything the backward launch reads is saved with save_for_backward (no state on the owner)."""

    @staticmethod
    def forward(ctx, head, labels, matched, gt_table, gt_offsets, gt_classes, owner, norm):
        sums = owner._run_loss(head, YoloAssignment(labels, matched, gt_table, gt_offsets), gt_classes, norm, None, None)
        ctx.owner, ctx.norm = owner, norm
        ctx.save_for_backward(head, labels, matched, gt_table, gt_offsets, gt_classes)
        return sums

    @staticmethod
    def backward(ctx, grad_sums):
        head, labels, matched, gt_table, gt_offsets, gt_classes = ctx.saved_tensors
        up = grad_sums[:3].contiguous().float()
        gh = torch.empty_like(head)
        ctx.owner._run_loss(head, YoloAssignment(labels, matched, gt_table, gt_offsets), gt_classes, ctx.norm, up, gh)
        return gh, None, None, None, None, None, None, None


class YoloAssignment:
    def __init__(self, labels, matched, gt_table, gt_offsets):
        self.labels, self.matched, self.gt_table, self.gt_offsets = labels, matched, gt_table, gt_offsets


class YoloGridTrainer:
    """Training side of the grid head: IoU target assignment of the S*S*B predictors (the reference's pairwise_iou +
    Matcher machinery on cell-centred prior boxes) and the fused localisation / objectness / class loss with its
    backward (specification: oracle/ref_torch.py yolo_grid_anchors, yolo_loss; no reference implementation)."""

    def __init__(self, head: YoloGridHead, iou_thresholds=(0.3, 0.7), iou_labels=(0, -1, 1),
                 allow_low_quality_matches: bool = True, lambda_coord: float = 5.0, lambda_noobj: float = 0.5):
        self.head = head
        self.matcher = Matcher(list(iou_thresholds), list(iou_labels), allow_low_quality_matches)
        self.lambda_coord, self.lambda_noobj = float(lambda_coord), float(lambda_noobj)
        self._anchors = {}

    def prior_boxes(self, device) -> torch.Tensor:
        """(S*S*B,4) cell-centred prior boxes, order (row,col,b)."""
        k = str(device)
        if k not in self._anchors:
            h = self.head
            H, W = h.image_size
            sx, sy = W / h.S, H / h.S
            cx = ((torch.arange(h.S, dtype=torch.float32) + 0.5) * sx).view(1, h.S, 1).expand(h.S, h.S, h.B)
            cy = ((torch.arange(h.S, dtype=torch.float32) + 0.5) * sy).view(h.S, 1, 1).expand(h.S, h.S, h.B)
            pw = h.priors[:, 0].view(1, 1, -1).expand(h.S, h.S, -1)
            ph = h.priors[:, 1].view(1, 1, -1).expand(h.S, h.S, -1)
            a = torch.stack((cx - 0.5 * pw, cy - 0.5 * ph, cx + 0.5 * pw, cy + 0.5 * ph), dim=-1).reshape(-1, 4)
            self._anchors[k] = a.to(device).contiguous()
        return self._anchors[k]

    def assign(self, gt_boxes: List[torch.Tensor]) -> YoloAssignment:
        dev = gt_boxes[0].device
        matched, labels, table, offsets = self.matcher.match_boxes(list(gt_boxes), self.prior_boxes(dev))
        return YoloAssignment(labels, matched, table, offsets)

    def assign_packed(self, gt_table: torch.Tensor, gt_offsets: torch.Tensor, n: int) -> YoloAssignment:
        matched, labels = self.matcher.match_packed(gt_table, gt_offsets, n, self.prior_boxes(gt_table.device))
        return YoloAssignment(labels, matched, gt_table, gt_offsets)

    def _run_loss(self, head_t, asg, gt_classes, norm, upstream, grad_head, peer=None):
        """One launch: returns sums (8) = [lambda_coord * loc, obj, cls] / norm, #pos, #neg, 0... -- scaled by the
        kernel's last CTA (no memset before, no scaling op after the launch)."""
        h = self.head
        n = head_t.shape[0]
        dev = head_t.device
        self._world_prev = None
        with torch.cuda.device(dev):
            sums = torch.empty((8,), dtype=torch.float32, device=dev)
            args = (N.ptr(head_t), N.ptr(asg.labels), N.ptr(asg.matched), N.ptr(asg.gt_table),
                    N.ptr(gt_classes), N.ptr(asg.gt_offsets), n, h.S, h.B, h.C, h.image_size[0], h.image_size[1],
                    N.ptr(h.priors_on(dev)), self.lambda_coord, self.lambda_noobj, 1.0 / norm,
                    N.ptr(upstream), N.ptr(N.accumulators(dev)), N.ptr(sums), N.ptr(grad_head))
            if peer is None:
                N.call("det_yolo_loss", *args, N.stream())
            else:  # the loss kernel's last CTA publishes the sums to every rank and collects the previous step's
                ctx, prev = peer.fused_ctx()
                N.call("det_yolo_loss_peer", *args, ctypes.byref(ctx), N.stream())
                self._world_prev = prev
        return sums

    def loss(self, head_t: torch.Tensor, asg: YoloAssignment, gt_classes: torch.Tensor,
             normalizer: Optional[float] = None, with_grads: bool = False, peer=None):
        """head (N,S,S,B*5+C) fp32; gt_classes (sum_G,) int64 packed like asg.gt_table.  Returns {"loc_loss",
        "obj_loss","cls_loss","num_pos","num_neg"} (autograd-connected) and, with_grads=True, "grad_head" from the same
        launch (fused forward+backward).  peer (det_b200.dist.PeerSums, with_grads only): the same launch also publishes
        the sums to every rank over NVLink peer memory and returns "world_sums_prev", the all-rank sum of the PREVIOUS
        step's scaled sums (None on the first step) -- compute + collective in one kernel, no NCCL call."""
        N.require_cuda(head_t, gt_classes)
        ht = head_t.contiguous()
        assert ht.dtype == torch.float32
        gc = gt_classes.to(torch.int64).contiguous()
        norm = float(ht.shape[0] if normalizer is None else normalizer)
        assert peer is None or with_grads, "the fused all-reduce rides on the fused forward+backward launch (with_grads=True)"
        if with_grads:
            gh = torch.empty_like(ht)
            sums = self._run_loss(ht.detach(), asg, gc, norm, None, gh, peer)
        else:
            sums = _FusedYoloLoss.apply(ht, asg.labels, asg.matched, asg.gt_table, asg.gt_offsets, gc, self, norm)
        out = {"loc_loss": sums[0], "obj_loss": sums[1], "cls_loss": sums[2], "num_pos": sums[3].detach(),
               "num_neg": sums[4].detach(), "sums": sums}
        if with_grads:
            out["grad_head"] = gh
            if peer is not None:
                prev = self._world_prev
                out["world_sums_prev"] = prev  # already the world sum of the previous step's reported (scaled) sums
        return out


class DenseAnchorHead:
    """Multi-level dense anchor head in the conv layout (N, A*(5+C), Hl, Wl) per level (YOLOv3-style decode)."""

    def __init__(self, strides: Sequence[int], anchors_wh: Sequence[Sequence[Sequence[float]]], num_classes: int,
                 scale_clamp: float = _DEFAULT_SCALE_CLAMP):
        self.strides = [int(s) for s in strides]
        self.anchors = [torch.tensor(a, dtype=torch.float32).reshape(-1, 2) for a in anchors_wh]
        assert len(self.anchors) == len(self.strides)
        self.C = int(num_classes)
        self.scale_clamp = float(scale_clamp)
        self._dev = {}

    def _anchors_on(self, device):
        k = str(device)
        if k not in self._dev:
            self._dev[k] = [a.to(device).contiguous() for a in self.anchors]
        return self._dev[k]

    def decode(self, heads: List[torch.Tensor], out=None):
        """-> boxes (N,R,4), scores (N,R), classes (N,R) int64 with all levels concatenated, order (level,h,w,a).
        bf16 / fp16 heads (all levels one dtype) are read as they are: bit-identical to the fp32 heads h.float()."""
        N.require_cuda(*heads)
        dev = heads[0].device
        n = heads[0].shape[0]
        sizes = [h.shape[2] * h.shape[3] * a.shape[0] for h, a in zip(heads, self.anchors)]
        R = sum(sizes)
        if out is None:
            out = (torch.empty((n, R, 4), dtype=torch.float32, device=dev),
                   torch.empty((n, R), dtype=torch.float32, device=dev),
                   torch.empty((n, R), dtype=torch.int64, device=dev))
        boxes, scores, classes = out
        anchors = self._anchors_on(dev)
        hcs, code = N.heads_c(heads)
        na = anchors[0].shape[0]
        if all(a.shape[0] == na for a in anchors):  # one persistent launch for the whole pyramid
            lv = self._level_array(hcs, anchors, na)
            with torch.cuda.device(dev):
                N.call("det_dense_decode_typed", ctypes.cast(lv, ctypes.c_void_p), len(hcs), n, na, self.C,
                       self.scale_clamp, N.ptr(boxes), N.ptr(scores), N.ptr(classes), R, code, N.stream())
            return boxes, scores, classes
        off = 0
        with torch.cuda.device(dev):
            for hc, a, s, sz in zip(hcs, anchors, self.strides, sizes):
                assert hc.shape[1] == a.shape[0] * (5 + self.C), hc.shape
                lv = N.DenseLevel(hc.data_ptr(), a.data_ptr(), hc.shape[2], hc.shape[3], s, 0, off)
                N.call("det_dense_decode_typed", ctypes.byref(lv), 1, n, a.shape[0], self.C, self.scale_clamp,
                       N.ptr(boxes), N.ptr(scores), N.ptr(classes), R, code, N.stream())
                off += sz
        return boxes, scores, classes

    def _level_array(self, hcs, anchors, na):
        """det_dense_level_t array over prepared heads that share the anchor count `na`."""
        lv = (N.DenseLevel * len(hcs))()
        off = 0
        for i, (hc, a, s) in enumerate(zip(hcs, anchors, self.strides)):
            assert hc.shape[1] == na * (5 + self.C), hc.shape
            lv[i].head, lv[i].anchors_wh = hc.data_ptr(), a.data_ptr()
            lv[i].h, lv[i].w, lv[i].stride, lv[i].reserved, lv[i].out_offset = hc.shape[2], hc.shape[3], s, 0, off
            off += hc.shape[2] * hc.shape[3] * na
        return lv

    def _levels(self, heads: List[torch.Tensor]):
        """(det_dense_level_t array, contiguous heads, n, A, R) for heads that share the anchor count; bf16 / fp16 heads
        are kept as they are (N.heads_c): the DET_DTYPE_* code is N.DTYPE_CODES[hcs[0].dtype]."""
        dev = heads[0].device
        anchors = self._anchors_on(dev)
        hcs, _ = N.heads_c(heads)
        na = anchors[0].shape[0]
        assert all(a.shape[0] == na for a in anchors), "levels must share the anchor count"
        lv = self._level_array(hcs, anchors, na)
        return lv, hcs, heads[0].shape[0], na, sum(h.shape[2] * h.shape[3] * na for h in hcs)

    def fused_ok(self, heads: List[torch.Tensor]) -> bool:
        """det_dense_detect's documented limits: equal anchor counts, every level h*w % 4 == 0."""
        na = self.anchors[0].shape[0]
        return all(a.shape[0] == na for a in self.anchors) and all((h.shape[2] * h.shape[3]) % 4 == 0 for h in heads)

    def detect_thresholded(self, heads: List[torch.Tensor], score_thresh: float, iou_thresh: float = 0.5,
                           max_det: int = 300, cand_cap: int = 1024, gate: bool = True, mode: int = MODE_AUTO,
                           check: bool = True, out=None, workspace: Optional[torch.Tensor] = None):
        """The detector's inference path: decode -> score > score_thresh -> per-class NMS -> top max_det
        (oracle/ref_torch.py dense_select_nms over dense_decode).  Two launches for the batch (det_dense_detect);
        nothing dense is written.  Returns a dict: idx (N,max_det) int64 rows in decode() order, boxes, scores,
        classes int64, count (N) int32 (rows past count are undefined).

        cand_cap (<= 4096) bounds the per-image candidate list.  With check=True (one 4-byte read-back) an image that
        overflows it -- or a pyramid outside det_dense_detect's limits -- is redone exactly by the unfused GPU path
        (decode + det_nms_batched); with check=False overflowing images carry count = -1 and `overflow` is set.
        bf16 / fp16 heads (all levels one dtype) are read as they are, on both routes: bit-identical to h.float()."""
        N.require_cuda(*heads)
        dev = heads[0].device
        n = heads[0].shape[0]
        max_det = int(max_det)
        if not self.fused_ok(heads) or cand_cap > 4096:
            return self._detect_thresholded_unfused(heads, score_thresh, iou_thresh, max_det, mode)
        if out is None:
            out = detection_buffers(n, max_det, dev)
        if n == 0:
            return out
        lv, hcs, _, na, _ = self._levels(heads)
        code = N.DTYPE_CODES[hcs[0].dtype]
        workspace, wsb, zeroed = detect_workspace(workspace, n, int(cand_cap), dev)
        flags = (1 if gate else 0) | zeroed
        with torch.cuda.device(dev):
            N.call("det_dense_detect_typed", ctypes.cast(lv, ctypes.c_void_p), len(hcs), n, na, self.C,
                   self.scale_clamp, float(score_thresh), float(iou_thresh), int(mode), flags, int(cand_cap), max_det,
                   N.ptr(out["idx"]), N.ptr(out["boxes"]), N.ptr(out["scores"]), N.ptr(out["classes"]),
                   N.ptr(out["count"]), N.ptr(out["overflow"]), N.ptr(workspace), wsb, code, N.stream())
        if check and int(out["overflow"].item()) != 0:
            return self._detect_thresholded_unfused(heads, score_thresh, iou_thresh, max_det, mode)
        return out

    def _detect_thresholded_unfused(self, heads, score_thresh, iou_thresh, max_det, mode):
        """Same contract through det_dense_decode -> nms.detect_unfused: any candidate count up to 131071 per image,
        library kernels only, no host sync."""
        boxes, scores, classes = self.decode(heads)
        return detect_unfused(boxes, scores, classes, score_thresh, iou_thresh, max_det, mode)

    def detect(self, heads: List[torch.Tensor], iou_thresh: float = 0.5, max_det: Optional[int] = None,
               mode: int = MODE_AUTO):
        """decode + per-class NMS over all R boxes of every image: (boxes, scores, classes, keep (N,max_det),
        keep_counts (N))."""
        boxes, scores, classes = self.decode(heads)
        keep, cnt = nms_images(boxes, scores, classes, None, iou_thresh, max_det, mode)
        return boxes, scores, classes, keep, cnt
