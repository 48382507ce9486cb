"""The fused YOLO kernel's pair filter (csrc/yolo_fast.cuh pair_may_suppress): one conservative test per predictor pair in
the unshifted frame must let through every pair that suppresses in ANY class's frame.  Under torchvision's offset trick
(<= 1000 candidates) class c's boxes are shifted by c * span in fp32, and that rounding moves a pair's IoU; a filter
that used the plain unshifted decision would drop the pairs that only suppress once shifted.

The pairs here are aimed to land on opposite sides of the threshold in the two frames, in both directions, for high
classes (the largest shifts); a census on the kernel's own decoded boxes asserts that such pairs are present before the
kept ids are compared with the oracle bit for bit."""
import math

import numpy as np
import pytest
import torch

from tests.test_gpu_nms_knife_edge import F32, ovr32, ulp_step
from tests.util import gen

pytestmark = pytest.mark.gpu

SPAN = F32(449.0)   # largest coordinate 448 (a clipped box reaches the image's edge) + 1
ACTIVE = [(r, c) for r in (2, 3, 4) for c in (2, 3, 4)]   # no box of these cells is clipped


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


def _decide(a, b, cls, thr):
    """(unshifted, shifted) suppression decisions of the pairs (a[k], b[k]) of class cls[k]."""
    off = (np.asarray(cls, dtype=F32) * SPAN)[:, None]
    return (ovr32(a, b).astype(np.float64) > thr), (ovr32(a + off, b + off).astype(np.float64) > thr)


def _cpu_boxes(row, col, tw, th, prior):
    """torch's fp32 decode of predictor boxes with tx = ty = 0 (centre of the cell), clipped to 448 x 448."""
    cx, cy = (0.5 + col) * 64.0, (0.5 + row) * 64.0
    w, h = torch.exp(tw) * prior, torch.exp(th) * prior
    b = torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], -1).clamp(0.0, 448.0)
    return b.numpy()


def _flip_logits(thr, row, col, cls, want, salt, u):
    """(tw, th) of predictor 0 of cell (row, col) within 30 ulps of real IoU thr with predictor 1 (logits u), chosen so
    that the unshifted and class-`cls` decisions differ: want 'up' (suppresses only when shifted) or 'down'."""
    t0 = F32(math.log(3 * math.sqrt(thr)) + 0.5 * (u[0] + u[1]))
    tw, th = np.meshgrid(ulp_step(t0, np.arange(-30, 31)), ulp_step(t0, np.arange(-30, 31)))
    tw, th = torch.from_numpy(tw.reshape(-1)), torch.from_numpy(th.reshape(-1))
    b0 = _cpu_boxes(row, col, tw, th, 64.0)
    ut = torch.tensor(u, dtype=torch.float32)
    b1 = np.repeat(_cpu_boxes(row, col, ut[0:1], ut[1:2], 192.0), b0.shape[0], 0)
    plain, shifted = _decide(b1, b0, np.full(b0.shape[0], cls), thr)
    hit = np.nonzero((shifted & ~plain) if want == "up" else (plain & ~shifted))[0]
    if hit.size == 0:
        hit = np.arange(b0.shape[0])
    j = hit[salt % hit.size]
    return float(tw[j]), float(th[j])


def _flip_head(n, C, classes, thr, seed):
    """n images: the nine ACTIVE cells carry an aimed pair each, in distinct classes drawn from `classes`; predictor 1 of
    cell (6, 6) is a class-0 box clipped to the whole image, which fixes the largest coordinate at 448."""
    rng = np.random.default_rng(seed)
    head = torch.full((n, 7, 7, 10 + C), -10.0)
    head[..., 0:2] = 0.0
    head[..., 5:7] = 0.0
    head[..., 2:4] = 0.0
    head[..., 7:9] = 0.0
    head[:, 6, 6, 7:9] = 2.0
    head[:, 6, 6, 9] = 4.0
    head[:, 6, 6, 10] = 4.0
    cls_of = np.zeros((n, 7, 7), dtype=np.int64)
    k = 0
    for i in range(n):
        for (r, c), cls in zip(ACTIVE, rng.permutation(classes)[:len(ACTIVE)]):
            u = [float(F32(v)) for v in rng.uniform(-0.1, 0.1, 2)]
            tw, th = _flip_logits(thr, r, c, int(cls), ("up", "down")[k % 2], k, u)
            k += 1
            head[i, r, c, 2], head[i, r, c, 3] = tw, th
            head[i, r, c, 7], head[i, r, c, 8] = u[0], u[1]
            head[i, r, c, 4] = 3.0 + float(rng.uniform(0, 1))
            head[i, r, c, 9] = 3.0 + float(rng.uniform(0, 1))
            head[i, r, c, 10 + int(cls)] = 4.0
            cls_of[i, r, c] = cls
    return head, cls_of


@pytest.mark.parametrize("C,classes", [(20, range(11, 20)), (32, range(23, 32))])
@pytest.mark.parametrize("thr", [0.5, 0.7, 0.3])
def test_yolo_pair_filter_frame_flips(det, C, classes, thr):
    """C = 20: the kernel specialised for the 7 x 7 x 30 head; C = 32: the generic instantiation (classes up to 31)."""
    from oracle import ref_torch as R
    n = 24
    yh = det.YoloGridHead(7, 2, C, (448, 448))
    head, cls_of = _flip_head(n, C, list(classes), thr, seed=C * 10 + int(thr * 10))
    r = yh.detect(head.cuda(), 0.25, thr, return_dense=True)
    gb, gs = r["dense_boxes"].cpu(), r["dense_scores"].cpu()
    bx = gb.numpy().reshape(n, 49, 2, 4)
    assert float(gb.max()) == 448.0
    a = np.stack([bx[i, rr * 7 + cc, 0] for i in range(n) for (rr, cc) in ACTIVE])
    b = np.stack([bx[i, rr * 7 + cc, 1] for i in range(n) for (rr, cc) in ACTIVE])
    cls = np.array([cls_of[i, rr, cc] for i in range(n) for (rr, cc) in ACTIVE])
    plain, shifted = _decide(b, a, cls, thr)
    up, down = int((shifted & ~plain).sum()), int((plain & ~shifted).sum())
    assert up >= 5 and down >= 5, (up, down)
    for i in range(n):
        assert int((gs[i] > 0.25).sum()) <= 1000   # the offset-trick branch
        want, _, _, _ = R.yolo_select_nms(gb[i], gs[i], 0.25, thr)
        k = int(r["count"][i])
        assert k == want.numel() and torch.equal(r["flat"][i, :k].cpu(), want), i


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_yolo_iou_threshold_zero(det, mode):
    """IoU threshold 0: every overlapping pair of a class suppresses (the filter makes every pair an edge)."""
    from tests.test_gpu_yolo import _check_detect
    from oracle import ref_torch as O
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(6, 7, 7, 30, generator=gen(31))
    _check_detect(det, O, yh, head, 0.25, 0.0, mode=mode)
    _check_detect(det, O, yh, head, 0.02, 0.0, max_det=50, mode=mode)


def test_yolo_nan_box_per_category_branch(det):
    """More than 1000 candidates (per-category branch) and a NaN box among them: the NaN box shares an edge with every
    box and the exact test decides."""
    from tests.test_gpu_yolo import _check_detect
    from oracle import ref_torch as O
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(4, 7, 7, 30, generator=gen(33))
    head[0, 3, 3, 2] = float("nan")   # NaN width of predictor 0 of a cell
    head[1, 2, 5, 8] = float("nan")   # NaN height of predictor 1
    head[2, 0, 0, 0] = float("nan")   # NaN x offset
    head[3, 4, 4, 2:4] = float("nan")
    r = _check_detect(det, O, yh, head, 0.02, 0.5)
    assert int(r["count"].min()) > 0
    assert bool((r["dense_scores"] > 0.02).sum((1, 2)).gt(1000).all())
    assert bool(torch.isnan(r["dense_boxes"]).any((1, 2)).all())
