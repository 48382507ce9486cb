"""GPU parity: FPN level assignment + ROIAlign over a pyramid (reference python/src/models/modules/roi_poolers.py;
SURVEY.md section 8f rank 2).  Oracle: the installed torchvision CPU roi_align (third-party arithmetic the reference
calls at roi_poolers.py:64) driven by a restatement of the reference's per-level loop (roi_poolers.py:269-331)."""
import math

import pytest
import torch
import torchvision

from tests.util import gen, rand_boxes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


def ref_levels(boxes, min_level, max_level, canonical_box_size=224, canonical_level=4):
    """reference assign_boxes_to_levels (roi_poolers.py:121-131) on CPU tensors"""
    area = (boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1])
    lv = torch.floor(canonical_level + torch.log2(torch.sqrt(area) / canonical_box_size + 1e-8))
    return torch.clamp(lv, min=min_level, max=max_level).to(torch.int64) - min_level


def ref_pooler(feats, scales, box_lists, out_size, sampling_ratio, aligned, min_level, max_level):
    """reference ROIPooler.forward (roi_poolers.py:269-331) with torchvision's CPU roi_align"""
    rois = torch.cat([torch.cat((torch.full_like(b[:, :1], i), b), 1) for i, b in enumerate(box_lists)], 0)
    if len(feats) == 1:
        return torchvision.ops.roi_align(feats[0], rois, out_size, scales[0], sampling_ratio, aligned)
    lv = ref_levels(torch.cat(box_lists, 0), min_level, max_level)
    out = torch.zeros((rois.shape[0], feats[0].shape[1]) + tuple(out_size))
    for l, (f, s) in enumerate(zip(feats, scales)):
        inds = torch.nonzero(lv == l, as_tuple=True)[0]
        out.index_put_((inds,), torchvision.ops.roi_align(f, rois[inds], out_size, s, sampling_ratio, aligned))
    return out


def _boxes(n_img, per_img, g, frame=448.0):
    out = []
    for i in range(n_img):
        m = per_img + 7 * i
        sz = torch.exp(torch.rand(m, generator=g) * math.log(400.0 / 6.0)) * 6.0       # sizes 6 .. 400 px: every level
        ar = torch.exp((torch.rand(m, generator=g) - 0.5) * 1.6)
        w, h = sz * torch.sqrt(ar), sz / torch.sqrt(ar)
        cx, cy = torch.rand(m, generator=g) * frame, torch.rand(m, generator=g) * frame
        out.append(torch.stack((cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2), 1))   # partly outside the image
    return out


def test_assign_boxes_to_levels_bit_exact(det):
    g = gen(3)
    box_lists = _boxes(3, 400, g)
    box_lists[0][0] = torch.tensor([0.0, 0.0, 224.0, 224.0])     # canonical size: exactly level 4
    box_lists[0][1] = torch.tensor([0.0, 0.0, 448.0, 448.0])     # exactly one level up
    box_lists[0][2] = torch.tensor([5.0, 5.0, 5.0, 9.0])         # empty box: clamped to the lowest level
    got = det.assign_boxes_to_levels([det.Boxes(b.cuda()) for b in box_lists], 2, 5, 224, 4)
    want = ref_levels(torch.cat(box_lists, 0), 2, 5)
    assert torch.equal(got.cpu(), want)
    assert set(want.tolist()) == {0, 1, 2, 3}


@pytest.mark.parametrize("ptype,sampling_ratio,out_size", [("ROIAlignV2", 0, (7, 7)), ("ROIAlignV2", 2, (7, 7)),
                                                           ("ROIAlign", 0, (7, 7)), ("ROIAlign", 3, (5, 9)),
                                                           ("ROIAlignV2", 0, (14, 14))])
def test_roi_pooler_pyramid_matches_torchvision_cpu(det, ptype, sampling_ratio, out_size):
    """reference default: features p1..p4 (strides 4..32), ROIAlignV2, sampling_ratio 0, 7x7 (config/roi.py:24-50)."""
    g = gen(11)
    n_img, C = 3, 24
    strides = [4, 8, 16, 32]
    feats = [torch.randn(n_img, C, 448 // s, 448 // s, generator=g) for s in strides]
    scales = [1.0 / s for s in strides]
    box_lists = _boxes(n_img, 60, g)
    pooler = det.ROIPooler(scales, sampling_ratio, out_size, ptype)
    assert (pooler.min_level, pooler.max_level) == (2, 5)
    got = pooler([f.cuda() for f in feats], [det.Boxes(b.cuda()) for b in box_lists])
    want = ref_pooler(feats, scales, box_lists, out_size, sampling_ratio, ptype == "ROIAlignV2", 2, 5)
    assert got.shape == want.shape
    torch.testing.assert_close(got.cpu(), want, rtol=1e-5, atol=1e-5)


def test_roi_align_single_level_and_edges(det):
    g = gen(12)
    feat = torch.randn(2, 8, 20, 30, generator=g)
    rois = torch.tensor([[0, 4.0, 4.0, 60.0, 40.0],
                         [1, -30.0, -20.0, 10.0, 12.0],      # mostly outside: out-of-range samples contribute 0
                         [1, 100.0, 70.0, 130.0, 90.0],      # beyond the right/bottom border
                         [0, 15.0, 15.0, 15.0, 15.0],        # empty box
                         [1, 0.0, 0.0, 119.9, 79.9]])        # the whole map
    for aligned in (True, False):
        ra = det.ROIAlign((7, 7), 0.25, 0, aligned)
        got = ra(feat.cuda(), rois.cuda())
        want = torchvision.ops.roi_align(feat, rois, (7, 7), 0.25, 0, aligned)
        torch.testing.assert_close(got.cpu(), want, rtol=1e-5, atol=1e-5)
    empty = det.ROIPooler([0.25], 0, 7, "ROIAlignV2")([feat.cuda()], [det.Boxes(torch.zeros(0, 4).cuda())] * 2)
    assert empty.shape == (0, 8, 7, 7)
    with pytest.raises(ValueError):
        det.ROIPooler([0.25], 0, 7, "Bilinear")


def test_roi_align_single_roi(det):
    """One roi: rois[:, 1:5] is then a contiguous view that starts 4 bytes into the row; the boxes handed to the kernel
    must still be 16-byte aligned."""
    g = gen(13)
    feat = torch.randn(1, 5, 16, 16, generator=g)
    rois = torch.tensor([[0, 3.0, 2.0, 40.0, 50.0]])
    ra = det.ROIAlign((3, 4), 0.25, 0, True)
    got = ra(feat.cuda(), rois.cuda())
    torch.testing.assert_close(got.cpu(), torchvision.ops.roi_align(feat, rois, (3, 4), 0.25, 0, True), rtol=1e-5,
                               atol=1e-5)


@pytest.mark.parametrize("ptype,sampling_ratio", [("ROIAlignV2", 0), ("ROIAlign", 2)])
def test_roi_pooler_backward_matches_torchvision_cpu(det, ptype, sampling_ratio):
    """Gradients w.r.t. every pyramid level against autograd through torchvision's CPU roi_align (atomics: 1e-5)."""
    g = gen(21)
    n_img, C = 2, 10
    strides = [4, 8, 16, 32]
    feats = [torch.randn(n_img, C, 224 // s, 224 // s, generator=g) for s in strides]
    scales = [1.0 / s for s in strides]
    box_lists = _boxes(n_img, 40, g, frame=224.0)
    weight = torch.randn(sum(b.shape[0] for b in box_lists), C, 7, 7, generator=g)
    cpu_feats = [f.clone().requires_grad_(True) for f in feats]
    want = ref_pooler(cpu_feats, scales, box_lists, (7, 7), sampling_ratio, ptype == "ROIAlignV2", 2, 5)
    (want * weight).sum().backward()
    gpu_feats = [f.cuda().requires_grad_(True) for f in feats]
    pooler = det.ROIPooler(scales, sampling_ratio, 7, ptype)
    got = pooler(gpu_feats, [det.Boxes(b.cuda()) for b in box_lists])
    (got * weight.cuda()).sum().backward()
    torch.testing.assert_close(got.detach().cpu(), want.detach(), rtol=1e-5, atol=1e-5)
    for gf, cf in zip(gpu_feats, cpu_feats):
        assert gf.grad is not None
        torch.testing.assert_close(gf.grad.cpu(), cf.grad, rtol=1e-4, atol=1e-5)
