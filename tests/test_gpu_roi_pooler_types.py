"""ROIPooler(type="ROIPool") and bf16 / fp16 feature pyramids in both poolers.

ROIPool restates torchvision's roi_pool (the reference builds torchvision RoIPools for this type,
python/src/models/modules/roi_poolers.py:224-231); the oracle is the installed CPU kernel driven by a restatement of the
reference's per-level loop (roi_poolers.py:269-331).  Outputs and argmax are compared exactly.

16-bit features follow torchvision's autocast rule: compute in fp32 from the widened input, round the result once to the
input dtype.  So the forward output must be BIT-identical to the GPU fp32 route on [f.float() for f in feats] followed by
.to(dtype); gradients come back in the feature dtype, within one ulp of the fp32 route's gradients cast to it, or within
1e-5 where cancellation makes the atomics' varying order visible (assert_grad_matches_fp32_route).

GPU tests carry their own gpu mark so the CPU tests at the end run without a device."""
import ctypes
import math
import os

import pytest
import torch
import torchvision

from tests.test_gpu_roi_pool import ref_levels
from tests.util import gen

gpu = pytest.mark.gpu
DTYPES = [torch.bfloat16, torch.float16]
DT_IDS = ["bf16", "fp16"]
STRIDES = [4, 8, 16, 32]
FLT_MAX = torch.finfo(torch.float32).max


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


# --------------------------------------------------------------------------------------------------- oracle and inputs
def ref_roi_pool(feats, scales, box_lists, out_size):
    """reference ROIPooler.forward with RoIPool levels (roi_poolers.py:224-231, 269-331) on torchvision's CPU kernel:
    (output, argmax), argmax relative to the box's level plane as torchvision stores it"""
    rois = torch.cat([torch.cat((torch.full_like(b[:, :1], i), b), 1) for i, b in enumerate(box_lists)], 0)
    op = lambda f, r, s: torch.ops.torchvision.roi_pool(f, r, s, out_size[0], out_size[1])
    if len(feats) == 1:
        o, a = op(feats[0], rois, scales[0])
        return o, a.to(torch.int32)
    lv = ref_levels(torch.cat(box_lists, 0), -int(math.log2(scales[0])), -int(math.log2(scales[-1])))
    out = torch.zeros((rois.shape[0], feats[0].shape[1]) + tuple(out_size), dtype=feats[0].dtype)
    arg = torch.full(out.shape, -1, dtype=torch.int32)
    for l, (f, s) in enumerate(zip(feats, scales)):
        inds = torch.nonzero(lv == l, as_tuple=True)[0]
        o, a = op(f, rois[inds], s)
        out = out.index_put((inds,), o)  # out of place: keeps autograd through every level
        arg[inds] = a.to(torch.int32)
    return out, arg


def special_boxes():
    """image-space boxes for a 448 px frame whose pooling is easy to get wrong"""
    return torch.tensor([
        [-60.0, -40.0, 30.0, 50.0],       # partly outside
        [500.0, 470.0, 560.0, 520.0],     # wholly outside, beyond the bottom-right: every bin empty
        [-90.0, -80.0, -20.0, -10.0],     # wholly outside, top-left
        [100.0, 100.0, 100.0, 100.0],     # empty: forced to 1x1
        [200.0, 150.0, 120.0, 90.0],      # inverted: forced to 1x1
        [2.0, 2.0, 2.0, 2.0],             # x * 1/4 = 0.5: round half away from zero takes pixel (1, 1), rintf (0, 0)
        [-2.0, -2.0, 6.0, 10.0],          # -0.5 -> -1, 1.5 -> 2, 2.5 -> 3
        [10.0, 18.0, 42.0, 26.0],         # 2.5, 4.5, 10.5, 6.5
        [-10.0, -18.0, 22.0, 2.0],        # -2.5, -4.5, 5.5, 0.5
        [4.0, 12.0, 124.0, 132.0],        # a level-1 box (stride 8): 0.5, 1.5, 15.5, 16.5
        [0.0, 0.0, 440.0, 440.0],         # large: one bin spans many pixels
        [-2000.0, -2000.0, 3000.0, 3000.0],  # huge: top level; ROIAlign's direct (untabulated) path
    ])


def random_boxes(g, n_img, per_img, frame=448.0):
    out = []
    for i in range(n_img):
        m = per_img + 5 * i
        sz = torch.exp(torch.rand(m, generator=g) * math.log(400.0 / 4.0)) * 4.0   # 4 .. 400 px: every level
        ar = torch.exp((torch.rand(m, generator=g) - 0.5) * 1.6)
        w, h = sz * torch.sqrt(ar), sz / torch.sqrt(ar)
        cx, cy = torch.rand(m, generator=g) * frame, torch.rand(m, generator=g) * frame
        out.append(torch.stack((cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2), 1))
    out[0] = torch.cat((special_boxes(), out[0]), 0)
    return out


def pyramid(g, n_img, C, nl, frame=448, dtype=torch.float32):
    strides = STRIDES[:nl] if nl > 1 else [4]
    return [torch.randn(n_img, C, frame // s, frame // s, generator=g).to(dtype) for s in strides], \
        [1.0 / s for s in strides]


def inject_non_finite(feats, g, frac=0.01):
    """NaN, +inf and -inf at random positions (set in the feature dtype)"""
    out = []
    for f in feats:
        f = f.clone()
        flat = f.view(-1)
        k = max(3, int(flat.numel() * frac))
        idx = torch.randint(0, flat.numel(), (k,), generator=g)
        flat[idx[0::3]] = float("nan")
        flat[idx[1::3]] = float("inf")
        flat[idx[2::3]] = float("-inf")
        out.append(f)
    return out


def bits16(t):
    return t.detach().contiguous().cpu().view(torch.int16)


def assert_bits_equal(got, want):
    assert got.dtype == want.dtype and got.shape == want.shape
    if got.dtype == torch.float32:
        assert torch.equal(got.detach().cpu().view(torch.int32), want.detach().cpu().view(torch.int32))
    else:
        assert torch.equal(bits16(got), bits16(want))


def ulp_distance(a, b):
    """|a - b| in units in the last place of their shared 16-bit dtype (sign-magnitude bits mapped to ordered ints)"""
    ia, ib = bits16(a).to(torch.int32), bits16(b).to(torch.int32)
    ia = torch.where(ia < 0, -32768 - ia, ia)
    ib = torch.where(ib < 0, -32768 - ib, ib)
    return (ia - ib).abs()


def assert_grad_matches_fp32_route(g16, g32):
    """g16: the fp32 atomic sums rounded once to the 16-bit dtype; g32: the fp32 route's fp32 gradient.  The sums hold
    the same addends in another order, so g16 is within one ulp of g32 rounded -- except where cancellation leaves a
    value far below its addends: there the fp32 order noise is many 16-bit ulps of the tiny result, and the bound is the
    1e-5 absolute of the fp32 backward tests."""
    assert g16.dtype in DTYPES and g32.dtype == torch.float32
    ok = (ulp_distance(g16, g32.to(g16.dtype)) <= 1) | ((g16.float() - g32).abs() <= 1e-5).cpu()
    assert ok.all(), int((~ok).sum())


def pool_c(det, feats, scales, box_lists, out_size, with_argmax=True):
    """det_roi_pool_levels called directly: (output, argmax or None)"""
    from det_b200.roi_pool import _level_table
    N = det._native
    ts = [b.cuda() for b in box_lists]
    boxes = N.f32c(torch.cat(ts, 0))
    bi = torch.cat([torch.full((t.shape[0],), i, dtype=torch.int32, device="cuda") for i, t in enumerate(ts)])
    level = None
    if len(feats) > 1:
        level = det.assign_boxes_to_levels(ts, -int(math.log2(scales[0])), -int(math.log2(scales[-1])), 224, 4)
    feats = [f.cuda().contiguous() for f in feats]
    m, c = boxes.shape[0], feats[0].shape[1]
    out = torch.full((m, c) + tuple(out_size), 7.0, dtype=feats[0].dtype, device="cuda")
    arg = torch.full(out.shape, -7, dtype=torch.int32, device="cuda") if with_argmax else None
    lv = _level_table(feats, scales)
    N.call("det_roi_pool_levels", ctypes.cast(lv, ctypes.c_void_p), len(feats), feats[0].shape[0], c, N.ptr(boxes),
           N.ptr(bi), N.ptr(level), m, out_size[0], out_size[1], N.ptr(out), N.ptr(arg), N.DTYPE_CODES[feats[0].dtype],
           N.stream())
    return out, arg


def run_pooler(det, ptype, feats, scales, box_lists, out_size, sampling_ratio=0, weight=None):
    """det.ROIPooler on CUDA copies of `feats`; with `weight`, also backward of (out * weight).sum()"""
    gf = [f.cuda().requires_grad_(weight is not None) for f in feats]
    out = det.ROIPooler(scales, sampling_ratio, out_size, ptype)(gf, [det.Boxes(b.cuda()) for b in box_lists])
    if weight is not None:
        (out * weight.cuda().to(out.dtype)).sum().backward()
    return out.detach(), [f.grad for f in gf]


# --------------------------------------------------------------------------------------------------- ROIPool, fp32
@gpu
@pytest.mark.parametrize("C", [24, 33])
@pytest.mark.parametrize("out_size", [(7, 7), (14, 14), (5, 9)], ids=["7x7", "14x14", "5x9"])
@pytest.mark.parametrize("nl", [1, 4], ids=["1level", "4levels"])
def test_roi_pool_forward_matches_torchvision_cpu(det, nl, out_size, C):
    g = gen(101 + C + nl)
    feats, scales = pyramid(g, 3, C, nl)
    box_lists = random_boxes(g, 3, 40, 448.0)
    want, want_arg = ref_roi_pool(feats, scales, box_lists, out_size)
    got, _ = run_pooler(det, "ROIPool", feats, scales, box_lists, out_size)
    assert got.dtype == torch.float32 and got.shape == want.shape
    assert torch.equal(got.cpu(), want)
    out, arg = pool_c(det, feats, scales, box_lists, out_size)
    assert torch.equal(out.cpu(), want)
    assert torch.equal(arg.cpu(), want_arg)        # plane-relative index h*W + w, -1 for empty bins
    assert (want_arg == -1).any() and (want == 0).any()


@gpu
def test_roi_pool_rounds_half_away_from_zero(det):
    """x = 2.0 at scale 1/4 is 0.5: torchvision's round() takes pixel (1, 1); rintf would take (0, 0)"""
    feat = torch.arange(16.0).view(1, 1, 4, 4)
    rois = torch.tensor([[0, 2.0, 2.0, 2.0, 2.0], [0, 6.0, 6.0, 6.0, 6.0], [0, 10.0, 2.0, 10.0, 2.0]])
    want = torchvision.ops.roi_pool(feat, rois, (1, 1), 0.25)
    assert want.view(-1).tolist() == [5.0, 10.0, 7.0]
    got, _ = run_pooler(det, "ROIPool", [feat], [0.25], [rois[:, 1:]], (1, 1))
    assert torch.equal(got.cpu(), want)


@gpu
def test_roi_pool_nan_and_minus_inf_bins(det):
    """a bin of only NaN / -inf outputs -FLT_MAX and takes no gradient; NaN never wins a mixed bin"""
    g = gen(107)
    feat = torch.randn(2, 5, 24, 24, generator=g)
    feat[0, :, 0:8, 0:8] = float("nan")
    feat[0, :, 8:16, 0:8] = float("-inf")
    feat[1, :, 0:8, 0:8] = float("nan")
    feat[1, :, 3, 5] = 2.5                              # one finite value among NaNs
    feat[1, :, 8:16, 8:16] = float("-inf")
    feat[1, :, 12, 9] = float("nan")
    box_lists = [torch.tensor([[0.0, 0.0, 28.0, 28.0], [0.0, 32.0, 28.0, 60.0], [0.0, 0.0, 60.0, 60.0]]),
                 torch.tensor([[0.0, 0.0, 28.0, 28.0], [32.0, 32.0, 60.0, 60.0]])]
    weight = torch.randn(5, 5, 2, 2, generator=g)
    cf = feat.clone().requires_grad_(True)
    want, _ = ref_roi_pool([cf], [0.25], box_lists, (2, 2))
    (want * weight).sum().backward()
    got, (grad,) = run_pooler(det, "ROIPool", [feat], [0.25], box_lists, (2, 2), weight=weight)
    assert torch.equal(got.cpu(), want.detach())
    assert (got[0] == -FLT_MAX).all() and (got[1] == -FLT_MAX).all() and (got[4] == -FLT_MAX).all()
    assert (got[3] == 2.5).any() and not got.isnan().any()
    torch.testing.assert_close(grad.cpu(), cf.grad, rtol=0, atol=1e-5)
    assert (grad[0, :, 0:16, 0:8] == 0).all() and (grad[1, :, 8:16, 8:16] == 0).all()


@gpu
@pytest.mark.parametrize("C", [10, 33])
@pytest.mark.parametrize("nl", [1, 4], ids=["1level", "4levels"])
def test_roi_pool_backward_matches_cpu_autograd(det, nl, C):
    g = gen(111 + nl + C)
    feats, scales = pyramid(g, 2, C, nl, frame=224)
    box_lists = random_boxes(g, 2, 30, 224.0)
    m = sum(b.shape[0] for b in box_lists)
    weight = torch.randn(m, C, 7, 7, generator=g)
    cf = [f.clone().requires_grad_(True) for f in feats]
    want, _ = ref_roi_pool(cf, scales, box_lists, (7, 7))
    (want * weight).sum().backward()
    got, grads = run_pooler(det, "ROIPool", feats, scales, box_lists, (7, 7), weight=weight)
    assert torch.equal(got.cpu(), want.detach())
    for gg, c in zip(grads, cf):
        assert gg.dtype == torch.float32
        torch.testing.assert_close(gg.cpu(), c.grad, rtol=1e-5, atol=1e-5)


@gpu
def test_roi_pool_tie_heavy_gradient_lands_on_first_maximum(det):
    """integer-valued features: most bins hold several equal maxima; the gradient goes to the first in scan order"""
    g = gen(113)
    feats = [torch.randint(0, 3, (2, 12, 448 // s, 448 // s), generator=g).float() for s in STRIDES]
    scales = [1.0 / s for s in STRIDES]
    box_lists = random_boxes(g, 2, 40)
    m = sum(b.shape[0] for b in box_lists)
    weight = torch.randn(m, 12, 7, 7, generator=g)
    cf = [f.clone().requires_grad_(True) for f in feats]
    want, want_arg = ref_roi_pool(cf, scales, box_lists, (7, 7))
    (want * weight).sum().backward()
    got, grads = run_pooler(det, "ROIPool", feats, scales, box_lists, (7, 7), weight=weight)
    assert torch.equal(got.cpu(), want.detach())
    _, arg = pool_c(det, feats, scales, box_lists, (7, 7))
    assert torch.equal(arg.cpu(), want_arg)
    for gg, c in zip(grads, cf):
        torch.testing.assert_close(gg.cpu(), c.grad, rtol=1e-5, atol=1e-5)


@gpu
def test_roi_pool_inference_writes_no_argmax(det, monkeypatch):
    """argmax is passed (and saved) only when a feature map requires grad; otherwise the kernel gets NULL"""
    from det_b200 import _native as N
    seen = []
    real = N.call

    def spy(name, *args):
        if name == "det_roi_pool_levels":
            seen.append(args[11])                       # the argmax pointer
        return real(name, *args)

    monkeypatch.setattr(N, "call", spy)
    g = gen(117)
    feats, scales = pyramid(g, 2, 8, 4, frame=224)
    box_lists = random_boxes(g, 2, 10, 224.0)
    plain, _ = run_pooler(det, "ROIPool", feats, scales, box_lists, (7, 7))
    assert seen == [None]
    gf = [f.cuda().requires_grad_(True) for f in feats]
    out = det.ROIPooler(scales, 0, 7, "ROIPool")(gf, [det.Boxes(b.cuda()) for b in box_lists])
    assert seen[1] is not None
    saved = out.grad_fn.saved_tensors
    assert saved[-1].dtype == torch.int32 and saved[-1].shape == out.shape
    assert torch.equal(out.detach(), plain)
    # and at the C level: NULL argmax, same output
    o1, a1 = pool_c(det, feats, scales, box_lists, (7, 7), with_argmax=False)
    assert a1 is None and torch.equal(o1, plain)


# --------------------------------------------------------------------------------------------------- 16-bit features
POOLERS = [("ROIAlignV2", 0, (7, 7)), ("ROIAlignV2", 2, (14, 14)), ("ROIAlign", 0, (7, 7)), ("ROIAlign", 2, (7, 7)),
           ("ROIAlignV2", 0, (14, 14)), ("ROIPool", 0, (7, 7)), ("ROIPool", 0, (5, 9))]
POOLER_IDS = [f"{t}-sr{s}-{o[0]}x{o[1]}" for t, s, o in POOLERS]


def oracle_cpu(ptype, feats, scales, box_lists, out_size, sampling_ratio):
    """torchvision CPU (fp32) through the reference's per-level loop, autograd-connected"""
    if ptype == "ROIPool":
        return ref_roi_pool(feats, scales, box_lists, out_size)[0]
    from tests.test_gpu_roi_pool import ref_pooler
    lv = (-int(math.log2(scales[0])), -int(math.log2(scales[-1])))
    return ref_pooler(feats, scales, box_lists, out_size, sampling_ratio, ptype == "ROIAlignV2", *lv)


TOL16 = {torch.bfloat16: dict(rtol=1.6e-2, atol=1e-3), torch.float16: dict(rtol=2e-3, atol=1e-4)}


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("ptype,sampling_ratio,out_size", POOLERS, ids=POOLER_IDS)
def test_16bit_forward_bit_identical_to_fp32_route(det, dt, ptype, sampling_ratio, out_size):
    g = gen(201)
    feats, scales = pyramid(g, 3, 33, 4, dtype=dt)
    feats = inject_non_finite(feats, g)
    box_lists = random_boxes(g, 3, 40)
    got, _ = run_pooler(det, ptype, feats, scales, box_lists, out_size, sampling_ratio)
    want, _ = run_pooler(det, ptype, [f.float() for f in feats], scales, box_lists, out_size, sampling_ratio)
    assert got.dtype == dt
    assert_bits_equal(got, want.to(dt))
    assert not got.isfinite().all()


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("ptype,sampling_ratio,out_size", POOLERS, ids=POOLER_IDS)
def test_16bit_backward(det, dt, ptype, sampling_ratio, out_size):
    g = gen(203)
    feats, scales = pyramid(g, 2, 20, 4, frame=224, dtype=dt)
    box_lists = random_boxes(g, 2, 30, 224.0)
    m = sum(b.shape[0] for b in box_lists)
    weight = torch.randn((m, 20) + out_size, generator=g).to(dt)
    got, grads = run_pooler(det, ptype, feats, scales, box_lists, out_size, sampling_ratio, weight=weight)
    f32 = [f.float() for f in feats]
    gf32 = [f.cuda().requires_grad_(True) for f in f32]
    out32 = det.ROIPooler(scales, sampling_ratio, out_size, ptype)(gf32, [det.Boxes(b.cuda()) for b in box_lists])
    (out32.to(dt) * weight.cuda()).sum().backward()       # the parent's route: fp32 call, then .to(dt)
    cf = [f.clone().requires_grad_(True) for f in f32]
    ref = oracle_cpu(ptype, cf, scales, box_lists, out_size, sampling_ratio)
    (ref * weight.float()).sum().backward()
    for gg, g32, c in zip(grads, gf32, cf):
        assert gg.dtype == dt
        assert_grad_matches_fp32_route(gg, g32.grad)
        torch.testing.assert_close(gg.float().cpu(), c.grad, **TOL16[dt])


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("aligned", [True, False])
def test_16bit_single_level_roi_align(det, dt, aligned):
    """det.ROIAlign (one level): tabulated and direct-path boxes, NaN / inf injected"""
    g = gen(207)
    feat = inject_non_finite([torch.randn(2, 9, 112, 112, generator=g).to(dt)], g, frac=0.002)[0]
    boxes = random_boxes(g, 1, 30)[0]                      # starts with special_boxes()
    rois = torch.cat((torch.randint(0, 2, (boxes.shape[0], 1), generator=g).float(), boxes), 1).cuda()
    for sr in (0, 2):
        ra = det.ROIAlign((7, 7), 0.25, sr, aligned)
        got = ra(feat.cuda(), rois)
        assert got.dtype == dt
        assert_bits_equal(got, ra(feat.cuda().float(), rois).to(dt))
    # backward on finite features
    feat = torch.randn(2, 9, 112, 112, generator=g).to(dt)
    weight = torch.randn(rois.shape[0], 9, 7, 7, generator=g).to(dt)
    gf = feat.cuda().requires_grad_(True)
    (det.ROIAlign((7, 7), 0.25, 0, aligned)(gf, rois) * weight.cuda()).sum().backward()
    g32 = feat.float().cuda().requires_grad_(True)
    (det.ROIAlign((7, 7), 0.25, 0, aligned)(g32, rois).to(dt) * weight.cuda()).sum().backward()
    cf = feat.float().requires_grad_(True)
    (torchvision.ops.roi_align(cf, rois.cpu(), (7, 7), 0.25, 0, aligned) * weight.float()).sum().backward()
    assert gf.grad.dtype == dt
    assert_grad_matches_fp32_route(gf.grad, g32.grad)
    torch.testing.assert_close(gf.grad.float().cpu(), cf.grad, **TOL16[dt])


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("ptype", ["ROIAlignV2", "ROIPool"])
def test_16bit_non_contiguous_and_offset_views(det, dt, ptype):
    g = gen(211)
    big = [torch.randn(2, 40, 448 // s, 448 // s + 1, generator=g).to(dt).cuda() for s in STRIDES]
    scales = [1.0 / s for s in STRIDES]
    box_lists = random_boxes(g, 2, 30)

    def offset_view(t):  # contiguous, one element (2 bytes) into its buffer
        buf = torch.zeros(t.numel() + 1, dtype=t.dtype, device=t.device)
        return buf[1:].view(t.shape).copy_(t)

    for feats in ([b[:, 3:27, :, 1:] for b in big],          # channel slice of an offset column slice
                  [b[..., 1:] for b in big],                  # starts one element into each row
                  [b[:1, 5:29] for b in big],                 # single image, channel slice: contiguous, offset
                  [offset_view(b[:, :, :, 1:]) for b in big]):
        bl = box_lists[:feats[0].shape[0]]
        got, _ = run_pooler(det, ptype, feats, scales, bl, (7, 7))
        want, _ = run_pooler(det, ptype, [f.float() for f in feats], scales, bl, (7, 7))
        assert_bits_equal(got, want.to(dt))


@gpu
@pytest.mark.parametrize("ptype", ["ROIAlignV2", "ROIAlign", "ROIPool"])
def test_mixed_dtypes_and_fp64_take_the_fp32_route(det, ptype):
    g = gen(213)
    base, scales = pyramid(g, 2, 12, 4, frame=224)
    box_lists = random_boxes(g, 2, 30, 224.0)
    for dts in ([torch.bfloat16, torch.float16, torch.float32, torch.bfloat16], [torch.float64] * 4,
                [torch.float32, torch.float64, torch.float32, torch.float32]):
        feats = [f.to(d) for f, d in zip(base, dts)]
        m = sum(b.shape[0] for b in box_lists)
        weight = torch.randn(m, 12, 7, 7, generator=g)
        got, grads = run_pooler(det, ptype, feats, scales, box_lists, (7, 7), weight=weight)
        gf32 = [f.float().cuda().requires_grad_(True) for f in feats]
        want = det.ROIPooler(scales, 0, 7, ptype)(gf32, [det.Boxes(b.cuda()) for b in box_lists])
        (want.to(dts[0]) * weight.cuda().to(dts[0])).sum().backward()
        assert got.dtype == dts[0]
        assert torch.equal(got, want.detach().to(dts[0]))
        for gg, g32, d in zip(grads, gf32, dts):
            assert gg.dtype == d
            torch.testing.assert_close(gg.float(), g32.grad.to(d).float(), rtol=1e-2, atol=1e-4)


@gpu
@pytest.mark.parametrize("seed", list(range(int(os.environ.get("DET_STRESS_SEEDS", "12")))))
def test_roi_pooler_types_stress(det, seed):
    """random shapes, dtypes and pooler types: fp32 against torchvision CPU, 16-bit bitwise against the fp32 route"""
    g = gen(3000 + seed)
    r = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    ptype = ["ROIAlignV2", "ROIAlign", "ROIPool"][r(0, 2)]
    dt = [torch.float32, torch.bfloat16, torch.float16][r(0, 2)]
    nl, n_img, C, frame = [1, 4][r(0, 1)], r(1, 3), r(1, 70), 32 * r(4, 10)
    out_size, sr = (r(1, 16), r(1, 16)), r(0, 3)
    feats, scales = pyramid(g, n_img, C, nl, frame=frame, dtype=dt)
    box_lists = random_boxes(g, n_img, r(0, 40), float(frame))
    got, _ = run_pooler(det, ptype, feats, scales, box_lists, out_size, sr)
    assert got.dtype == dt
    if dt == torch.float32:
        want = oracle_cpu(ptype, feats, scales, box_lists, out_size, sr)
        if ptype == "ROIPool":
            assert torch.equal(got.cpu(), want)
        else:
            torch.testing.assert_close(got.cpu(), want, rtol=1e-5, atol=1e-5)
    else:
        want, _ = run_pooler(det, ptype, [f.float() for f in feats], scales, box_lists, out_size, sr)
        assert_bits_equal(got, want.to(dt))


# --------------------------------------------------------------------------------------------------- CPU
def test_roi_pool_pooler_constructs_without_gpu():
    import det_b200 as det
    p = det.ROIPooler([1 / 4, 1 / 8, 1 / 16, 1 / 32], 0, 7, "ROIPool")
    assert (p.type, p.output_size, p.min_level, p.max_level) == ("ROIPool", (7, 7), 2, 5)
    with pytest.raises(ValueError):
        det.ROIPooler([0.25], 0, 7, "ROIMaxPool")


def test_pooling_entry_points_reject_unknown_dtype_without_gpu():
    """an unknown feature / gradient dtype is refused with DET_ERR_BAD_ARG and a message before any CUDA call; m == 0
    returns DET_OK without reading a pointer"""
    from det_b200 import _native as N
    null, one = ctypes.c_void_p(0), ctypes.c_void_p(16)   # `one` is never dereferenced
    lv = (N.FeatureLevel * 1)()
    lv[0].data, lv[0].h, lv[0].w, lv[0].spatial_scale = 16, 8, 8, 0.25
    lvp = ctypes.cast(lv, ctypes.c_void_p)
    err = N.fn("det_last_error")
    calls = {
        "det_roi_align_levels_typed": lambda m, d, p: (p, 1, 1, 4, p, p, null, m, 7, 7, 0, 1, p, d, null),
        "det_roi_align_levels_backward_typed": lambda m, d, p: (p, 1, 1, 4, p, p, null, m, 7, 7, 0, 1, p, d, null),
        "det_roi_pool_levels": lambda m, d, p: (p, 1, 1, 4, p, p, null, m, 7, 7, p, p, d, null),
        "det_roi_pool_levels_backward": lambda m, d, p: (p, 1, 1, 4, p, null, m, 7, 7, p, p, d, null),
    }
    for name, args in calls.items():
        f = N.fn(name)
        for bad in (3, -1, 7):
            a = list(args(5, bad, one))
            a[0] = lvp
            assert f(*a) == -1, name
            assert b"dtype" in err(), name
        for code in (0, 1, 2):
            assert f(*args(0, code, null)) == 0, name   # m == 0: nothing to do, NULL pointers accepted
        a = list(args(5, 0, null))
        assert f(*a) == -1 and b"null pointer" in err(), name
