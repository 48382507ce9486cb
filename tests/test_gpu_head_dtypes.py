"""16-bit detection heads read natively: for a bf16 / fp16 head h, every output of the decode and detect paths must be
BIT-identical to the fp32 path fed h.float() -- indices, counts, boxes, scores, classes, logits and dense outputs, NaN
compared by bit pattern.  (The kernels widen each element to fp32 as they load it and then run the fp32 instructions.)

GPU tests carry their own gpu mark so the CPU tests at the end run without a device."""
import ctypes
import os

import pytest
import torch

from tests.util import gen

DTYPES = [torch.bfloat16, torch.float16]
DT_IDS = ["bf16", "fp16"]
gpu = pytest.mark.gpu

STRIDES = [8, 16, 32]
WH = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]]


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


def bits(t):
    """exact comparison key: floating tensors by bit pattern (NaN == NaN of the same bits), integers as they are"""
    t = t.detach().contiguous().cpu()
    if t.dtype == torch.float32:
        return t.view(torch.int32)
    return t


def assert_same(a, b, what=""):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    assert torch.equal(bits(a), bits(b)), f"{what}: outputs differ"


def padded(h):
    """`h` on the GPU as the leading view of a zero-filled buffer three times its size: a kernel that walks planes with
    the wrong stride reads zeros (and gets a wrong answer) instead of leaving the allocation"""
    buf = torch.zeros(3 * h.numel(), dtype=h.dtype, device="cuda")
    v = buf[:h.numel()].view(h.shape)
    v.copy_(h.cuda())
    return v


def make_heads(n, image, C, seed, obj_bias, dtype, strides=STRIDES, a=3):
    g = gen(seed)
    heads = [torch.randn(n, a * (5 + C), image // s, image // s, generator=g) for s in strides]
    for h in heads:
        h.view(n, a, 5 + C, h.shape[2], h.shape[3])[:, :, 4] += obj_bias
    return [h.to(dtype) for h in heads]


def assert_detect_same(r16, r32):
    cnt = r16["count"].cpu()
    assert_same(cnt, r32["count"].cpu(), "count")
    for i in range(cnt.shape[0]):  # rows past the count are undefined
        k = max(int(cnt[i]), 0)
        for key in ("idx", "boxes", "scores", "classes"):
            assert_same(r16[key][i, :k], r32[key][i, :k], f"{key} of image {i}")


def assert_decode_same(d16, d32):
    for a, b, w in zip(d16, d32, ("boxes", "scores", "classes")):
        assert_same(a, b, w)


# ------------------------------------------------------------------------------------------------ dense decode
@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_dense_decode_flat_pyramid(det, dt):
    """640 px pyramid (80^2, 40^2, 20^2): one flat launch, vector loads of 4 positions"""
    C = 80
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    heads = [padded(h) for h in make_heads(2, 640, C, 3, -1.0, dt)]
    assert_decode_same(dh.decode(heads), dh.decode([h.float() for h in heads]))


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_dense_decode_levels_not_multiple_of_four(det, dt):
    """13x13 and 7x9 levels (h*w % 4 != 0): scalar loads inside the one flat launch"""
    C = 20
    dh = det.DenseAnchorHead([32, 64], WH[1:], C)
    g = gen(17)
    heads = [(torch.randn(3, 3 * (5 + C), h, w, generator=g) * 2).to(dt).cuda() for h, w in [(13, 13), (7, 9)]]
    assert_decode_same(dh.decode(heads), dh.decode([h.float() for h in heads]))


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_dense_decode_unequal_anchor_counts(det, dt):
    """levels with 3 and 2 anchors: one typed launch per level"""
    C = 11
    dh = det.DenseAnchorHead([16, 32], [WH[0], WH[1][:2]], C)
    g = gen(23)
    heads = [torch.randn(2, 3 * (5 + C), 20, 20, generator=g).to(dt).cuda(),
             torch.randn(2, 2 * (5 + C), 10, 10, generator=g).to(dt).cuda()]
    assert_decode_same(dh.decode(heads), dh.decode([h.float() for h in heads]))


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_dense_decode_unaligned_view(det, dt):
    """a head that starts one element into its buffer: the wrapper copies it to an aligned buffer, and the C entry point
    handed the unaligned pointer itself reads it with scalar loads -- both equal to the fp32 path"""
    C, n, hh = 20, 2, 16
    dh = det.DenseAnchorHead([32], [WH[2]], C)
    src = torch.randn(n, 3 * (5 + C), hh, hh, generator=gen(29)).to(dt)
    buf = torch.zeros(src.numel() + 1, dtype=dt, device="cuda")
    view = buf[1:].view(src.shape)
    view.copy_(src.cuda())
    assert view.is_contiguous() and view.data_ptr() % 8 != 0
    want = dh.decode([view.float()])
    assert_decode_same(dh.decode([view]), want)
    R = hh * hh * 3
    boxes = torch.empty((n, R, 4), device="cuda")
    scores = torch.empty((n, R), device="cuda")
    classes = torch.empty((n, R), dtype=torch.int64, device="cuda")
    a = dh._anchors_on(view.device)[0]
    lv = det._native.DenseLevel(view.data_ptr(), a.data_ptr(), hh, hh, 32, 0, 0)
    det._native.call("det_dense_decode_typed", ctypes.byref(lv), 1, n, 3, C, dh.scale_clamp, det._native.ptr(boxes),
                     det._native.ptr(scores), det._native.ptr(classes), R, det._native.DTYPE_CODES[dt],
                     det._native.stream())
    assert_decode_same((boxes, scores, classes), want)


# ------------------------------------------------------------------------------------------------ dense detect
DETECT_CASES = [  # image, n, obj bias, thr, iou, cand_cap, max_det
    pytest.param(256, 4, -4.0, 0.1, 0.5, 1024, 300, id="offset-trick"),    # <= 1000 candidates
    pytest.param(256, 3, -1.0, 0.25, 0.5, 2048, 300, id="per-category"),   # > 1000 candidates
    pytest.param(256, 3, 0.0, 0.3, 0.5, 4096, 100, id="tier-cut"),         # the best ~1.25 max_det yield max_det
    pytest.param(256, 3, 0.0, 0.3, 0.01, 4096, 100, id="tier-short"),      # heavy suppression: everything is swept
    pytest.param(128, 5, -2.0, 0.05, 0.5, 1024, 7, id="max-det"),          # max_det cuts the list
]


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("gate", [True, False], ids=["gate", "nogate"])
@pytest.mark.parametrize("image,n,bias,thr,iou,cap,max_det", DETECT_CASES)
def test_dense_detect(det, dt, gate, image, n, bias, thr, iou, cap, max_det):
    C = 80
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    heads = [padded(h) for h in make_heads(n, image, C, 41 + image + n, bias, dt)]
    r16 = dh.detect_thresholded(heads, thr, iou, max_det=max_det, cand_cap=cap, gate=gate, check=False)
    r32 = dh.detect_thresholded([h.float() for h in heads], thr, iou, max_det=max_det, cand_cap=cap, gate=gate,
                                check=False)
    assert int(r16["overflow"].item()) == 0 and int(r32["overflow"].item()) == 0
    assert int(r32["count"].min()) >= (1 if thr < 0.5 else 0)
    assert_detect_same(r16, r32)


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("gate", [True, False], ids=["gate", "nogate"])
def test_dense_detect_non_finite_logits(det, dt, gate):
    """NaN and +-Inf injected in 16 bit into box, objectness and class planes (the arg-max's exact NaN rescan)"""
    C = 80
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    heads = make_heads(3, 256, C, 53, -1.0, dt)
    g = gen(54)
    for h in heads:
        for val in (float("nan"), float("inf"), float("-inf")):
            m = torch.rand(h.shape, generator=g) < 0.002
            h[m] = torch.tensor(val, dtype=dt)
        v = h.view(3, 3, 5 + C, h.shape[2], h.shape[3])
        v[0, 1, 5 + 40, :2, :2] = float("nan")   # NaN class logits in whole columns of the arg-max
        v[1, 0, 5 + 7, 1, :] = float("inf")
    heads = [padded(h) for h in heads]
    h32 = [h.float() for h in heads]
    assert_decode_same(dh.decode(heads), dh.decode(h32))
    r16 = dh.detect_thresholded(heads, 0.2, 0.5, max_det=300, cand_cap=4096, gate=gate, check=False)
    r32 = dh.detect_thresholded(h32, 0.2, 0.5, max_det=300, cand_cap=4096, gate=gate, check=False)
    assert_detect_same(r16, r32)


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_dense_detect_owned_workspace_and_overflow(det, dt):
    """a DenseDetectWorkspace over several calls, one of them overflowing: with check=True the overflowing batch takes
    the unfused route (decode -> compact -> NMS -> gather) on the 16-bit head"""
    C = 80
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    ws16 = det.DenseDetectWorkspace(3, 1024, "cuda")
    ws32 = det.DenseDetectWorkspace(3, 1024, "cuda")
    for seed, bias, check in [(61, -4.0, False), (62, 1.0, True), (63, -3.0, False), (64, 0.0, True)]:
        heads = [h.cuda() for h in make_heads(3, 256, C, seed, bias, dt)]
        h32 = [h.float() for h in heads]
        r16 = dh.detect_thresholded(heads, 0.2, 0.5, max_det=300, cand_cap=1024, check=check, workspace=ws16)
        r32 = dh.detect_thresholded(h32, 0.2, 0.5, max_det=300, cand_cap=1024, check=check, workspace=ws32)
        if check:  # the unfused route ran (the fused call overflowed)
            n_cand = (dh.decode(h32)[1] > 0.2).sum(1)
            assert int(n_cand.max()) > 1024
        assert_detect_same(r16, r32)
        assert int(ws16.buf[:det._native.fn("det_dense_detect_counter_bytes")(3)].count_nonzero()) == 0


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("iou,max_det", [(0.5, 300), (0.3, 40)])
def test_dense_detect_tie_heavy(det, dt, iou, max_det):
    """heads drawn from a few dozen distinct 16-bit values: many exactly equal scores, so the row-order tie handling
    of the fast and general NMS forms decides the output order"""
    C = 12
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    vals = torch.linspace(-3.0, 3.0, 40).to(dt)
    g = gen(71)
    heads = []
    for s in STRIDES:
        idx = torch.randint(0, vals.numel(), (4, 3 * (5 + C), 256 // s, 256 // s), generator=g)
        heads.append(vals[idx].cuda())
    h32 = [h.float() for h in heads]
    scores = dh.decode(h32)[1]
    for i in range(4):  # the premise: equal scores among the candidates
        s = scores[i][scores[i] > 0.3]
        assert s.numel() - s.unique().numel() > s.numel() // 2
    for gate in (True, False):
        r16 = dh.detect_thresholded(heads, 0.3, iou, max_det=max_det, cand_cap=4096, gate=gate, check=False)
        r32 = dh.detect_thresholded(h32, 0.3, iou, max_det=max_det, cand_cap=4096, gate=gate, check=False)
        assert_detect_same(r16, r32)
    b16 = dh.detect(heads, iou, max_det=max_det)
    b32 = dh.detect(h32, iou, max_det=max_det)
    for a, b in zip(b16, b32):
        assert_same(a, b)


# ------------------------------------------------------------------------------------------------ RPN
RPN_STRIDES = [4, 8, 16, 32, 64]
RPN_SIZES = [[32], [64], [128], [256], [512]]
ANCHOR_SETS = {  # anchors per position: (sizes per level, ratios)
    1: (RPN_SIZES, [[1.0]]),
    2: (RPN_SIZES, [[0.5, 2.0]]),
    3: (RPN_SIZES, [[0.5, 1.0, 2.0]]),
    4: ([[s[0], s[0] * 1.5] for s in RPN_SIZES], [[0.5, 2.0]]),
    9: ([[s[0], s[0] * 1.26, s[0] * 1.59] for s in RPN_SIZES], [[0.5, 1.0, 2.0]]),
}


def rpn_heads(n, img, a, g, dt, scale=4.0, beyond_clamp=True):
    obj = [torch.randn(n, a, img // s, img // s, generator=g) for s in RPN_STRIDES]
    dlt = [torch.randn(n, 4 * a, img // s, img // s, generator=g) * scale for s in RPN_STRIDES]
    if beyond_clamp:
        for d in dlt:  # beyond scale_clamp after dividing by the weight 5, both signs of dx / dy
            d[:, 2::4, ::3, ::2] = 30.0
            d[:, 3::4, 1::3, ::2] = 25.0
            d[:, 0::4, ::2, 1::3] *= -3.0
    return [o.to(dt).cuda() for o in obj], [d.to(dt).cuda() for d in dlt]


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("img,a", [(448, 3), (224, 1), (224, 2), (448, 4), (448, 9)],
                         ids=["448-a3", "224-a1", "224-a2", "448-a4", "448-a9"])
def test_rpn_decode_heads(det, dt, img, a):
    """a <= 4: one flat launch (7x7 level with scalar loads at 448); a = 9: one launch per level (vec and scalar)"""
    sizes, ratios = ANCHOR_SETS[a]
    rpn = det.RegionProposalNetwork(RPN_STRIDES, sizes, ratios, box2box_weights=(10.0, 10.0, 5.0, 5.0))
    obj, dlt = rpn_heads(3, img, a, gen(img + a), dt)
    got = rpn.decode_heads(obj, dlt)
    want = rpn.decode_heads([o.float() for o in obj], [d.float() for d in dlt])
    assert got[2] == want[2]
    assert_same(got[0], want[0], "logits")
    assert_same(got[1], want[1], "boxes")


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_rpn_proposals_and_forward_eval(det, dt):
    rpn = det.RegionProposalNetwork(RPN_STRIDES, RPN_SIZES, [[0.5, 1.0, 2.0]]).eval()
    obj, dlt = rpn_heads(2, 224, 3, gen(81), dt, scale=0.3, beyond_clamp=False)
    o32, d32 = [o.float() for o in obj], [d.float() for d in dlt]
    sizes = torch.tensor([[224, 224], [200, 210]], dtype=torch.int32, device="cuda")
    for a, b in zip(rpn.proposals_from_heads(obj, dlt, sizes), rpn.proposals_from_heads(o32, d32, sizes)):
        assert_same(a, b)
    p16, l16 = rpn.forward([(224, 224), (200, 210)], head_outputs=(obj, dlt))
    p32, l32 = rpn.forward([(224, 224), (200, 210)], head_outputs=(o32, d32))
    assert l16 == {} and l32 == {}
    for a, b in zip(p16, p32):
        assert_same(a.proposal_boxes.tensor, b.proposal_boxes.tensor)
        assert_same(a.objectness_logits, b.objectness_logits)


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_rpn_forward_training(det, dt):
    """training: the proposals equal the fp32 run's; a 16-bit head takes the generic matcher + dense loss (as before),
    whose losses equal that route run by hand on the same values in fp32 with the same sampling seed -- to 1e-5: the
    loss kernel sums with atomics, so the last bits depend on the order the CTAs arrive in"""
    rpn = det.RegionProposalNetwork(RPN_STRIDES, RPN_SIZES, [[0.5, 1.0, 2.0]]).train()
    n, img = 2, 256
    obj, dlt = rpn_heads(n, img, 3, gen(91), dt, scale=0.3, beyond_clamp=False)
    o32, d32 = [o.float() for o in obj], [d.float() for d in dlt]
    gts = [torch.tensor([[10.0, 12.0, 90.0, 100.0], [30.0, 40.0, 200.0, 160.0]]),
           torch.tensor([[5.0, 5.0, 120.0, 80.0]])]
    insts = []
    for b in gts:
        inst = det.Instances((img, img))
        inst.gt_boxes = det.Boxes(b.cuda())
        insts.append(inst)
    rpn._sample_seed = 40
    p16, l16 = rpn.forward([(img, img)] * n, head_outputs=(obj, dlt), gt_instances=insts)
    p32, _ = rpn.forward([(img, img)] * n, head_outputs=(o32, d32), gt_instances=insts)
    for a, b in zip(p16, p32):
        assert_same(a.proposal_boxes.tensor, b.proposal_boxes.tensor)
        assert_same(a.objectness_logits, b.objectness_logits)
    anchors = torch.cat(rpn.anchor_generator.grid_anchors([(img // s, img // s) for s in RPN_STRIDES], "cuda"), 0)
    asg = rpn.assign(anchors, [b.cuda() for b in gts], seed=41)
    logits = torch.cat([o.permute(0, 2, 3, 1).reshape(n, -1) for o in o32], 1)
    deltas = torch.cat([d.view(n, -1, 4, d.shape[-2], d.shape[-1]).permute(0, 3, 4, 1, 2).reshape(n, -1, 4)
                        for d in d32], 1)
    want = rpn.fused_losses(anchors, logits, deltas, asg)
    assert torch.isfinite(l16["cls_loss"]) and torch.isfinite(l16["loc_loss"])
    torch.testing.assert_close(l16["cls_loss"], want["cls_loss"], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(l16["loc_loss"], want["loc_loss"], rtol=1e-5, atol=1e-7)


# ------------------------------------------------------------------------------------------------ YOLO
def yolo_same(r16, r32, dense=False):
    cnt = r16["count"].cpu()
    assert_same(cnt, r32["count"].cpu(), "count")
    for i in range(cnt.shape[0]):
        k = int(cnt[i])
        for key in ("flat", "boxes", "scores"):
            assert_same(r16[key][i, :k], r32[key][i, :k], f"{key} of image {i}")
    if dense:
        for key in ("dense_boxes", "dense_conf", "dense_scores"):
            assert_same(r16[key], r32[key], key)


YOLO_SHAPES = [  # S, B, C, image, clip, thr, iou
    pytest.param(7, 2, 20, (448, 448), True, 0.25, 0.5, id="baseline-fast"),   # compile-time shape of the fast kernel
    pytest.param(8, 2, 32, (512, 512), True, 0.2, 0.5, id="fast-generic"),     # fast kernel, shape from parameters
    pytest.param(5, 3, 7, (320, 480), False, 0.1, 0.45, id="generic"),         # unclipped: the generic kernel
    pytest.param(9, 3, 10, (416, 416), True, 0.2, 0.5, id="generic-large"),    # 243 predictors: the generic kernel
]


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("S,B,C,hw,clip,thr,iou", YOLO_SHAPES)
def test_yolo_detect(det, dt, S, B, C, hw, clip, thr, iou):
    yh = det.YoloGridHead(S, B, C, hw, clip=clip)
    head = (torch.randn(9, S, S, B * 5 + C, generator=gen(S * 10 + C)) * 1.3).to(dt).cuda()
    for index_dtype in (torch.int64, torch.int32):
        r16 = yh.detect(head, thr, iou, return_dense=True, index_dtype=index_dtype)
        r32 = yh.detect(head.float(), thr, iou, return_dense=True, index_dtype=index_dtype)
        yolo_same(r16, r32, dense=True)
    for a, b in zip(yh.decode(head), yh.decode(head.float())):
        assert_same(a, b)


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("S,B,C,clip", [(7, 2, 20, True), (5, 3, 7, False)], ids=["fast", "generic"])
def test_yolo_non_finite_logits(det, dt, S, B, C, clip):
    yh = det.YoloGridHead(S, B, C, (448, 448), clip=clip)
    head = torch.randn(6, S, S, B * 5 + C, generator=gen(97)).to(dt)
    head[0, 3, 3, 2] = float("nan")
    head[1, 1, 2, 4] = float("inf")
    head[2, 0, 0, B * 5 + 1] = float("nan")
    head[3, 2, 1, 3] = float("-inf")
    head[4, 4, 4, 0] = float("inf")
    head = head.cuda()
    yolo_same(yh.detect(head, 0.2, 0.5, return_dense=True), yh.detect(head.float(), 0.2, 0.5, return_dense=True), True)


@gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "stream"])
def test_yolo_host_pipeline_16bit_input(det, dt, use_graph):
    """pinned 16-bit host input -> 16-bit device input -> kernel: equal to detect() on the same head, and half the
    upload bytes of the fp32 pipeline"""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    pipe = det.YoloHostPipeline(yh, 32, 0.25, 0.5, 300, depth=3, use_graph=use_graph, index_dtype=torch.int32,
                                input_dtype=dt)
    ref = det.YoloHostPipeline(yh, 32, 0.25, 0.5, 300, depth=1, use_graph=False, index_dtype=torch.int32)
    assert pipe.h2d_bytes * 2 == ref.h2d_bytes == 32 * 7 * 7 * 30 * 4
    assert all(t.dtype == dt for t in pipe.h_in + pipe.d_in)
    heads = (torch.randn(5, 32, 7, 7, 30, generator=gen(101)) * 1.5).to(dt)
    got = []
    for i in range(5):
        s = i % 3
        if i >= 3:
            got.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in pipe.wait(s).items()})
        pipe.input(s).copy_(heads[i])
        pipe.launch(s)
    for i in (2, 3, 4):  # the batches still in flight, in slots 2, 0, 1
        got.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in pipe.wait(i % 3).items()})
    for i in range(5):
        want = yh.detect(heads[i].cuda().float(), 0.25, 0.5, max_det=300, index_dtype=torch.int32)
        yolo_same(got[i], {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in want.items()})


# ------------------------------------------------------------------------------------------------ stress
@gpu
@pytest.mark.parametrize("seed", list(range(int(os.environ.get("DET_STRESS_SEEDS", "12")))))
def test_head_dtypes_stress(det, seed):
    """random shapes, dtypes, thresholds and injected NaN / Inf through every native 16-bit route"""
    g = gen(1000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    rf = lambda lo, hi: float(torch.empty(()).uniform_(lo, hi, generator=g))
    dt = DTYPES[ri(0, 1)]

    def inject(t):
        for val in (float("nan"), float("inf"), float("-inf")):
            m = torch.rand(t.shape, generator=g) < rf(0.0, 0.003)
            t[m] = torch.tensor(val, dtype=t.dtype)
        return t

    # dense head: random pyramid, some levels not a multiple of 4 positions
    C, n = ri(1, 40), ri(1, 5)
    nl = ri(1, 3)
    hws = [(ri(1, 24), ri(1, 24)) if ri(0, 2) == 0 else (4 * ri(1, 8), ri(1, 12)) for _ in range(nl)]
    dh = det.DenseAnchorHead([8 * 2 ** i for i in range(nl)], [WH[i] for i in range(nl)], C)
    heads = [padded(inject((torch.randn(n, 3 * (5 + C), h, w, generator=g) * rf(0.5, 3.0)).to(dt))) for h, w in hws]
    h32 = [h.float() for h in heads]
    assert_decode_same(dh.decode(heads), dh.decode(h32))
    thr, iou, max_det = rf(0.05, 0.6), rf(0.2, 0.8), ri(1, 400)
    r16 = dh.detect_thresholded(heads, thr, iou, max_det=max_det, cand_cap=4096, gate=bool(ri(0, 1)))
    r32 = dh.detect_thresholded(h32, thr, iou, max_det=max_det, cand_cap=4096, gate=True)
    assert_detect_same(r16, r32)
    # RPN
    a = [1, 2, 3, 4, 9][ri(0, 4)]
    sizes, ratios = ANCHOR_SETS[a]
    rpn = det.RegionProposalNetwork(RPN_STRIDES, sizes, ratios, box2box_weights=(rf(1, 10), rf(1, 10), rf(1, 5), rf(1, 5)))
    img = 32 * ri(2, 9)
    obj, dlt = rpn_heads(ri(1, 3), img, a, g, dt, scale=rf(0.2, 6.0), beyond_clamp=bool(ri(0, 1)))
    obj, dlt = [inject(o) for o in obj], [inject(d) for d in dlt]
    got = rpn.decode_heads(obj, dlt)
    want = rpn.decode_heads([o.float() for o in obj], [d.float() for d in dlt])
    assert_same(got[0], want[0], "logits")
    assert_same(got[1], want[1], "boxes")
    # YOLO
    S, B, Cy = ri(2, 9), ri(1, 3), ri(1, 32)
    if S * S * B * Cy > 4096:
        Cy = max(1, 4096 // (S * S * B))
    yh = det.YoloGridHead(S, B, Cy, (32 * ri(4, 16), 32 * ri(4, 16)), clip=bool(ri(0, 1)))
    head = inject((torch.randn(ri(1, 12), S, S, B * 5 + Cy, generator=g) * rf(0.3, 2.5)).to(dt)).cuda()
    thr_y, mode, iou_y, md = rf(0.05, 0.5), ri(0, 2), rf(0.2, 0.8), ri(1, 300)
    yolo_same(yh.detect(head, thr_y, iou_y, max_det=md, return_dense=True, mode=mode),
              yh.detect(head.float(), thr_y, iou_y, max_det=md, return_dense=True, mode=mode), dense=True)


# ------------------------------------------------------------------------------------------------ CPU
def test_typed_entry_points_reject_unknown_dtype_without_gpu():
    """an unknown head_dtype is refused with DET_ERR_BAD_ARG and a message before any CUDA call"""
    from det_b200 import _native as N
    null = ctypes.c_void_p(0)
    err = N.fn("det_last_error")
    for bad in (3, -1, 7):
        assert N.fn("det_dense_decode_typed")(null, 1, 2, 3, 80, 4.0, null, null, null, 100, bad, null) == -1
        assert b"head_dtype" in err()
        assert N.fn("det_dense_detect_typed")(null, 1, 2, 3, 80, 4.0, 0.1, 0.5, 0, 1, 1024, 300, null, null, null, null,
                                              null, null, null, 0, bad, null) == -1
        assert b"head_dtype" in err()
        assert N.fn("det_rpn_decode_typed")(null, 1, 2, 3, 0.0, 1.0, 1.0, 1.0, 1.0, 4.0, null, null, 100, bad, null) == -1
        assert b"head_dtype" in err()
        assert N.fn("det_yolo_decode_nms_typed")(null, bad, 2, 7, 2, 20, 448, 448, null, 4.0, 1, 0.25, 0.5, 0, null,
                                                 null, null, 300, null, 8, null, null, null, null) == -1
        assert b"head_dtype" in err()
    assert N.fn("det_yolo_decode_nms_typed")(null, 0, 2, 7, 2, 20, 448, 448, null, 4.0, 1, 0.25, 0.5, 0, null, null, null,
                                             300, null, 2, null, null, null, null) == -1
    assert b"index_bytes" in err()
    # the known codes pass the dtype check and stop at the next argument check (n = 0 / null pointers), no CUDA call
    for code in (0, 1, 2):
        assert N.fn("det_dense_decode_typed")(null, 1, 0, 3, 80, 4.0, null, null, null, 100, code, null) == 0
        assert N.fn("det_rpn_decode_typed")(null, 0, 2, 3, 0.0, 1.0, 1.0, 1.0, 1.0, 4.0, null, null, 100, code, null) == 0


def test_heads_c_routing_without_gpu():
    """fp32 / bf16 / fp16 lists that share a dtype stay in it; fp64 and mixed lists go through f32c (code 0)"""
    from det_b200 import _native as N
    base = torch.randn(2, 6, 4, 4)
    for dt, code in ((torch.float32, 0), (torch.bfloat16, 1), (torch.float16, 2)):
        t = base.to(dt)
        out, c = N.heads_c([t, t[:1]])
        assert c == code and all(o.dtype == dt for o in out)
        assert out[0].data_ptr() == t.data_ptr()                      # aligned and contiguous: no copy
        nc = t.transpose(2, 3)
        (o,), c = N.heads_c([nc])
        assert c == code and o.is_contiguous() and torch.equal(o, nc)
        buf = torch.zeros(t.numel() + 1, dtype=dt)
        view = buf[1:].view(t.shape)                                  # contiguous, not 16-byte aligned
        (o,), c = N.heads_c([view])
        assert c == code and o.data_ptr() % 16 == 0 and torch.equal(o, view)
    out, c = N.heads_c([base.double()])
    assert c == 0 and out[0].dtype == torch.float32
    for mixed in ([base.bfloat16(), base.half()], [base, base.bfloat16()], [base.half(), base.double()]):
        out, c = N.heads_c(mixed)
        assert c == 0 and all(o.dtype == torch.float32 and o.data_ptr() % 16 == 0 for o in out)
        assert all(torch.equal(o, m.float()) for o, m in zip(out, mixed))
