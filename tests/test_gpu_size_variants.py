"""GPU parity for the kernel variants that only production-sized inputs select: ROIAlign channel groups and its direct
(untabulated) path, the YOLO loss's direct kernel and multi-image shared-memory tile, the RPN loss's grid-stride loop,
the generic IoU matcher with several images per CTA and more than one chunk of gt boxes in pass 2, and the RPN
proposal path's multi-tile sorts and rekey / pad / sort / emit finish.

Every test first restates the launcher's selection arithmetic (a small helper naming the source line) and asserts that
its inputs reach the variant, so that retuning a constant makes the test fail instead of quietly covering the other
path.  The SM count comes from det_sm_count, as the launchers read it.  Oracles: torchvision's CPU roi_align and
oracle/ref_torch.py."""
import math
import os

import pytest
import torch
import torchvision

from tests.test_gpu_roi_pool import ref_levels, ref_pooler
from tests.util import gen, rand_boxes

pytestmark = pytest.mark.gpu

STRIDES = [4, 8, 16, 32, 64]
SIZES = [[32], [64], [128], [256], [512]]
RATIOS = [[0.5, 1.0, 2.0]]


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


@pytest.fixture(scope="module")
def O():
    from oracle import ref_torch
    return ref_torch


@pytest.fixture(scope="module")
def sms(det):
    n = det._native.fn("det_sm_count")()
    assert n > 0, det._native.fn("det_last_error")()
    return n


# ---------------------------------------------------------------------------------------------------------------------
# ROIAlign (csrc/roi_pool.cu)
# ---------------------------------------------------------------------------------------------------------------------
ROI_CHANS = 32   # kRoiChans, roi_pool.cu:74: channels per CTA (grid.y = channel groups, roi_pool.cu:299,331)
ROI_TAPS = 128   # kRoiTaps, roi_pool.cu:75: per-axis taps a CTA tabulates in shared memory


def roi_channel_groups(c):
    """grid.y of det_roi_align_levels / _backward (roi_pool.cu:299,331)"""
    return (c + ROI_CHANS - 1) // ROI_CHANS


def roi_tabulated(rois, scale, out_size, sampling_ratio, aligned):
    """Per box: True when the kernels tabulate its taps, False when they take the direct path.  Restates the fp32
    arithmetic of roi_pool.cu:110-124 (forward) and :197-211 (backward)."""
    b = rois[:, 1:5].to(torch.float32)
    off = 0.5 if aligned else 0.0
    x1, y1 = b[:, 0] * scale - off, b[:, 1] * scale - off
    rw, rh = (b[:, 2] * scale - off) - x1, (b[:, 3] * scale - off) - y1
    if not aligned:
        rw, rh = rw.clamp(min=1.0), rh.clamp(min=1.0)
    oh, ow = out_size
    if sampling_ratio > 0:
        gh = gw = torch.full((b.shape[0],), sampling_ratio, dtype=torch.int64)
    else:
        gh, gw = torch.ceil(rh / oh).to(torch.int64), torch.ceil(rw / ow).to(torch.int64)
    return (gh >= 0) & (gw >= 0) & (oh * gh <= ROI_TAPS) & (ow * gw <= ROI_TAPS)


def _box_batch(g, m, n_img, lo, hi, frame_hw, spill=0.15):
    """(m,5) rois (batch index, x0, y0, x1, y1): sides log-uniform in [lo, hi] image pixels, aspect up to ~3:1, centres
    up to `spill` of the frame outside it, so many boxes are partly outside the feature map."""
    fh, fw = frame_hw
    sz = torch.exp(torch.rand(m, generator=g) * math.log(hi / lo)) * lo
    ar = torch.exp((torch.rand(m, generator=g) - 0.5) * 2.2)
    w, h = (sz * torch.sqrt(ar)).clamp(lo, hi), (sz / torch.sqrt(ar)).clamp(lo, hi)
    cx = (torch.rand(m, generator=g) * (1 + 2 * spill) - spill) * fw
    cy = (torch.rand(m, generator=g) * (1 + 2 * spill) - spill) * fh
    bi = torch.randint(0, n_img, (m,), generator=g).float()
    return torch.stack((bi, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2), 1)


def _check_roi_align(det, feat, rois, out_size, scale, sampling_ratio, aligned, g):
    """det.ROIAlign forward and backward against torchvision's CPU roi_align (and autograd through it)."""
    weight = torch.randn((rois.shape[0], feat.shape[1]) + tuple(out_size), generator=g)
    cf = feat.clone().requires_grad_(True)
    want = torchvision.ops.roi_align(cf, rois, out_size, scale, sampling_ratio, aligned)
    (want * weight).sum().backward()
    gf = feat.cuda().requires_grad_(True)
    got = det.ROIAlign(out_size, scale, sampling_ratio, aligned)(gf, rois.cuda())
    (got * weight.cuda()).sum().backward()
    torch.testing.assert_close(got.detach().cpu(), want.detach(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(gf.grad.cpu(), cf.grad, rtol=1e-4, atol=1e-5)
    return want.detach(), cf.grad


@pytest.mark.parametrize("C,ptype,sampling_ratio", [(256, "ROIAlignV2", 0), (33, "ROIAlign", 2)])
def test_roi_pooler_channel_groups(det, C, ptype, sampling_ratio):
    """C = 256 (the reference FPN width: 8 channel groups) and C = 33 (a last group of one channel): forward, and the
    gradient of every pyramid level, against torchvision's CPU roi_align driven by the reference's per-level loop."""
    groups = roi_channel_groups(C)
    assert groups >= 2
    if C == 33:
        assert C - (groups - 1) * ROI_CHANS == 1
    g = gen(500 + C)
    n_img, frame = 2, 448.0
    scales = [1.0 / s for s in (4, 8, 16, 32)]
    feats = [torch.randn(n_img, C, int(frame * s), int(frame * s), generator=g) for s in scales]
    rois = _box_batch(g, 40 * n_img, n_img, 8.0, 700.0, (frame, frame))
    box_lists = [rois[rois[:, 0] == i, 1:].contiguous() for i in range(n_img)]
    lv = ref_levels(torch.cat(box_lists, 0), 2, 5)
    assert set(lv.tolist()) == {0, 1, 2, 3}                      # every level pools some boxes
    weight = torch.randn((lv.shape[0], C, 7, 7), generator=g)
    cpu_feats = [f.clone().requires_grad_(True) for f in feats]
    want = ref_pooler(cpu_feats, scales, box_lists, (7, 7), sampling_ratio, ptype == "ROIAlignV2", 2, 5)
    (want * weight).sum().backward()
    gpu_feats = [f.cuda().requires_grad_(True) for f in feats]
    got = det.ROIPooler(scales, sampling_ratio, 7, ptype)(gpu_feats, [det.Boxes(b.cuda()) for b in box_lists])
    (got * weight.cuda()).sum().backward()
    torch.testing.assert_close(got.detach().cpu(), want.detach(), rtol=1e-5, atol=1e-5)
    for gf, cf in zip(gpu_feats, cpu_feats):
        assert float(cf.grad[:, (groups - 1) * ROI_CHANS:].abs().max()) > 0   # the last group receives gradient
        torch.testing.assert_close(gf.grad.cpu(), cf.grad, rtol=1e-4, atol=1e-5)


# (out_size, sampling_ratio, box sides in image pixels, which path the boxes must take); feature map 96 x 128 at
# spatial scale 0.5 (a 192 x 256 image), 36 channels (two channel groups, the second of 4)
_DIRECT_CASES = {
    # sampling_ratio 0: a side of more than 128/7 feature pixels per bin -> more than 128 taps on that axis
    "adaptive_large": ((7, 7), 0, (270.0, 420.0), "direct"),
    # a fixed ratio straddling the boundary at 7x7: 7 * 18 = 126 taps (tabulated), 7 * 19 = 133 taps (direct)
    "ratio18": ((7, 7), 18, (20.0, 200.0), "tabulated"),
    "ratio19": ((7, 7), 19, (20.0, 200.0), "direct"),
    # one call, both kinds of box
    "mixed": ((7, 7), 0, (10.0, 420.0), "mixed"),
    # non-square output: 5 rows (direct above 128/5 feature pixels of height per bin), 9 columns (above 128/9)
    "non_square": ((5, 9), 0, (60.0, 420.0), "mixed"),
}


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("case", sorted(_DIRECT_CASES))
def test_roi_align_direct_path(det, case, aligned):
    """Boxes whose tap tables would not fit shared memory: the forward samples without tables and the backward
    recomputes each sample's taps.  Boxes partly outside the map, forward and gradients."""
    out_size, sr, (lo, hi), want_path = _DIRECT_CASES[case]
    g = gen(600 + sorted(_DIRECT_CASES).index(case) + (50 if aligned else 0))
    scale, n_img, C = 0.5, 2, 36
    feat = torch.randn(n_img, C, 96, 128, generator=g)
    rois = _box_batch(g, 24, n_img, lo, hi, (192.0, 256.0), spill=0.3)
    if case == "mixed":  # make sure of both kinds: one tall box, one small box
        rois[0, 1:] = torch.tensor([10.0, -40.0, 50.0, 300.0])
        rois[1, 1:] = torch.tensor([100.0, 80.0, 130.0, 110.0])
    tab = roi_tabulated(rois, scale, out_size, sr, aligned)
    if want_path == "direct":
        assert not bool(tab.any())
    elif want_path == "tabulated":
        assert bool(tab.all())
    else:
        assert bool(tab.any()) and not bool(tab.all())
    assert roi_channel_groups(C) == 2
    want, grad = _check_roi_align(det, feat, rois, out_size, scale, sr, aligned, g)
    assert float(want.abs().max()) > 0 and float(grad.abs().max()) > 0


@pytest.mark.parametrize("seed", list(range(int(os.environ.get("DET_STRESS_SEEDS", "12")))))
def test_roi_align_stress_random_shapes(det, seed):
    """Random ROIAlign problems: channels around the group size, output size, sampling ratio (adaptive, small, and the
    18 / 19 straddle), aligned, spatial scale, box sizes from a pixel to larger than the map, image count -- forward
    and gradients against torchvision's CPU roi_align."""
    g = gen(17000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    C = [1, 5, 31, 32, 33, 64, 70][ri(0, 6)]
    out_size = (ri(1, 9), ri(1, 9))
    sr = [0, 0, 0, 1, 2, 5, 15, 18, 19, 20][ri(0, 9)]
    aligned = bool(ri(0, 1))
    scale = [1.0, 0.5, 0.25][ri(0, 2)]
    n_img = ri(1, 3)
    fh, fw = ri(8, 96), ri(8, 96)
    feat = torch.randn(n_img, C, fh, fw, generator=g)
    frame = (fh / scale, fw / scale)
    rois = _box_batch(g, ri(1, 8) * n_img, n_img, 1.0, min(400.0 / scale, 2.5 * max(frame)), frame, spill=0.25)
    if ri(0, 1) == 0:
        rois[-1, 4] = rois[-1, 2] + 150.0 / scale  # 150 feature pixels tall: direct unless a small sampling ratio
    if ri(0, 3) == 0:
        rois[0, 3:5] = rois[0, 1:3] - 2.0  # an inverted box
    _check_roi_align(det, feat, rois, out_size, scale, sr, aligned, g)


# ---------------------------------------------------------------------------------------------------------------------
# YOLO grid loss (csrc/assign_loss.cu, yolo_loss_impl)
# ---------------------------------------------------------------------------------------------------------------------
YOLO_LOSS_TILE = 5888  # kYoloLossTile, assign_loss.cu:921: floats of head staged per CTA


def yolo_loss_plan(n, S, B, C, sms):
    """The launch yolo_loss_impl chooses (assign_loss.cu:1258-1270): the direct kernel when one image's head exceeds the
    tile, else the tile kernel with `imgs` images per CTA; the last CTA holds `last` images and stages them with 16-byte
    loads only if its base and length are multiples of 4 floats (assign_loss.cu:938-943)."""
    per_img = S * S * (B * 5 + C)
    if per_img > YOLO_LOSS_TILE:
        return {"kernel": "direct", "per_img": per_img}
    imgs = YOLO_LOSS_TILE // per_img
    fill = (n + 2 * sms - 1) // (2 * sms)
    if imgs > fill:
        imgs = max(fill, 1)
    ctas = (n + imgs - 1) // imgs
    last = n - (ctas - 1) * imgs
    vec = lambda i0, k: (i0 * per_img) % 4 == 0 and (k * per_img) % 4 == 0
    return {"kernel": "tile", "per_img": per_img, "imgs": imgs, "tile_imgs": YOLO_LOSS_TILE // per_img, "ctas": ctas,
            "last": last, "full_vec": vec(0, imgs) and (ctas < 3 or vec(imgs, imgs)), "last_vec": vec((ctas - 1) * imgs, last)}


def _yolo_gts(n, g, hw, C, gmax=12):
    """Boxes inside an H x W image (every fifth image from the second on has no gt) and their classes."""
    H, W = hw
    boxes, classes = [], []
    for i in range(n):
        k = 0 if i % 5 == 1 else int(torch.randint(1, gmax + 1, (1,), generator=g))
        xy = torch.rand(k, 2, generator=g) * torch.tensor([0.85 * W, 0.85 * H])
        wh = torch.rand(k, 2, generator=g) * torch.tensor([0.35 * W, 0.35 * H]) + 4.0
        boxes.append(torch.cat([xy, torch.minimum(xy + wh, torch.tensor([float(W), float(H)]))], 1))
        classes.append(torch.randint(0, C, (k,), generator=g))
    return boxes, classes


@pytest.mark.parametrize("variant", ["direct", "tile"])
def test_yolo_loss_size_variants(det, O, sms, variant):
    """direct: S = 13, B = 3, C = 80 (16 055 floats per image, more than the tile).  tile: 7x7x30 at n = 6 * SMs + 1, so
    CTAs hold as many images as the tile does and the last CTA holds one, staged without vector loads.  A rectangular
    image (stride_x != stride_y), non-default lambdas, images without gt and an explicit normaliser; the autograd path
    with a non-unit upstream (0.5 loc + 2 obj + 3 cls) and the fused forward+backward launch.  The sums cover hundreds
    of images, so the losses are checked against the oracle run in float64."""
    hw = (384, 640)
    if variant == "direct":
        S, B, C, n = 13, 3, 80, 24
        plan = yolo_loss_plan(n, S, B, C, sms)
        assert plan["kernel"] == "direct" and plan["per_img"] == 16055
    else:
        S, B, C, n = 7, 2, 20, 6 * sms + 1
        plan = yolo_loss_plan(n, S, B, C, sms)
        assert plan["kernel"] == "tile" and plan["imgs"] >= 2 and plan["imgs"] == plan["tile_imgs"]
        assert plan["last"] == 1 and plan["full_vec"] and not plan["last_vec"]
    lc, ln, norm = 3.5, 0.25, 37.5
    g = gen(700 + S)
    yh = det.YoloGridHead(S, B, C, hw)
    tr = det.YoloGridTrainer(yh, lambda_coord=lc, lambda_noobj=ln)
    gts, gcls = _yolo_gts(n, g, hw, C)
    head = torch.randn(n, S, S, B * 5 + C, generator=g)
    anchors = O.yolo_grid_anchors(S, hw, yh.priors)
    wl, wi = O.label_anchors(anchors, gts)
    wl, wi = torch.stack(wl), torch.stack(wi)
    asg = tr.assign([b.cuda() for b in gts])
    assert torch.equal(asg.labels.cpu(), wl) and torch.equal(asg.matched.cpu(), wi)
    assert int((wl == 1).sum()) > n  # positives in most images
    with torch.no_grad():  # the sums: float64, so that only the kernel's rounding is measured
        want = O.yolo_loss(head.double(), wl, wi, [b.double() for b in gts], gcls, B, C, hw, yh.priors.double(), lc, ln,
                           norm)
    # per-element gradients (no long sums): autograd through the fp32 oracle, as test_yolo_assign_and_loss_vs_oracle
    hc = head.clone().requires_grad_(True)
    w32 = O.yolo_loss(hc, wl, wi, gts, gcls, B, C, hw, yh.priors, lc, ln, norm)
    g_up, = torch.autograd.grad(0.5 * w32["loc_loss"] + 2.0 * w32["obj_loss"] + 3.0 * w32["cls_loss"], hc,
                                retain_graph=True)
    g_one, = torch.autograd.grad(w32["loc_loss"] + w32["obj_loss"] + w32["cls_loss"], hc)
    gc = torch.cat(gcls).cuda()
    hg = head.cuda().requires_grad_(True)
    res = tr.loss(hg, asg, gc, normalizer=norm)
    (0.5 * res["loc_loss"] + 2.0 * res["obj_loss"] + 3.0 * res["cls_loss"]).backward()
    res2 = tr.loss(head.cuda(), asg, gc, normalizer=norm, with_grads=True)
    for r in (res, res2):
        for k in ("loc_loss", "obj_loss", "cls_loss"):
            torch.testing.assert_close(r[k].detach().cpu(), want[k].float(), rtol=1e-5, atol=1e-7)
        assert int(r["num_pos"]) == int((wl == 1).sum()) and int(r["num_neg"]) == int((wl == 0).sum())
    torch.testing.assert_close(hg.grad.cpu(), g_up, rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(res2["grad_head"].cpu(), g_one, rtol=1e-5, atol=1e-8)


# ---------------------------------------------------------------------------------------------------------------------
# RPN loss grid-stride loop (csrc/assign_loss.cu, det_rpn_loss)
# ---------------------------------------------------------------------------------------------------------------------
LOSS_THREADS = 256  # kLossThreads, assign_loss.cu:759
LOSS_GRID_FACTOR = 16  # kLossGridFactor, assign_loss.cu:1045: CTAs per SM of the loss grid


def rpn_loss_iterations(total, sms, factor):
    """Grid-stride iterations of the first warp of det_rpn_loss (assign_loss.cu:1195-1199, :793-795): a warp owns 128
    labels per iteration, the grid is capped at SMs * factor CTAs of 8 warps."""
    nwarps = (total + 127) // 128
    blocks = min((nwarps + LOSS_THREADS // 32 - 1) // (LOSS_THREADS // 32), sms * factor)
    return (nwarps + blocks * (LOSS_THREADS // 32) - 1) // (blocks * (LOSS_THREADS // 32))


RPN_LOSS_CONFIGS = [("smooth_l1", 0.0), ("smooth_l1", 0.11), ("giou", 0.0)]


@pytest.fixture(scope="module")
def rpn_big(O):
    """64 images x the 50 127 anchors of a 448 x 448 pyramid, labels before subsampling (dense: almost every label
    word has a non-ignored label), one image without gt; the oracle's sums in float64 and its gradients, per config."""
    g = gen(801)
    cells = [O.cell_anchors(s, RATIOS[0]) for s in SIZES]
    anc = torch.cat(O.grid_anchors([(448 // s, 448 // s) for s in STRIDES], STRIDES, cells, 0.0), 0)
    n = 64
    gts = []
    for i in range(n):
        k = 0 if i == 5 else int(torch.randint(1, 17, (1,), generator=g))
        b = rand_boxes(k, 448.0, g)
        b[:, 2:].clamp_(max=448.0)
        gts.append(b)
    labs, idxs = O.label_anchors(anc, gts)
    labels, matched = torch.stack(labs), torch.stack(idxs)
    mboxes = torch.stack([torch.zeros_like(anc) if len(b) == 0 else b[i] for b, i in zip(gts, idxs)])
    logits = torch.randn(n, anc.shape[0], generator=g)
    deltas = torch.randn(n, anc.shape[0], 4, generator=g) * 0.5
    case = {"anchors": anc, "gts": gts, "labels": labels, "matched": matched, "logits": logits, "deltas": deltas}
    oracle = {}
    for lt, beta in RPN_LOSS_CONFIGS:
        with torch.no_grad():
            w64 = O.rpn_losses(anc.double(), logits.double(), labels, deltas.double(), mboxes.double(),
                               box_reg_loss_type=lt, smooth_l1_beta=beta)
        lg, dl = logits.clone().requires_grad_(True), deltas.clone().requires_grad_(True)
        w = O.rpn_losses(anc, lg, labels, dl, mboxes, box_reg_loss_type=lt, smooth_l1_beta=beta)
        up = torch.autograd.grad(w["cls_loss"] + 2.0 * w["loc_loss"], (lg, dl), retain_graph=True)
        one = torch.autograd.grad(w["cls_loss"] + w["loc_loss"], (lg, dl))
        oracle[(lt, beta)] = {"cls": w64["cls_loss"].float(), "loc": w64["loc_loss"].float(), "num_pos": w64["num_pos"],
                              "num_neg": w64["num_neg"], "grad_up": up, "grad_one": one}
    case["oracle"] = oracle
    return case


def _rpn_asg(det, case):
    gts = case["gts"]
    table = torch.cat(gts, 0).cuda()
    off = torch.tensor([0] + [int(x) for x in torch.tensor([len(b) for b in gts]).cumsum(0)], dtype=torch.int32).cuda()
    return det.Assignment(case["labels"].cuda(), case["matched"].cuda(), table, off)


def _check_rpn_sums(cls, loc, npos, nneg, want, loss_type):
    torch.testing.assert_close(cls, want["cls"], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(loc, want["loc"], rtol=2e-5 if loss_type == "giou" else 1e-5, atol=1e-7)
    assert int(npos) == want["num_pos"] and int(nneg) == want["num_neg"]


def _check_rpn_grads(gl, gd, want, loss_type):
    torch.testing.assert_close(gl, want[0], rtol=1e-5, atol=1e-9)
    if loss_type == "giou":
        torch.testing.assert_close(gd, want[1], rtol=1e-4, atol=1e-8)
    else:
        torch.testing.assert_close(gd, want[1], rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize("loss_type,beta", RPN_LOSS_CONFIGS)
def test_rpn_loss_grid_stride_loop(det, O, sms, rpn_big, loss_type, beta):
    """n * R above SMs * 16 CTAs * 8 warps * 128 labels: warps walk more than one block of labels, prefetching the next
    label word while the current one is processed.  Losses, counts and both gradients against the oracle, through
    autograd (upstream 1 and 2) and through the fused forward+backward launch."""
    n, r = rpn_big["labels"].shape
    assert rpn_loss_iterations(n * r, sms, LOSS_GRID_FACTOR) >= 2
    want = rpn_big["oracle"][(loss_type, beta)]
    rpn = det.RegionProposalNetwork(STRIDES, SIZES, RATIOS, smooth_l1_beta=beta, box_reg_loss_type=loss_type)
    asg = _rpn_asg(det, rpn_big)
    anc = rpn_big["anchors"].cuda()
    glg = rpn_big["logits"].cuda().requires_grad_(True)
    gdl = rpn_big["deltas"].cuda().requires_grad_(True)
    res = rpn.fused_losses(anc, glg, gdl, asg)
    (res["cls_loss"] + 2.0 * res["loc_loss"]).backward()
    _check_rpn_sums(res["cls_loss"].detach().cpu(), res["loc_loss"].detach().cpu(), res["num_pos_anchors"],
                    res["num_neg_anchors"], want, loss_type)
    _check_rpn_grads(glg.grad.cpu(), gdl.grad.cpu(), want["grad_up"], loss_type)
    res2 = rpn.fused_losses(anc, rpn_big["logits"].cuda(), rpn_big["deltas"].cuda(), asg, with_grads=True)
    _check_rpn_sums(res2["cls_loss"].cpu(), res2["loc_loss"].cpu(), res2["num_pos_anchors"], res2["num_neg_anchors"],
                    want, loss_type)
    _check_rpn_grads(res2["grad_logits"].cpu(), res2["grad_deltas"].cpu(), want["grad_one"], loss_type)


def test_rpn_loss_many_iterations_per_warp(det, sms, rpn_big):
    """The 64-image batch tiled 16 times: 1 024 images x 50 127 anchors (the training batch of DESIGN section 4), so
    every warp of the default grid walks tens of label blocks.  The normaliser batch_size_per_image * N grows with the
    batch, so the losses are the 64-image ones and 16 x every copy's gradients are the 64-image gradients, for
    smooth-L1 (beta 0 and 0.11) and GIoU through the fused forward+backward launch.  num_pos is compared exactly at
    16 x the 64-image count; num_neg (about 50 M) lies beyond fp32's exact integers, and each CTA's atomic add of its
    exact partial count into the fp32 accumulator (assign_loss.cu:849-852) rounds by at most 2 below 2^26."""
    copies = 16
    n, r = rpn_big["labels"].shape
    assert rpn_loss_iterations(copies * n * r, sms, LOSS_GRID_FACTOR) >= 16
    ctas = sms * LOSS_GRID_FACTOR
    assert copies * n * r > ctas * (LOSS_THREADS // 32) * 128  # the grid is at its cap: the bound below counts its CTAs
    assert copies * max(w["num_neg"] for w in rpn_big["oracle"].values()) < 2 ** 26
    asg = _rpn_asg(det, {"gts": rpn_big["gts"] * copies, "labels": rpn_big["labels"].cuda().repeat(copies, 1),
                         "matched": rpn_big["matched"].cuda().repeat(copies, 1)})
    anc = rpn_big["anchors"].cuda()
    logits = rpn_big["logits"].cuda().repeat(copies, 1)
    deltas = rpn_big["deltas"].cuda().repeat(copies, 1, 1)
    for lt, beta in RPN_LOSS_CONFIGS:
        want = rpn_big["oracle"][(lt, beta)]
        rpn = det.RegionProposalNetwork(STRIDES, SIZES, RATIOS, smooth_l1_beta=beta, box_reg_loss_type=lt)
        res = rpn.fused_losses(anc, logits, deltas, asg, with_grads=True)
        got_neg = int(res["num_neg_anchors"])
        assert abs(got_neg - copies * want["num_neg"]) <= 2 * ctas, (got_neg, copies * want["num_neg"])
        _check_rpn_sums(res["cls_loss"].cpu(), res["loc_loss"].cpu(), res["num_pos_anchors"], got_neg,
                        dict(want, num_pos=copies * want["num_pos"], num_neg=got_neg), lt)
        grad_one = tuple(w.cuda().expand(copies, *w.shape) for w in want["grad_one"])
        _check_rpn_grads(copies * res["grad_logits"].view(copies, n, r), copies * res["grad_deltas"].view(copies, n, r, 4),
                         grad_one, lt)


# ---------------------------------------------------------------------------------------------------------------------
# IoU matching (csrc/assign_loss.cu, det_match_anchors)
# ---------------------------------------------------------------------------------------------------------------------
MATCH_ANCHORS_PER_CTA = 256 * 4  # kMatchThreads * kMatchPerThread, assign_loss.cu:17-18
MATCH_IMGS = 8                   # kMatchImgs, assign_loss.cu:34
GT_CHUNK = 512                   # kGtChunk, assign_loss.cu:19: gt boxes pass 2 considers per round


def match_images_per_cta(n, r, sms):
    """`imgs` of det_match_anchors (assign_loss.cu:1094-1097)."""
    bx = (r + MATCH_ANCHORS_PER_CTA - 1) // MATCH_ANCHORS_PER_CTA
    return min(max((bx * n) // (sms * 16), 1), MATCH_IMGS)


@pytest.fixture(scope="module")
def match_big(det, O, sms):
    """A batch for which every CTA of det_match_anchors walks several images and the last grid row is partial, with an
    image without gt, an image with more than GT_CHUNK gt boxes and a gt box that overlaps no anchor."""
    rpn = det.RegionProposalNetwork(STRIDES, SIZES, RATIOS)
    hw = [(448 // s, 448 // s) for s in STRIDES]
    at = torch.cat(rpn.anchor_generator.grid_anchors(hw, torch.device("cuda")), 0)
    r = at.shape[0]
    bx = (r + MATCH_ANCHORS_PER_CTA - 1) // MATCH_ANCHORS_PER_CTA
    n = (4 * sms * 16 + bx - 1) // bx
    while n % match_images_per_cta(n, r, sms) == 0:
        n += 1
    g = gen(901)
    gts = []
    for i in range(n):
        k = int(torch.randint(1, 17, (1,), generator=g))
        b = rand_boxes(k, 448.0, g)
        b[:, 2:].clamp_(max=448.0)
        gts.append(b)
    gts[1] = torch.zeros(0, 4)                                                        # image without gt
    gts[2] = rand_boxes(600, 448.0, g, wh_frac=0.15)                                  # two chunks of gt boxes
    gts[3] = torch.cat([gts[3], torch.tensor([[-5000.0, -5000.0, -4900.0, -4900.0]])])  # overlaps no anchor
    gts[n - 1] = rand_boxes(530, 448.0, g, wh_frac=0.1)                               # in the partial last row
    return rpn, hw, at, n, gts


@pytest.mark.parametrize("lq", [True, False])
def test_match_anchors_several_images_per_cta(det, O, sms, match_big, lq):
    """Labels and matched indices bit-exact against pairwise_iou -> Matcher per image; the grid matcher
    (det_match_grid) on the same batch gives the same result unless it declines the layout."""
    rpn, hw, at, n, gts = match_big
    r = at.shape[0]
    imgs = match_images_per_cta(n, r, sms)
    assert imgs >= 2 and n % imgs != 0                      # several images per CTA, partial last row
    assert max(len(b) for b in gts) > GT_CHUNK and min(len(b) for b in gts) == 0
    wl, wi = O.label_anchors(at.cpu(), gts, allow_low_quality=lq)
    if lq:
        assert bool((wl[3] == 1).all())                     # row maximum 0 promotes every anchor of image 3
    m = det.Matcher([0.3, 0.7], [0, -1, 1], lq)
    dev_gts = [b.cuda() for b in gts]
    gi, gl, _, _ = m.match_boxes(dev_gts, at)
    for i in range(n):
        assert torch.equal(gl[i].cpu(), wl[i]), i
        assert torch.equal(gi[i].cpu(), wi[i]), i
    try:
        ri, rl, _, _ = m.match_boxes(dev_gts, at, grid=rpn.anchor_generator.grid_layout(hw))
    except det._native.DetError as e:
        assert "status -2" in str(e), str(e)                # DET_ERR_UNSUPPORTED
    else:
        assert torch.equal(ri, gi) and torch.equal(rl, gl)


# ---------------------------------------------------------------------------------------------------------------------
# RPN proposal selection for large pyramids (csrc/proposals.cu, det_rpn_proposals)
# ---------------------------------------------------------------------------------------------------------------------
RPN_TILE = 2048               # kTile, nms_large.cuh:16: keys of one shared-memory tile sort
RPN_FINISH_SMEM = 200 * 1024  # proposals.cu:755: shared memory the one-CTA finish kernel may stage kept keys in


def rpn_proposal_plan(level_sizes, pre, post):
    """The sort and the finish det_rpn_proposals launches.  Sort (proposals.cu:725-730): one tile sort per (image,
    level) while no level keeps more than kTile keys, else sort_rows (tile sort + merge passes).  Finish
    (proposals.cu:753-755): the one-CTA finish kernel while an image's kept keys, 8 bytes for each of at most
    min(size, pre, post) per level, fit 200 KB, else rekey / pad / sort_rows / emit."""
    kept_bytes = 8 * sum(min(s, pre, post) for s in level_sizes)
    return {"sort": "levels" if min(max(level_sizes), pre) <= RPN_TILE else "sort_rows",
            "finish": "kernel" if kept_bytes <= RPN_FINISH_SMEM else "rekey", "kept_bytes": kept_bytes}


def test_rpn_proposals_large_pyramid_sort_and_finish(det, O):
    """pre = post = 14 000 on a 448 x 448 pyramid: the select's keys go through sort_rows and the kept ones through
    rekey / pad / sort_rows / emit.  Quantised logits on the finest level (ties at its top-k cut), ragged image sizes,
    three images; kept boxes, logits and counts bit-exact against the oracle's find_top_rpn_proposals."""
    from tests.test_gpu_rpn import _heads, _oracle_decode
    n, img, pre, post = 3, 448, 14000, 14000
    g = gen(77)
    obj, dlt = _heads(n, img, g, 0.4)
    obj[0] = (obj[0] * 4).round() / 4
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, img)
    level_sizes = [a.shape[0] for a in anchors]
    assert level_sizes == [37632, 9408, 2352, 588, 147]
    plan = rpn_proposal_plan(level_sizes, pre, post)
    assert plan == {"sort": "sort_rows", "finish": "rekey", "kept_bytes": 211960}
    ranked = lg[0].sort(1, descending=True).values
    assert bool((ranked[:, pre - 1] == ranked[:, pre]).all())  # every image's finest-level cut splits equal logits
    sizes = [(448, 448), (430, 400), (448, 360)]
    want = O.find_top_rpn_proposals([p.clone() for p in props], lg, sizes, 0.7, pre, post, 0.0, False)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, 0.7, pre, post, 0.0,
                                     False)
    for i in range(n):
        wb, ws = want[i]
        assert len(got[i]) == wb.shape[0], (i, len(got[i]), wb.shape[0])
        assert torch.equal(got[i].objectness_logits.cpu(), ws), i
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), wb), i
