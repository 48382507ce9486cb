"""GPU parity: YOLO-grid fused decode+NMS and dense-head decode vs the oracle (own spec; unpinned by reference)."""
import pytest
import torch

from tests.util import gen, assert_boxes_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


@pytest.fixture(scope="module")
def O():
    from oracle import ref_torch
    return ref_torch


@pytest.mark.parametrize("n,seed,thr", [(16, 0, 0.25), (256, 1, 0.25), (256, 1, 0.2)])
def test_yolo_grid_decode_and_nms(det, O, n, seed, thr):
    """BASELINE.json configs[0]/[1]: 7x7x(2*5+20) head, 448x448, score thr 0.25, per-class NMS IoU 0.5."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(n, 7, 7, 30, generator=gen(seed))
    r = yh.detect(head.cuda(), thr, 0.5, return_dense=True)
    ob, oc, osc = O.yolo_decode(head, 2, 20, (448, 448), yh.priors)
    gb, gc, gs = r["dense_boxes"].cpu(), r["dense_conf"].cpu(), r["dense_scores"].cpu()
    # decode: fp32 within 1e-5 relative (transcendentals differ by a few ulp between CUDA and the CPU library)
    assert_boxes_close(gb, ob, rtol=1e-5)
    torch.testing.assert_close(gc, oc, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(gs, osc, rtol=1e-5, atol=1e-6)
    # NMS: bit-exact kept indices and counts on identical inputs (the GPU's own decoded values)
    cnt = r["count"].cpu()
    flat, kb, ks = r["flat"].cpu(), r["boxes"].cpu(), r["scores"].cpu()
    modes = set()
    for i in range(n):
        wf, wb, ws, wc = O.yolo_select_nms(gb[i], gs[i], thr, 0.5)
        modes.add(int((gs[i] > thr).sum()) <= 1000)
        k = int(cnt[i])
        assert k == wf.numel(), i
        assert torch.equal(flat[i, :k], wf), i
        assert torch.equal(kb[i, :k], wb) and torch.equal(ks[i, :k], ws)
    if thr < 0.25:
        assert modes == {True, False}  # both the offset-trick and the per-category branch were exercised


def test_yolo_grid_end_to_end_indices_match_full_oracle(det, O):
    """Kept (predictor,class) ids of the fused kernel vs the oracle run from the raw logits; the only admissible
    differences are knife-edge score/IoU comparisons moved by the few-ulp transcendental differences."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(64, 7, 7, 30, generator=gen(5))
    r = yh.detect(head.cuda(), 0.25, 0.5)
    ob, oc, osc = O.yolo_decode(head, 2, 20, (448, 448), yh.priors)
    same = 0
    for i in range(64):
        wf, _, _, _ = O.yolo_select_nms(ob[i], osc[i], 0.25, 0.5)
        k = int(r["count"][i])
        if k == wf.numel() and torch.equal(r["flat"][i, :k].cpu(), wf):
            same += 1
    assert same >= 62, same


def test_yolo_no_clip_and_other_shapes(det, O):
    yh = det.YoloGridHead(5, 3, 7, (320, 480), priors=[[30, 60], [100, 80], [200, 220]], clip=False)
    head = torch.randn(9, 5, 5, 22, generator=gen(8)) * 1.5
    r = yh.detect(head.cuda(), 0.1, 0.45, return_dense=True)
    ob, oc, osc = O.yolo_decode(head, 3, 7, (320, 480), yh.priors, clip=False)
    gb, gs = r["dense_boxes"].cpu(), r["dense_scores"].cpu()
    assert_boxes_close(gb, ob, rtol=1e-5)
    for i in range(9):
        wf, wb, ws, wc = O.yolo_select_nms(gb[i], gs[i], 0.1, 0.45)
        k = int(r["count"][i])
        assert k == wf.numel() and torch.equal(r["flat"][i, :k].cpu(), wf)


def test_yolo_max_det_and_empty(det, O):
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(4, 7, 7, 30, generator=gen(2))
    r = yh.detect(head.cuda(), 0.25, 0.5, max_det=10, return_dense=True)
    assert r["flat"].shape == (4, 10)
    for i in range(4):
        wf, _, _, _ = O.yolo_select_nms(r["dense_boxes"][i].cpu(), r["dense_scores"][i].cpu(), 0.25, 0.5, max_det=10)
        assert int(r["count"][i]) == wf.numel() and torch.equal(r["flat"][i, :wf.numel()].cpu(), wf)
    r = yh.detect(head.cuda(), 2.0, 0.5)  # nothing passes
    assert r["count"].cpu().tolist() == [0, 0, 0, 0]


@pytest.mark.parametrize("hw", [(20, 20), (7, 9)])
def test_dense_decode_level(det, O, hw):
    A, C, stride = 3, 80, 32
    wh = [[116.0, 90.0], [156.0, 198.0], [373.0, 326.0]]
    head = torch.randn(3, A * (5 + C), hw[0], hw[1], generator=gen(4))
    dh = det.DenseAnchorHead([stride], [wh], C)
    gb, gs, gc = dh.decode([head.cuda()])
    ob, os_, oc = O.dense_decode(head, A, C, stride, torch.tensor(wh))
    assert torch.equal(gc.cpu(), oc)
    assert_boxes_close(gb.cpu(), ob, rtol=1e-5)
    torch.testing.assert_close(gs.cpu(), os_, rtol=1e-5, atol=1e-6)


def test_dense_head_detect_three_levels(det, O):
    """BASELINE.json configs[3] geometry at reduced spatial size: 3 levels, A=3, C=80, all boxes to NMS."""
    C = 80
    strides = [8, 16, 32]
    wh = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]]
    g = gen(3)
    heads = [torch.randn(2, 3 * (5 + C), 160 // s, 160 // s, generator=g) for s in strides]
    dh = det.DenseAnchorHead(strides, wh, C)
    boxes, scores, classes, keep, cnt = dh.detect([h.cuda() for h in heads], 0.5)
    R = boxes.shape[1]
    assert R == 3 * (20 * 20 + 10 * 10 + 5 * 5)
    for i in range(2):
        want = O.batched_nms(boxes[i].cpu(), scores[i].cpu(), classes[i].cpu(), 0.5)
        assert int(cnt[i]) == want.numel() and torch.equal(keep[i, :want.numel()].cpu(), want)


# ---- warp-per-class fast path (csrc/yolo_fast.cuh): small clipped grids ---------------------------------------------
def _select_nms_forced(O, boxes, scores, thr, iou, max_det, mode):
    """yolo_select_nms with one branch of the reference's batched_nms forced (det_nms_batched's `mode`): 1 = per category
    (torchvision's vanilla loop), 2 = coordinate-offset trick.  Built from the oracle's own primitives."""
    C = scores.shape[1]
    pi, ci = torch.nonzero(scores > thr, as_tuple=True)
    cb, cs = boxes[pi].float(), scores[pi, ci]
    if cb.numel() == 0:
        keep = torch.empty((0,), dtype=torch.int64)
    elif mode == 2:
        span = cb.max() + torch.tensor(1).to(cb)
        keep = O.nms(cb + (ci.to(cb) * span)[:, None], cs, iou)
    else:
        hit = torch.zeros_like(cs, dtype=torch.bool)
        for c in torch.unique(ci):
            members = torch.nonzero(ci == c, as_tuple=True)[0]
            hit[members[O.nms(cb[members], cs[members], iou)]] = True
        kept = torch.nonzero(hit, as_tuple=True)[0]
        keep = kept[O.stable_desc_order(cs[kept])]
    if max_det is not None:
        keep = keep[:max_det]
    return (pi[keep] * C + ci[keep]), cb[keep], cs[keep], ci[keep]


def _check_detect(det, O, yh, head, thr, iou, max_det=None, mode=0):
    r = yh.detect(head.cuda(), thr, iou, max_det=max_det, return_dense=True, mode=mode)
    gb, gs = r["dense_boxes"].cpu(), r["dense_scores"].cpu()
    cnt, flat, kb, ks = r["count"].cpu(), r["flat"].cpu(), r["boxes"].cpu(), r["scores"].cpu()
    for i in range(head.shape[0]):
        if mode == 0:
            wf, wb, ws, _ = O.yolo_select_nms(gb[i], gs[i], thr, iou, max_det=max_det)
        else:
            wf, wb, ws, _ = _select_nms_forced(O, gb[i], gs[i], thr, iou, max_det, mode)
        k = int(cnt[i])
        assert k == wf.numel(), (i, k, wf.numel())
        assert torch.equal(flat[i, :k], wf), i
        assert torch.equal(kb[i, :k], wb, ) or bool((torch.isnan(kb[i, :k]) == torch.isnan(wb)).all())
        assert torch.equal(ks[i, :k], ws)
    return r


@pytest.mark.parametrize("S,B,C,hw,thr,iou,n", [
    (5, 3, 7, (320, 480), 0.1, 0.45, 9),      # odd sizes, rectangular image
    (8, 2, 32, (512, 512), 0.2, 0.5, 7),      # 128 predictors x 32 classes: the limits of the fast path
    (3, 1, 1, (96, 96), 0.0, 0.3, 5),         # single class, every predictor a candidate
    (7, 2, 20, (448, 448), 0.02, 0.6, 6),     # low threshold: ~98 candidates per class, per-category branch
    (7, 2, 20, (448, 448), 0.6, 0.2, 6),      # few candidates, aggressive suppression
    (2, 1, 3, (64, 64), 0.3, 0.5, 33),        # tiny
])
def test_yolo_fast_path_shapes(det, O, S, B, C, hw, thr, iou, n):
    yh = det.YoloGridHead(S, B, C, hw)
    head = torch.randn(n, S, S, B * 5 + C, generator=gen(S * 100 + C)) * 1.3
    _check_detect(det, O, yh, head, thr, iou)
    _check_detect(det, O, yh, head, thr, iou, max_det=5)


def test_yolo_fast_path_heavy_overlap(det, O):
    """Small w/h logits spread and centred boxes: long suppression chains inside every class."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448), priors=[[300, 300], [380, 380]])
    head = torch.randn(12, 7, 7, 30, generator=gen(77))
    head[..., 2:4] *= 0.05
    head[..., 7:9] *= 0.05
    r = _check_detect(det, O, yh, head, 0.2, 0.3)
    assert int(r["count"].max()) < 200  # most candidates really were suppressed


def test_yolo_fast_path_ties(det, O):
    """Identical logits in many cells -> exactly tied scores: order must be (score desc, predictor*C+class asc)."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(4, 7, 7, 30, generator=gen(5))
    head[:, :, :, 4] = 0.5    # same confidence everywhere
    head[:, :, :, 9] = 0.5
    head[:, :, :, 10:] = head[:, :1, :1, 10:]  # same class logits in every cell
    _check_detect(det, O, yh, head, 0.25, 0.5)
    _check_detect(det, O, yh, head, 0.25, 0.5, max_det=40)


def test_yolo_fast_path_nonfinite_logits(det, O):
    """NaN / Inf logits: NaN boxes make the offset-trick branch non-separable -> the kernel's slow exact path."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    head = torch.randn(6, 7, 7, 30, generator=gen(9))
    head[0, 3, 3, 2] = float("nan")      # NaN width of one predictor
    head[1, 0, 0, 0] = float("inf")      # sigmoid(inf) = 1: finite box
    head[2, 6, 6, 7] = float("-inf")     # exp(-inf) = 0 width
    head[3, 2, 2, 4] = float("nan")      # NaN confidence: its scores are NaN and never pass the threshold
    head[4, 1, 5, 12] = float("nan")     # NaN class probability
    head[5] *= 0.4                        # fewer candidates (<= 1000): offset-trick branch ...
    head[5, 4, 4, 3] = float("nan")      # ... with a NaN box
    _check_detect(det, O, yh, head, 0.25, 0.5, max_det=300)
    _check_detect(det, O, yh, head, 0.35, 0.5)


@pytest.mark.parametrize("use_graph,index_dtype", [(True, torch.int64), (False, torch.int64), (True, torch.int32)])
def test_yolo_host_pipeline_matches_detect(det, O, use_graph, index_dtype):
    """The serving pipeline (pinned host in -> H2D -> fused kernel -> D2H -> pinned host out, one slot per stream)
    returns exactly what detect() returns, for every slot and across slot reuse."""
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    pipe = det.YoloHostPipeline(yh, 32, 0.25, 0.5, 300, depth=3, use_graph=use_graph, index_dtype=index_dtype)
    heads = torch.randn(7, 32, 7, 7, 30, generator=gen(21))
    got = []
    for i in range(7):
        slot = i % 3
        if i >= 3:
            got.append({k: v.clone() for k, v in pipe.wait(slot).items() if isinstance(v, torch.Tensor)})
        pipe.input(slot).copy_(heads[i])
        pipe.launch(slot)
    for i in range(4, 7):
        got.append({k: v.clone() for k, v in pipe.wait(i % 3).items() if isinstance(v, torch.Tensor)})
    assert len(got) == 7
    for i in range(7):
        r = yh.detect(heads[i].cuda(), 0.25, 0.5, max_det=300)
        cnt = r["count"].cpu()
        assert torch.equal(got[i]["count"], cnt)
        for j in range(32):
            k = int(cnt[j])
            assert got[i]["flat"].dtype == index_dtype
            assert torch.equal(got[i]["flat"][j, :k].long(), r["flat"][j, :k].cpu())
            assert torch.equal(got[i]["boxes"][j, :k], r["boxes"][j, :k].cpu())
            assert torch.equal(got[i]["scores"][j, :k], r["scores"][j, :k].cpu())
    # and against the oracle for one batch
    r = pipe.run(heads[0])
    d = yh.detect(heads[0].cuda(), 0.25, 0.5, return_dense=True)
    for j in range(0, 32, 5):
        wf, _, _, _ = O.yolo_select_nms(d["dense_boxes"][j].cpu(), d["dense_scores"][j].cpu(), 0.25, 0.5, max_det=300)
        assert int(r["count"][j]) == wf.numel() and torch.equal(r["flat"][j, :wf.numel()].long(), wf)


@pytest.mark.parametrize("n,C,sizes", [
    (3, 80, [(24, 24), (12, 12), (6, 6)]),     # every level a multiple of 4 positions: the bulk-copy pipeline
    (2, 80, [(80, 80), (40, 40), (20, 20)]),   # BASELINE configs[3] geometry (640 px)
    (5, 7, [(16, 12), (2, 2)]),                # few classes, tiny levels, odd class count
    (2, 1, [(8, 8)]),                          # single class
    (2, 80, [(20, 20), (10, 10), (5, 5)]),     # 25 positions: the last level reads scalar; a stray write hits image 1
    (2, 80, [(7, 9), (13, 13), (20, 20)]),     # scalar levels first: arg-max corner cases and the partial last group
])
def test_dense_decode_all_levels_one_launch(det, O, n, C, sizes):
    """det_dense_decode (one persistent launch, csrc/dense_decode.cu) vs the oracle, level by level.  Levels whose h*w
    is not a multiple of 4 ride in the same launch with scalar loads; the rows after each such level (the next level's,
    or the next image's) show a write past its last position."""
    A = 3
    strides = [8, 16, 32][:len(sizes)]
    wh = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]][:len(sizes)]
    g = gen(11)
    heads = [torch.randn(n, A * (5 + C), h, w, generator=g) * 2 for (h, w) in sizes]
    # arg-max corner cases: NaN class logit (NaN wins, first NaN), all -inf, exact ties (first maximum wins)
    v = heads[0].view(n, A, 5 + C, *sizes[0])
    v[0, 0, 5 + C // 2, 0, 0] = float("nan")
    v[0, 1, 5:, 0, 1] = float("-inf")
    v[0, 2, 5:, 1, 0] = 0.25
    if C > 3:
        v[0, 0, 5 + 1, 1, 1] = float("nan")
        v[0, 0, 5 + 3, 1, 1] = float("nan")
    dh = det.DenseAnchorHead(strides, wh, C)
    gb, gs, gc = dh.decode([h.cuda() for h in heads])
    off = 0
    for h, s, a in zip(heads, strides, wh):
        ob, os_, oc = O.dense_decode(h, A, C, s, torch.tensor(a, dtype=torch.float32))
        r = ob.shape[1]
        assert torch.equal(gc[:, off:off + r].cpu(), oc)
        assert_boxes_close(gb[:, off:off + r].cpu(), ob, rtol=1e-5)
        torch.testing.assert_close(gs[:, off:off + r].cpu(), os_, rtol=1e-5, atol=1e-6, equal_nan=True)
        off += r
    assert off == gb.shape[1]


@pytest.mark.parametrize("seed", list(range(int(__import__("os").environ.get("DET_STRESS_SEEDS", "16")))))
def test_yolo_fused_kernel_stress_random_shapes(det, O, seed):
    """Random grid shapes (fast path and generic kernel), logit scales, thresholds, max_det, clip on/off, NMS branch forced or
    automatic, occasional ties and non-finite logits: kept ids, counts, boxes and scores bit-exact against the oracle NMS on
    the GPU's own decoded values (every tier of the tier cut, the slow exact path and the merge are hit across the seeds)."""
    g = gen(7000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    rf = lambda lo, hi: float(torch.rand(1, generator=g)) * (hi - lo) + lo
    S, B = ri(1, 9), ri(1, 3)
    C = [1, 3, 20, 32, 7][ri(0, 4)]
    if S * S * B * C > 4096:
        C = max(1, 4096 // (S * S * B))
    hw = (32 * ri(2, 16), 32 * ri(2, 16))
    clip = ri(0, 3) > 0
    yh = det.YoloGridHead(S, B, C, hw, clip=clip)
    n = ri(1, 12)
    head = torch.randn(n, S, S, B * 5 + C, generator=g) * rf(0.3, 2.5)
    head[..., 4::5][..., :B] += rf(-2.0, 2.0)                     # confidence bias: from nearly nothing to everything passing
    if ri(0, 3) == 0:                                             # ties: identical cells
        head[:, :, :, :] = head[:, :1, :1, :]
    if ri(0, 4) == 0:
        head.view(-1)[ri(0, head.numel() - 1)] = float("nan")
    if ri(0, 6) == 0:
        head.view(-1)[ri(0, head.numel() - 1)] = float("inf")
    thr, iou = rf(0.0, 0.6), rf(0.05, 0.9)
    max_det = [None, 1, 5, 50, 300][ri(0, 4)]
    _check_detect(det, O, yh, head, thr, iou, max_det=max_det, mode=ri(0, 2))
