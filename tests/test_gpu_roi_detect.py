"""Second-stage (Fast R-CNN box predictor) inference: det_roi_detect_typed / det_roi_decode_dense_typed
(csrc/roi_detect.cu) and det_b200.FastRCNNOutputs against tests/fast_rcnn_oracle.py fast_rcnn_inference_single_image
(own specification after detectron2's fast_rcnn_inference_single_image).  The oracle's elementwise steps run on the GPU
(torch's fp32 kernels: the same IEEE operations, expf included) and its selection and NMS on the CPU, so kept flat ids,
classes and counts must be equal and boxes and scores equal bit for bit.  The last tests need no GPU."""
import ctypes
import math

import pytest
import torch

from tests.util import gen

WEIGHTS = (10.0, 10.0, 5.0, 5.0)
CLAMP = math.log(1000.0 / 16)


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


@pytest.fixture(scope="module")
def O():
    from tests import fast_rcnn_oracle
    return fast_rcnn_oracle


def make_batch(counts, K, seed, agnostic=False, scale=2.0, bg=0.0, sizes=None, quant=None, dscale=1.0, hot=0):
    """Packed rows of a batch: logits (M, K+1), deltas (M, K*4) or (M, 4), proposals (M, 4) inside each image, and the
    per-image (h, w).  scale / bg set how many (row, class) pairs pass a threshold, `hot` classes get +6 in every row
    (~hot candidates per row); quant rounds the logits to a grid (ties); dscale scales the deltas (large values push
    boxes out of the frame)."""
    g = gen(seed)
    M = sum(counts)
    sizes = sizes or [(480 + 37 * i, 640 + 53 * i) for i in range(len(counts))]
    logits = torch.randn(M, K + 1, generator=g) * scale
    logits[:, K] += bg
    logits[:, :hot] += 6.0
    if quant is not None:
        logits = (logits / quant).round() * quant
    deltas = torch.randn(M, 4 if agnostic else 4 * K, generator=g) * dscale
    props = []
    for n, (h, w) in zip(counts, sizes):
        xy = torch.rand(n, 2, generator=g) * torch.tensor([w * 0.9, h * 0.9])
        wh = 8.0 + torch.rand(n, 2, generator=g) * torch.tensor([w * 0.4, h * 0.4])
        props.append(torch.cat([xy, xy + wh], 1))
    return logits, deltas, torch.cat(props, 0) if props else torch.zeros(0, 4), sizes


def offsets_of(counts):
    off = [0]
    for c in counts:
        off.append(off[-1] + c)
    return off


def run(det, K, logits, deltas, props, counts, sizes, thr=0.05, iou=0.5, topk=100, mode=0, agnostic=False, cap=4096,
        check=False, workspace=None, out=None):
    fr = det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP), thr, iou, topk, agnostic, cap, mode)
    off = torch.tensor(offsets_of(counts), dtype=torch.int32, device="cuda")
    sz = torch.tensor(sizes, dtype=torch.int32, device="cuda").reshape(-1, 2)
    return fr.inference_batched(logits.cuda(), deltas.cuda(), props.cuda(), off, sz, out=out, workspace=workspace,
                                check=check)


def check_against_oracle(O, r, logits, deltas, props, counts, sizes, thr=0.05, iou=0.5, topk=100, mode=0):
    off = offsets_of(counts)
    idx, gb, gs, gc, cnt = [r[k].cpu() for k in ("idx", "boxes", "scores", "classes", "count")]
    bits = lambda t: t.contiguous().view(torch.int32)
    for b in range(len(counts)):
        a, e = off[b], off[b + 1]
        wi, wb, ws, wc = O.fast_rcnn_inference_single_image(logits[a:e].cuda(), deltas[a:e].cuda(), props[a:e].cuda(),
                                                            sizes[b], WEIGHTS, CLAMP, thr, iou, topk, mode)
        k = wi.numel()
        assert int(cnt[b]) == k, (b, int(cnt[b]), k)
        assert torch.equal(idx[b, :k], wi), b
        assert torch.equal(gc[b, :k], wc), b
        assert torch.equal(bits(gb[b, :k]), bits(wb)) and torch.equal(bits(gs[b, :k]), bits(ws)), b
    return cnt


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 20, 80, 130])  # 130: more classes than the register path holds
@pytest.mark.parametrize("agnostic", [False, True])
@pytest.mark.parametrize("scale,bg", [(2.0, 3.0), (2.0, 0.0), (1.0, -4.0)])  # low, medium, high pass rates
def test_roi_detect_parity(det, O, K, agnostic, scale, bg):
    counts = [300, 0, 171, 257]  # an empty image; K + 1 = 81 / 21 / 131 logits: pitches that are not 16-byte multiples
    logits, deltas, props, sizes = make_batch(counts, K, 100 + K + int(agnostic), agnostic, scale, bg)
    r = run(det, K, logits, deltas, props, counts, sizes, agnostic=agnostic)
    assert int(r["overflow"].item()) == 0
    cnt = check_against_oracle(O, r, logits, deltas, props, counts, sizes)
    assert int(cnt[1]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("topk", [-1, 100, 7])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_roi_detect_topk_and_modes(det, O, topk, mode):
    K = 20
    counts = [400, 90, 333]  # ~1000+ candidates on the first image, a few hundred on the others: both AUTO branches
    logits, deltas, props, sizes = make_batch(counts, K, 7, scale=2.5, bg=-1.0)
    r = run(det, K, logits, deltas, props, counts, sizes, thr=0.05, iou=0.4, topk=topk, mode=mode)
    assert int(r["overflow"].item()) == 0
    check_against_oracle(O, r, logits, deltas, props, counts, sizes, 0.05, 0.4, topk, mode)


@pytest.mark.gpu
def test_roi_detect_vector_rows_and_iou_extremes(det, O):
    """K = 3 and K = 151: K + 1 = 4 / 152 logits per row (151: the general path's 16-byte logit loads); IoU thresholds
    from 0.05 to 0.9."""
    for K in (3, 151):
        counts = [250, 300]
        logits, deltas, props, sizes = make_batch(counts, K, 40 + K, scale=1.5, bg=-1.0)
        for iou in (0.05, 0.9):
            r = run(det, K, logits, deltas, props, counts, sizes, thr=0.1, iou=iou, topk=-1)
            check_against_oracle(O, r, logits, deltas, props, counts, sizes, 0.1, iou, -1)


@pytest.mark.gpu
def test_roi_detect_nonfinite_rows_are_dropped(det, O):
    """NaN / Inf in logits or deltas drops exactly that row; idx keeps the ORIGINAL row numbering."""
    K = 20
    counts = [120, 80]
    logits, deltas, props, sizes = make_batch(counts, K, 3, scale=2.0, bg=-2.0)
    logits[5, 3] = float("nan")
    logits[9, K] = float("inf")     # +inf logit: inf - inf in the softmax, NaN probabilities
    logits[11, 0] = float("-inf")   # -inf logit: probability 0, the row stays valid
    deltas[17, 4 * 7 + 0] = float("inf")  # an infinite centre: a non-finite box (an infinite dw would be clamped)
    deltas[18, 4 * 9 + 2] = float("inf")  # clamped by scale_clamp: a finite box, the row stays
    deltas[130, 1] = float("nan")
    deltas[131, 4 * 19 + 3] = 1e30  # clamped by scale_clamp: a finite box
    r = run(det, K, logits, deltas, props, counts, sizes, topk=-1)
    check_against_oracle(O, r, logits, deltas, props, counts, sizes, topk=-1)
    rows0 = r["idx"][0, :int(r["count"][0])].cpu() // K
    rows1 = r["idx"][1, :int(r["count"][1])].cpu() // K
    for bad in (5, 9, 17):
        assert bad not in rows0.tolist()
    assert 10 not in rows1.tolist()
    assert rows0.max() > 17  # numbering did not shift: rows after the dropped ones keep their index


@pytest.mark.gpu
def test_roi_detect_ties_resolve_by_flat_id(det, O):
    """Quantised logits, and 40 rows with identical logits on different proposals: many exactly equal scores among the
    kept detections, decided by the lower flat id."""
    K = 20
    counts = [300, 200]
    logits, deltas, props, sizes = make_batch(counts, K, 13, scale=1.0, bg=-2.0, quant=0.5)
    logits[40:80] = logits[40]
    for topk in (30, -1):
        r = run(det, K, logits, deltas, props, counts, sizes, topk=topk)
        check_against_oracle(O, r, logits, deltas, props, counts, sizes, topk=topk)
    s = r["scores"][0, :int(r["count"][0])].cpu()
    assert (s[1:] == s[:-1]).any()  # ties really occur among the kept detections


@pytest.mark.gpu
def test_roi_detect_boxes_leaving_the_frame(det, O):
    """Large deltas push most boxes out of the frame; clipping happens before the NMS, and the clipped boxes of different
    classes share coordinates (0 and the image size): the offset-trick branch (<= 1000 candidates) and the
    per-category branch must agree with the oracle on the clipped coordinates."""
    K = 10
    counts = [200, 200, 600]
    logits, deltas, props, sizes = make_batch(counts, K, 21, scale=1.5, bg=-0.5, dscale=8.0)
    for mode in (0, 1, 2):
        r = run(det, K, logits, deltas, props, counts, sizes, iou=0.3, topk=-1, mode=mode)
        check_against_oracle(O, r, logits, deltas, props, counts, sizes, iou=0.3, topk=-1, mode=mode)
    b = r["boxes"][2, :int(r["count"][2])].cpu()
    assert bool((b[:, 0] == 0).any()) and bool((b[:, 2] == sizes[2][1]).any())


@pytest.mark.gpu
def test_roi_detect_overflow_reported_then_redone_exactly(det, O):
    K = 80
    counts = [500, 60, 700]
    logits, deltas, props, sizes = make_batch(counts, K, 5, scale=1.0, bg=-6.0, hot=8)  # ~8 candidates per row
    r = run(det, K, logits, deltas, props, counts, sizes, cap=512, check=False)
    cnt = r["count"].cpu()
    assert int(r["overflow"].item()) == 1 and int(cnt[0]) == -1 and int(cnt[1]) >= 0 and int(cnt[2]) == -1
    for topk in (100, -1):
        r = run(det, K, logits, deltas, props, counts, sizes, cap=512, check=True, topk=topk)
        check_against_oracle(O, r, logits, deltas, props, counts, sizes, topk=topk)


@pytest.mark.gpu
def test_roi_detect_dense_form(det, O):
    """det_roi_decode_dense_typed: probabilities and clipped boxes of every (row, class), NaN for invalid rows and for
    the padding rows, bit-identical to the oracle's decode."""
    import det_b200._native as N
    K = 20
    counts = [50, 0, 31]
    logits, deltas, props, sizes = make_batch(counts, K, 8)
    logits[3, 2] = float("nan")
    n, p_max = len(counts), 64
    lg, dl, pr = logits.cuda(), deltas.cuda(), props.cuda()
    off = torch.tensor(offsets_of(counts), dtype=torch.int32, device="cuda")
    sz = torch.tensor(sizes, dtype=torch.int32, device="cuda")
    scores = torch.zeros((n, p_max, K), device="cuda")
    boxes = torch.zeros((n, p_max, K, 4), device="cuda")
    N.call("det_roi_decode_dense_typed", N.ptr(lg), N.ptr(dl), 0, N.ptr(pr), N.ptr(off), n, lg.shape[0], K, 0, N.ptr(sz),
           *WEIGHTS, CLAMP, 0, p_max, N.ptr(scores), N.ptr(boxes), N.stream())
    bits = lambda t: t.contiguous().view(torch.int32)
    o = offsets_of(counts)
    for b in range(n):
        a, e = o[b], o[b + 1]
        probs, wb, valid = O.fast_rcnn_decode_single_image(lg[a:e], dl[a:e], pr[a:e], sizes[b], WEIGHTS, CLAMP)
        k = e - a
        want_s = torch.where(valid[:, None], probs[:, :K], float("nan"))
        want_b = torch.where(valid[:, None, None], wb, float("nan"))
        assert torch.equal(bits(scores[b, :k]), bits(want_s)) and torch.equal(bits(boxes[b, :k]), bits(want_b)), b
        assert bool(scores[b, k:].isnan().all()) and bool(boxes[b, k:].isnan().all())
    assert bool(scores[0, 3].isnan().all())


@pytest.mark.gpu
def test_roi_detect_owned_workspace_and_graph_replay(det, O):
    """DenseDetectWorkspace (gate bit 1): the counter block is zero after every call, an overflowing one included, and
    the call captures into a CUDA graph and replays to the same result."""
    import det_b200._native as N
    K = 80
    counts = [300, 250, 280]
    ws = det.DenseDetectWorkspace(3, 1024, "cuda:0")
    nctr = N.fn("det_roi_detect_counter_bytes")(3)
    batches = [make_batch(counts, K, 60 + j, scale=s, bg=bg, hot=hot)
               for j, (s, bg, hot) in enumerate(((1.0, 4.0, 0), (1.0, -6.0, 8), (1.5, 4.0, 0)))]
    out = None
    for j, (logits, deltas, props, sizes) in enumerate(batches):
        out = run(det, K, logits, deltas, props, counts, sizes, cap=1024, workspace=ws, out=out)
        assert int(ws.buf[:nctr].view(torch.int32).abs().sum()) == 0
        if j == 1:
            assert int(out["overflow"].item()) == 1
        else:
            assert int(out["overflow"].item()) == 0
            check_against_oracle(O, out, logits, deltas, props, counts, sizes)
    logits, deltas, props, sizes = batches[2]
    fr = det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP), cand_cap=1024)
    lg, dl, pr = logits.cuda(), deltas.cuda(), props.cuda()
    off = torch.tensor(offsets_of(counts), dtype=torch.int32, device="cuda")
    sz = torch.tensor(sizes, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fr.inference_batched(lg, dl, pr, off, sz, out=out, workspace=ws, check=False)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(st)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fr.inference_batched(lg, dl, pr, off, sz, out=out, workspace=ws, check=False)
    for k in out:
        if k != "overflow":
            out[k].fill_(-3)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    assert int(ws.buf[:nctr].view(torch.int32).abs().sum()) == 0
    check_against_oracle(O, out, logits, deltas, props, counts, sizes)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("agnostic", [False, True])
def test_roi_detect_16bit_rows_match_fp32(det, dtype, agnostic):
    K = 80
    counts = [333, 97, 410]
    logits, deltas, props, sizes = make_batch(counts, K, 90, agnostic, scale=2.0, bg=0.0)
    lo, de = logits.to(dtype), (deltas * 0.5).to(dtype)
    a = run(det, K, lo, de, props, counts, sizes, agnostic=agnostic)
    b = run(det, K, lo.float(), de.float(), props, counts, sizes, agnostic=agnostic)
    assert torch.equal(a["count"], b["count"]) and int(a["count"].min()) > 0
    for i in range(len(counts)):
        k = int(a["count"][i])
        for key in ("idx", "boxes", "scores", "classes"):
            assert torch.equal(a[key][i, :k], b[key][i, :k]), key
    # the overflow route reads 16-bit rows natively too
    c = run(det, K, lo, de, props, counts, sizes, agnostic=agnostic, cap=16, check=True)
    assert torch.equal(c["count"], b["count"])
    for i in range(len(counts)):
        k = int(c["count"][i])
        for key in ("idx", "boxes", "scores", "classes"):
            assert torch.equal(c[key][i, :k], b[key][i, :k]), key


@pytest.mark.gpu
def test_fast_rcnn_outputs_inference_on_instances(det, O):
    """detectron2's contract end to end: List[Instances] in, (List[Instances], List[kept proposal index]) out, equal to
    a per-image loop over the oracle."""
    K = 80
    counts = [200, 0, 150]
    logits, deltas, props, sizes = make_batch(counts, K, 31, scale=2.0, bg=0.0)
    fr = det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP), 0.05, 0.5, 100)
    off = offsets_of(counts)
    proposals = [det.Instances(sizes[b], proposal_boxes=det.Boxes(props[off[b]:off[b + 1]].cuda()))
                 for b in range(len(counts))]
    results, kept = fr.inference((logits.cuda(), deltas.cuda()), proposals)
    assert len(results) == len(kept) == len(counts)
    for b in range(len(counts)):
        a, e = off[b], off[b + 1]
        wi, wb, ws, wc = O.fast_rcnn_inference_single_image(logits[a:e].cuda(), deltas[a:e].cuda(), props[a:e].cuda(),
                                                            sizes[b], WEIGHTS, CLAMP, 0.05, 0.5, 100)
        res = results[b]
        assert res.image_size == tuple(sizes[b]) and len(res) == wi.numel()
        assert torch.equal(res.pred_boxes.tensor.cpu(), wb) and torch.equal(res.scores.cpu(), ws)
        assert torch.equal(res.pred_classes.cpu(), wc) and torch.equal(kept[b].cpu(), wi // K)


@pytest.mark.gpu
def test_fast_rcnn_inference_on_decoded_boxes(det, O):
    """fast_rcnn_inference over boxes and probabilities the caller decoded: the oracle's selection on the same values."""
    from oracle import ref_torch
    K = 20
    counts = [180, 90]
    logits, deltas, props, sizes = make_batch(counts, K, 17, scale=2.0, bg=-1.0)
    off = offsets_of(counts)
    boxes, scores = [], []
    for b in range(len(counts)):
        a, e = off[b], off[b + 1]
        probs = O.softmax_rows_sequential(logits[a:e])
        probs[3, 1] = float("nan") if b == 0 else probs[3, 1]
        scores.append(probs.cuda())
        boxes.append(ref_torch.apply_deltas(deltas[a:e], props[a:e], WEIGHTS, CLAMP).cuda() * 1.3)  # some leave the frame
    results, kept = det.fast_rcnn_inference(boxes, scores, sizes, 0.05, 0.5, 100)
    for b in range(len(counts)):
        P = counts[b]
        bx = boxes[b].cpu().reshape(P, K, 4)
        pr = scores[b].cpu()
        valid = torch.isfinite(bx).flatten(1).all(1) & torch.isfinite(pr).all(1)
        lim = torch.tensor([sizes[b][1], sizes[b][0]] * 2, dtype=torch.float32)
        bx = torch.where(bx < 0, torch.zeros(()), bx)
        bx = torch.where(bx > lim, lim, bx)
        wi, wb, ws, wc = O.fast_rcnn_select_single_image(pr, bx, valid, 0.05, 0.5, 100)
        assert torch.equal(kept[b].cpu(), wi // K) and torch.equal(results[b].pred_classes.cpu(), wc)
        assert torch.equal(results[b].pred_boxes.tensor.cpu(), wb) and torch.equal(results[b].scores.cpu(), ws)
    assert 3 not in kept[0].tolist()


# ---- no GPU needed -----------------------------------------------------------------------------------------------------
def test_oracle_softmax_sum_is_sequential():
    """The oracle's row sum is e[0] + e[1] + ... + e[K] in fp32, in that order: equal to a Python loop of fp32 additions.
    (CPU torch.cumsum(e, -1)[:, -1] is not that sum -- it accumulates in a wider type and rounds once -- which is why the
    oracle spells the loop out.)"""
    import numpy as np
    from tests import fast_rcnn_oracle as O
    g = gen(4)
    x = torch.randn(64, 81, generator=g) * 3
    x[7, 5] = float("-inf")
    p = O.softmax_rows_sequential(x)
    e = torch.exp(x - x.max(dim=1, keepdim=True).values)
    en = e.numpy()
    for r in range(x.shape[0]):
        s = np.float32(en[r, 0])
        for c in range(1, en.shape[1]):
            s = np.float32(s + en[r, c])
        assert torch.equal(p[r], e[r] / torch.tensor(s)), r


def test_roi_detect_queries_and_argument_checks_need_no_gpu():
    """Size queries and argument validation of det_roi_detect_typed / det_roi_decode_dense_typed: rejected before any
    CUDA call is made."""
    from det_b200 import _native as N
    wsb, ctr = N.fn("det_roi_detect_workspace_bytes"), N.fn("det_roi_detect_counter_bytes")
    assert wsb(8, 4096) == N.fn("det_dense_detect_workspace_bytes")(8, 4096) == 8 * 128 + 8 * 4096 * 28
    assert ctr(8) == 8 * 128 and ctr(0) == 0
    f = N.fn("det_roi_detect_typed")
    null = ctypes.c_void_p(0)

    def args(dtype=0, cap=4096, max_det=100, mode=0, K=80, m=1000):
        return (null, null, dtype, null, null, 4, m, K, 0, null, *WEIGHTS, CLAMP, 0.05, 0.5, mode, 2, cap, max_det,
                null, null, null, null, null, null, null, 0, null)
    assert f(*args(dtype=3)) == -1        # unknown dtype: DET_ERR_BAD_ARG
    assert b"head_dtype" in N.fn("det_last_error")()
    assert f(*args(cap=4097)) == -2       # cand_cap > 4096: DET_ERR_UNSUPPORTED
    assert f(*args(cap=0)) == -2
    assert f(*args(K=4097)) == -2         # num_classes beyond the limit
    assert f(*args(K=80, m=1 << 25)) == -2  # m * K >= 2^31: flat ids would not fit int32
    assert f(*args(max_det=0)) == -1
    assert f(*args(mode=3)) == -1
    assert f(*args()) == -1               # null outputs
    assert b"null output" in N.fn("det_last_error")()
    d = N.fn("det_roi_decode_dense_typed")
    assert d(null, null, 5, null, null, 2, 10, 80, 0, null, *WEIGHTS, CLAMP, 0, 8, null, null, null) == -1
    assert d(null, null, 0, null, null, 2, 10, 80, 0, null, *WEIGHTS, CLAMP, 0, 8, null, null, null) == -1
    assert d(null, null, 0, null, null, 2, 10, 80, 0, null, *WEIGHTS, CLAMP, 0, 0, null, null, null) == 0  # nothing to do
