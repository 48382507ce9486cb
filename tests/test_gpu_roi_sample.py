"""Batched ROI-head proposal sampling: det_roi_sample_proposals (csrc/roi_sample.cu) through
ROIHeads.sample_proposals_batched / label_and_sample_proposals_batched, against tests/roi_sample_oracle.py (the CPU
oracle's roi_label_proposals + subsample_counts, selection by the documented hash keys).  Rows, classes, matched
indices and counts are compared exactly and boxes bit for bit.  The last tests need no GPU."""
import ctypes

import pytest
import torch

from tests.util import gen, rand_boxes

K = 80
MATCHERS = {"plain": ([0.5], [0, 1], False), "lowq": ([0.4, 0.5], [0, -1, 1], True)}
KEYS = ("boxes", "gt_classes", "gt_boxes", "matched", "src")


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


@pytest.fixture(scope="module")
def OS():
    from tests import roi_sample_oracle
    return roi_sample_oracle


def heads(det, rule="plain", S=512, f=0.25, append=True):
    thr, lab, lq = MATCHERS[rule]
    return det.ROIHeads(K, S, f, det.Matcher(thr, lab, allow_low_quality_matches=lq), append)


def make_image(P, G, g, frame=800.0, nan_rows=0, zero_area_gt=False, dup_gt=0):
    """Proposals (P,4) with some near the gt boxes, gt (G,4) and classes (G,).  nan_rows proposals are NaN and as many
    are degenerate (zero width); dup_gt gt boxes repeat earlier ones (argmax ties); zero_area_gt makes gt 0 a point."""
    gt = rand_boxes(G, frame, g, 0.3)
    if dup_gt and G > dup_gt:
        gt[-dup_gt:] = gt[:dup_gt]
    if zero_area_gt and G:
        gt[0, 2:] = gt[0, :2]
    props = rand_boxes(P, frame, g, 0.3)
    k = min(P // 2, G)
    if k:
        props[:k] = gt[:k] + (torch.rand(k, 4, generator=g) - 0.5) * 12
    if nan_rows and P > 2 * nan_rows:
        props[-nan_rows:] = float("nan")
        props[-2 * nan_rows:-nan_rows, 2] = props[-2 * nan_rows:-nan_rows, 0]
    return props, gt, torch.randint(0, K, (G,), generator=g)


def batch(images, pad_value=float("nan")):
    """Device tensors of sample_proposals_batched for [(props, gt, classes), ...]: rows past each count are filled with
    pad_value (never read)."""
    p_stride = max(max(p.shape[0] for p, _, _ in images), 1)
    pb = torch.full((len(images), p_stride, 4), pad_value)
    for i, (p, _, _) in enumerate(images):
        pb[i, :p.shape[0]] = p
    counts = torch.tensor([p.shape[0] for p, _, _ in images], dtype=torch.int32)
    off = [0]
    for _, gt, _ in images:
        off.append(off[-1] + gt.shape[0])
    table = torch.cat([gt for _, gt, _ in images]).reshape(-1, 4)
    classes = torch.cat([c for _, _, c in images]).to(torch.int64)
    return (pb.cuda(), counts.cuda(), table.cuda(), torch.tensor(off, dtype=torch.int32).cuda(), classes.cuda())


def seed_t(s):
    return torch.tensor([s], dtype=torch.int64, device="cuda")


def check(OS, h, res, images, seed, rule="plain"):
    thr, lab, lq = MATCHERS[rule]
    S = h.batch_size_per_image
    res = {k: v.cpu() for k, v in res.items()}
    for i, (p, gt, c) in enumerate(images):
        want = OS.sample_image(p, gt, c, K, S, h.positive_fraction, seed, i, thr, lab, lq, h.proposal_append_gt)
        n = want["count"]
        assert int(res["count"][i]) == n and int(res["num_fg"][i]) == want["num_fg"], f"image {i}"
        for k in KEYS:
            got = res[k][i, :n]
            if got.dtype == torch.float32:
                assert torch.equal(got.view(torch.int32), want[k].contiguous().view(torch.int32)), f"image {i} {k}"
            else:
                assert torch.equal(got, want[k].to(got.dtype)), f"image {i} {k}"
        assert bool((res["src"][i, n:] == -1).all()) and bool((res["gt_classes"][i, n:] == -1).all())
        assert bool((res["matched"][i, n:] == -1).all())
        assert bool((res["boxes"][i, n:] == 0).all()) and bool((res["gt_boxes"][i, n:] == 0).all())
    under = any(int(res["count"][i]) < S for i in range(len(images)))
    assert int(res["underfull"][0]) == int(under)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["plain", "lowq"])
@pytest.mark.parametrize("append", [True, False])
@pytest.mark.parametrize("G", [0, 1, 7, 100, 1024])
def test_parity_with_oracle(det, OS, G, append, rule):
    """Images with P in {0, 1, 300, 2000, 4096 - G} proposals and G gt boxes (duplicates, a zero-area one under the
    low-quality rule, NaN and degenerate proposals, NaN padding past each count)."""
    g = gen(1000 + G)
    images = [make_image(P, G, g, nan_rows=3, dup_gt=2 if G > 4 else 0, zero_area_gt=(rule == "lowq" and i == 4))
              for i, P in enumerate([0, 1, 300, 2000, 4096 - G])]
    h = heads(det, rule, append=append)
    res = h.sample_proposals_batched(*batch(images), seed_t(77 + G))
    check(OS, h, res, images, 77 + G, rule)


@pytest.mark.gpu
@pytest.mark.parametrize("S,f", [(100, 0.29), (64, 0.5), (1, 1.0), (600, 0.0)])
def test_counts_and_underfull(det, OS, S, f):
    """S*f evaluated in double (100 * 0.29 -> 28), S above the candidate count (underfull), f at both ends."""
    g = gen(5)
    images = [make_image(P, G, g) for P, G in [(300, 20), (50, 60), (10, 0), (2000, 3)]]
    h = heads(det, "plain", S=S, f=f)
    res = h.sample_proposals_batched(*batch(images), seed_t(-12345))
    check(OS, h, res, images, -12345)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["plain", "lowq"])
def test_labels_equal_existing_matcher(det, rule):
    """With S >= P + G and f = 1 every labelled candidate comes back; its class and matched gt equal label_proposals
    (det_match_anchors) on the same image."""
    g = gen(9)
    images = [make_image(P, G, g, zero_area_gt=(i == 1)) for i, (P, G) in enumerate([(900, 30), (500, 12), (200, 0)])]
    h = heads(det, rule, S=2048, f=1.0)
    res = h.sample_proposals_batched(*batch(images), seed_t(3))
    for i, (p, gt, c) in enumerate(images):
        allp = torch.cat([p, gt]).cuda()
        mi, _, cls = h.label_proposals(allp, gt.cuda(), c.cuda())
        n = int(res["count"][i])
        src = res["src"][i, :n].long()
        assert n == int((cls != -1).sum())
        assert torch.equal(torch.sort(src).values, torch.nonzero(cls != -1)[:, 0])
        assert torch.equal(res["gt_classes"][i, :n], cls[src])
        if gt.shape[0]:
            assert torch.equal(res["matched"][i, :n].long(), mi[src])


@pytest.mark.gpu
def test_inclusion_frequency(det, OS):
    """One image in 4096 slots (each slot has its own image seed): every candidate's inclusion frequency is within 6
    sigma of want / #class, and the counts equal the reference's."""
    from oracle import ref_torch as R
    g = gen(11)
    p, gt, c = make_image(300, 30, g)  # ~60 foreground candidates: both classes are thinned
    n = 4096
    h = heads(det, "plain", S=64, f=0.25)
    args = batch([(p, gt, c)] * n)
    res = h.sample_proposals_batched(*args, seed_t(2024))
    _, _, _, cls = R.roi_label_proposals(p, gt, c, K)
    fg, bg = (cls != -1) & (cls != K), cls == K
    want_pos, want_neg = R.subsample_counts(int(fg.sum()), int(bg.sum()), 64, 0.25)
    assert bool((res["num_fg"] == want_pos).all()) and bool((res["count"] == want_pos + want_neg).all())
    src = res["src"][:, :want_pos + want_neg].long().cpu()
    hits = torch.bincount(src.reshape(-1), minlength=cls.numel()).double()
    for mask, want in ((fg, want_pos), (bg, want_neg)):
        prob = want / int(mask.sum())
        sigma = (n * prob * (1 - prob)) ** 0.5
        dev = (hits[mask] - n * prob).abs()
        assert bool((dev <= 6 * sigma + 1e-9).all()), f"max deviation {float(dev.max()):.1f} vs sigma {sigma:.2f}"
    assert float(hits[~(fg | bg)].sum()) == 0.0


def _instances(det, images):
    proposals, targets = [], []
    g = gen(21)
    for p, gt, c in images:
        pi = det.Instances((800, 800))
        pi.proposal_boxes = det.Boxes(p.cuda())
        pi.objectness_logits = torch.randn(p.shape[0], generator=g).cuda()
        t = det.Instances((800, 800))
        t.gt_boxes = det.Boxes(gt.cuda())
        t.gt_classes = c.cuda()
        proposals.append(pi)
        targets.append(t)
    return proposals, targets


@pytest.mark.gpu
def test_list_wrapper(det, OS):
    """label_and_sample_proposals_batched returns the batched call's rows with every field gathered, sets the logged
    means, and holds the properties of label_and_sample_proposals' contract."""
    from oracle import ref_torch as R
    g = gen(7)
    images = [make_image(P, G, g) for P, G in [(500, 6), (40, 3), (300, 0)]]
    proposals, targets = _instances(det, images)
    h = heads(det, "plain", S=128, f=0.25)
    out = h.label_and_sample_proposals_batched(proposals, targets, seed=99)
    res = h.sample_proposals_batched(*batch(images), seed_t(99))
    nfg, nbg = [], []
    for i, ((p, gt, c), r) in enumerate(zip(images, out)):
        n = int(res["count"][i])
        assert len(r) == n
        src = res["src"][i, :n].long()
        allb = torch.cat([p, gt]).cuda()
        assert torch.equal(r.proposal_boxes.tensor, allb[src])
        logits = torch.cat([proposals[i].objectness_logits, torch.full((gt.shape[0],), R.GT_LOGIT).cuda()])
        assert torch.equal(r.objectness_logits, logits[src])
        assert torch.equal(r.gt_classes, res["gt_classes"][i, :n])
        cls = r.gt_classes.cpu()
        _, _, _, wc = R.roi_label_proposals(p, gt, c, K)
        want_pos, want_neg = R.subsample_counts(int(((wc != -1) & (wc != K)).sum()), int((wc == K).sum()), 128, 0.25)
        assert int((cls != K).sum()) == want_pos and int((cls == K).sum()) == want_neg
        nfg.append(want_pos)
        nbg.append(want_neg)
        if gt.shape[0]:
            assert torch.equal(r.gt_boxes.tensor, res["gt_boxes"][i, :n])
            fg = cls != K
            iou = R.pairwise_iou(r.gt_boxes.tensor.cpu()[fg], r.proposal_boxes.tensor.cpu()[fg]).diagonal()
            assert bool((iou >= 0.5).all())
            assert int(fg.sum()) >= min(gt.shape[0], 32)  # the appended gt boxes are positives themselves
        else:
            assert not r.has("gt_boxes") and bool((cls == K).all())
    assert h.last_num_fg_samples == sum(nfg) / 3 and h.last_num_bg_samples == sum(nbg) / 3
    torch.manual_seed(5)
    a = h.label_and_sample_proposals_batched(proposals, targets)
    torch.manual_seed(5)
    b = h.label_and_sample_proposals_batched(proposals, targets)
    assert all(torch.equal(x.proposal_boxes.tensor, y.proposal_boxes.tensor) for x, y in zip(a, b))


@pytest.mark.gpu
def test_graph_replay_advances_seed_and_determinism(det, OS):
    """Captured with seed.add_(1) in the graph, three replays equal the oracle at seeds s, s+1, s+2; 26 eager launches
    are bitwise identical, with and without a second stream busy; an eager call makes no host synchronisation."""
    g = gen(31)
    images = [make_image(P, G, g) for P, G in [(2000, 40), (1000, 5), (1500, 60), (700, 0)]]
    args = batch(images)
    h = heads(det, "lowq")
    seed = seed_t(1234)
    first = {k: v.clone() for k, v in h.sample_proposals_batched(*args, seed).items()}
    other = torch.cuda.Stream()
    x = torch.randn(2048, 2048, device="cuda")
    for i in range(25):
        if i % 2:
            other.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(other):
                for _ in range(4):
                    x = torch.tanh(x @ x * 1e-3)
        again = h.sample_proposals_batched(*args, seed)
        for k in first:
            assert torch.equal(again[k], first[k]), k
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        h.sample_proposals_batched(*args, seed)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ws = h.sample_workspace(len(images), args[0].shape[1], args[2].shape[0], "cuda")
        out = {k: torch.empty_like(v) for k, v in first.items()}
        h.sample_proposals_batched(*args, seed, out=out, workspace=ws)
    torch.cuda.current_stream().wait_stream(st)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        h.sample_proposals_batched(*args, seed, out=out, workspace=ws)
        seed.add_(1)
    for r in range(3):
        for v in out.values():
            v.fill_(-7)
        graph.replay()
        torch.cuda.synchronize()
        check(OS, h, out, images, 1234 + r, "lowq")
    assert int(seed) == 1237


@pytest.mark.gpu
def test_second_stage_step_captured(det):
    """proposals_from_heads -> sample_proposals_batched -> ROIPooler -> Linear head -> losses_batched(with_grads=True),
    captured in one CUDA graph and replayed: losses and sampled rows equal the eager run's."""
    g = gen(41)
    n, K2, C, R = 2, 20, 8, 7
    rpn = det.RegionProposalNetwork([8, 16, 32], [[32], [64], [128]], [[0.5, 1.0, 2.0]])
    rpn.training = True  # 2000 proposals per image
    hw = [(32, 32), (16, 16), (8, 8)]
    obj = [torch.randn(n, 3, a, b, generator=g).cuda() for a, b in hw]
    dlt = [(torch.randn(n, 12, a, b, generator=g) * 0.3).cuda() for a, b in hw]
    sizes = torch.tensor([[256, 256]] * n, dtype=torch.int32).cuda()
    gts = [rand_boxes(G, 256.0, g, 0.3) for G in (4, 6)]
    table, off = det.Matcher.pack_gt([x.cuda() for x in gts], torch.device("cuda"))
    classes = torch.randint(0, K2, (10,), generator=g).cuda()
    h = det.ROIHeads(K2, 64, 0.25, det.Matcher([0.5], [0, 1], allow_low_quality_matches=False), True)
    feats = [torch.randn(n, C, 256 // s, 256 // s, generator=g).cuda() for s in (8, 16, 32)]
    pooler = det.ROIPooler([1 / 8, 1 / 16, 1 / 32], 0, R, "ROIAlignV2")
    torch.manual_seed(0)
    fc = torch.nn.Linear(C * R * R, 5 * K2 + 1).cuda()
    fr = det.FastRCNNOutputs(K2)
    seed = seed_t(8)

    def step(out=None, ws=None):
        props, _, counts, _ = rpn.proposals_from_heads(obj, dlt, sizes)
        res = h.sample_proposals_batched(props, counts, table, off, classes, seed, out=out, workspace=ws)
        x = pooler(feats, [det.Boxes(res["boxes"][i]) for i in range(n)])
        y = fc(x.flatten(1))
        loss = fr.losses_batched(y[:, :K2 + 1], y[:, K2 + 1:], res["boxes"].reshape(-1, 4),
                                 res["gt_classes"].reshape(-1), res["gt_boxes"].reshape(-1, 4), with_grads=True)
        return res, loss

    eager_res, eager_loss = step()
    eager_res = {k: v.clone() for k, v in eager_res.items()}
    eager_loss = {k: v.detach().clone() for k, v in eager_loss.items()}
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ws = h.sample_workspace(n, rpn.post_nms_topk[True], 10, "cuda")
        out = {k: torch.empty_like(v) for k, v in eager_res.items()}
        step(out, ws)
    torch.cuda.current_stream().wait_stream(st)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        _, cap_loss = step(out, ws)
    graph.replay()
    torch.cuda.synchronize()
    for k in eager_res:
        assert torch.equal(out[k], eager_res[k]), k
    assert int(out["num_fg"].sum()) > 0
    for k, v in eager_loss.items():  # the loss sums are added by atomics in arrival order
        torch.testing.assert_close(cap_loss[k].detach(), v, rtol=1e-5, atol=1e-7)


# ---------------------------------------------------------------------------------------------------- no GPU needed
def _raw_call(S=64, f=0.25, n=1, p_stride=8, sum_g=2, null_out=False, labels=(0, 1)):
    import det_b200
    N = det_b200._native
    fake = ctypes.c_void_p(1 << 20)  # never dereferenced: every checked case returns before any CUDA call
    thr = (ctypes.c_float * 1)(0.5)
    lab = (ctypes.c_int32 * len(labels))(*labels)
    outs = [None if null_out else fake] * 8
    return N.fn("det_roi_sample_proposals")(fake, fake, n, p_stride, fake, fake, fake, sum_g, K, thr, lab, 1, 0, S,
                                            f, 1, fake, *outs, fake, 1 << 30, None)


def test_argument_checks():
    assert _raw_call(S=0) == -1
    assert _raw_call(f=-0.1) == -1
    assert _raw_call(f=1.5) == -1
    assert _raw_call(f=float("nan")) == -1
    assert _raw_call(null_out=True) == -1
    assert _raw_call(n=-1) == -1
    assert _raw_call(p_stride=1 << 24) == -2
    assert _raw_call(sum_g=1 << 24) == -2
    assert _raw_call(n=70000) == -2
    assert _raw_call(S=1 << 24) == -2
    assert _raw_call(n=0) == 0


def test_workspace_bytes():
    import det_b200
    f = det_b200._native.fn("det_roi_sample_workspace_bytes")
    assert f(16, 2000, 100) == 400 + (16 * 2000 + 100) * 4
    assert f(2, 10, 3) == 16 + 23 * 4
