"""Second-stage training losses: det_fast_rcnn_loss_typed (csrc/fast_rcnn_loss.cu) and FastRCNNOutputs.losses /
losses_batched against tests/fast_rcnn_loss_oracle.py (detectron2's FastRCNNOutputLayers.losses and
_log_classification_stats in fp32 CPU autograd).  Losses and gradients within 1e-5 relative (GIoU delta gradients
1e-4), the four statistics counts exact; fused forward+backward equal to autograd's backward bit for bit; 16-bit rows
bit-identical to the fp32 call followed by .to(dtype).  The last tests need no GPU."""
import copy
import ctypes
import math

import pytest
import torch

from tests.util import gen

WEIGHTS = (10.0, 10.0, 5.0, 5.0)
CLAMP = math.log(1000.0 / 16)
STATS = ("num_fg", "num_accurate", "fg_num_accurate", "num_false_negative")


@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


@pytest.fixture(scope="module")
def O():
    from tests import fast_rcnn_loss_oracle
    return fast_rcnn_loss_oracle


def make_rows(M, K, seed, agnostic=False, fg_frac=0.25, scale=2.0):
    """Rows as ROIHeads samples them: proposals inside a 640 x 480 frame, fg rows with a gt box near their proposal and
    a class in [0, K), bg rows labelled K with their proposal as gt box."""
    g = gen(seed)
    logits = torch.randn(M, K + 1, generator=g) * scale
    deltas = torch.randn(M, 4 if agnostic else 4 * K, generator=g) * 0.5
    xy = torch.rand(M, 2, generator=g) * torch.tensor([576.0, 432.0])
    wh = 8.0 + torch.rand(M, 2, generator=g) * torch.tensor([200.0, 150.0])
    props = torch.cat([xy, xy + wh], 1)
    jitter = (torch.rand(M, 4, generator=g) - 0.5) * 0.3 * torch.cat([wh, wh], 1)
    nfg = int(round(fg_frac * M))
    fg = torch.zeros(M, dtype=torch.bool)
    fg[torch.randperm(M, generator=g)[:nfg]] = True
    classes = torch.where(fg, torch.randint(0, K, (M,), generator=g), torch.full((M,), K))
    gtb = torch.where(fg[:, None], props + jitter, props)
    return logits, deltas, props, classes, gtb


def outputs(det, K, agnostic=False, loss_type="smooth_l1", beta=0.0, loss_weight=1.0):
    return det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP), class_agnostic=agnostic,
                               box_reg_loss_type=loss_type, smooth_l1_beta=beta, loss_weight=loss_weight)


def oracle(O, rows, K, loss_type="smooth_l1", beta=0.0, loss_weight=1.0, upstream=(1.0, 1.0)):
    """Oracle losses, statistics and the gradients of upstream[0] * loss_cls + upstream[1] * loss_box_reg."""
    logits, deltas, props, classes, gtb = rows
    lg, dl = logits.clone().requires_grad_(True), deltas.clone().requires_grad_(True)
    want, stats = O.fast_rcnn_losses(lg, dl, props, classes, gtb, K, loss_type, beta, WEIGHTS, CLAMP, loss_weight)
    (upstream[0] * want["loss_cls"] + upstream[1] * want["loss_box_reg"]).backward()
    return want, stats, lg.grad, dl.grad


def cuda(rows):
    return [t.cuda() for t in rows]


def assert_stats(sums, stats, bad=0):
    s = sums.cpu()
    got = {k: int(s[2 + i]) for i, k in enumerate(STATS)}
    assert got == {k: stats[k] for k in STATS}
    assert int(s[6]) == bad and float(s[7]) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 263])
@pytest.mark.parametrize("fg_frac", [0.0, 0.25, 1.0])
@pytest.mark.parametrize("loss", [("smooth_l1", 0.0), ("smooth_l1", 0.5), ("giou", 0.0)])
@pytest.mark.parametrize("agnostic", [False, True])
@pytest.mark.parametrize("K", [1, 20, 80, 130, 1000])
def test_parity_with_oracle(det, O, K, agnostic, loss, fg_frac, M):
    """Losses, statistics and the fused launch's gradients against the oracle: every column count path (register
    path with one and four column chunks, general path), both regression forms, both loss types."""
    loss_type, beta = loss
    rows = make_rows(M, K, 1000 * K + M + int(agnostic), agnostic, fg_frac)
    want, stats, wgl, wgd = oracle(O, rows, K, loss_type, beta)
    res = outputs(det, K, agnostic, loss_type, beta).losses_batched(*cuda(rows), with_grads=True)
    torch.testing.assert_close(res["loss_cls"].cpu(), want["loss_cls"].detach(), rtol=1e-5, atol=0.0)
    torch.testing.assert_close(res["loss_box_reg"].cpu(), want["loss_box_reg"].detach(), rtol=1e-5, atol=1e-12)
    assert_stats(res["sums"], stats)
    s = 1.0 / M  # the largest gradient magnitude of a column (|softmax - onehot| <= 1) times the loss scale
    torch.testing.assert_close(res["grad_logits"].cpu(), wgl, rtol=1e-5, atol=1e-6 * s)
    rd = 1e-4 if loss_type == "giou" else 1e-5
    torch.testing.assert_close(res["grad_deltas"].cpu(), wgd, rtol=rd, atol=rd * 0.1 * s)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [80, 1000])
@pytest.mark.parametrize("loss_type", ["smooth_l1", "giou"])
def test_fused_equals_autograd_and_scales(det, O, K, loss_type):
    """with_grads=True gives the gradients autograd's backward gives, bit for bit; loss_weight and an upstream
    gradient scale them as s_x = w_x / M * upstream[x]."""
    M = 517
    rows = cuda(make_rows(M, K, 5, False, 0.3))
    fr = outputs(det, K, loss_type=loss_type)
    fused = fr.losses_batched(*rows, with_grads=True)
    lg, dl = rows[0].clone().requires_grad_(True), rows[1].clone().requires_grad_(True)
    res = fr.losses_batched(lg, dl, *rows[2:])
    (res["loss_cls"] + res["loss_box_reg"]).backward()
    assert torch.equal(lg.grad, fused["grad_logits"]) and torch.equal(dl.grad, fused["grad_deltas"])
    assert torch.equal(res["sums"][2:], fused["sums"][2:])
    torch.testing.assert_close(res["sums"][:2], fused["sums"][:2], rtol=1e-6, atol=0.0)
    w = {"loss_cls": 0.7, "loss_box_reg": 1.3}
    lg2, dl2 = rows[0].clone().requires_grad_(True), rows[1].clone().requires_grad_(True)
    res2 = outputs(det, K, loss_type=loss_type, loss_weight=w).losses_batched(lg2, dl2, *rows[2:])
    (0.37 * (res2["loss_cls"] + res2["loss_box_reg"])).backward()
    torch.testing.assert_close(res2["loss_cls"], fused["loss_cls"] * 0.7, rtol=1e-6, atol=0.0)
    torch.testing.assert_close(res2["loss_box_reg"], fused["loss_box_reg"] * 1.3, rtol=1e-6, atol=0.0)
    torch.testing.assert_close(lg2.grad, fused["grad_logits"] * (0.7 * 0.37), rtol=1e-6, atol=1e-12)
    torch.testing.assert_close(dl2.grad, fused["grad_deltas"] * (1.3 * 0.37), rtol=1e-6, atol=1e-12)
    want, _, wgl, wgd = oracle(O, [t.cpu() for t in rows], K, loss_type, loss_weight=w, upstream=(0.37, 0.37))
    torch.testing.assert_close(lg2.grad.cpu(), wgl, rtol=1e-5, atol=1e-6 / M)
    torch.testing.assert_close(dl2.grad.cpu(), wgd, rtol=1e-4, atol=1e-6 / M)
    # a loss the caller does not use gets upstream 0: its gradient vanishes
    lg3 = rows[0].clone().requires_grad_(True)
    dl3 = rows[1].clone().requires_grad_(True)
    fr.losses_batched(lg3, dl3, *rows[2:])["loss_cls"].backward()
    assert torch.equal(lg3.grad, fused["grad_logits"]) and not bool(dl3.grad.any())


@pytest.mark.gpu
@pytest.mark.parametrize("K", [5, 80, 130])
def test_argmax_ties_and_nan_counts(det, O, K):
    """pred = torch.argmax: the first maximum, and the first NaN when a row has one -- across lanes and chunks."""
    nan, inf = float("nan"), float("inf")

    def row(**cols):
        r = torch.zeros(K + 1)
        for c, v in cols.items():
            r[int(c[1:]) % (K + 1)] = v
        return r
    rows = [torch.zeros(K + 1),                                  # all tied: column 0
            row(c1=3.0, c2=3.0, c5=3.0),                          # tie between the lowest columns
            row(c1=nan, c2=5.0, c3=nan),                          # first NaN
            row(c0=-1.0, **{f"c{K}": 9.0}),                       # background wins
            row(**{f"c{K}": nan}),                                # NaN in the background column
            torch.full((K + 1,), -inf),                           # all -inf: column 0
            row(c40=7.0, c7=7.0, c70=7.0),                        # ties across lanes / chunks
            row(c70=nan, c33=nan, c100=9.0),                      # NaNs across chunks
            row(c3=-2.0, c35=nan, c67=inf, c99=inf)]
    logits = torch.stack(rows)
    M = logits.shape[0]
    gt = torch.tensor([0, 1, 1, 2, 3 % K, K, 7 % K, 33 % (K + 1), 3 % K])
    rows_all = [logits, torch.zeros(M, 4 * K), make_rows(M, K, 3)[2], gt, make_rows(M, K, 3)[2]]
    _, stats = O.fast_rcnn_losses(*rows_all, K)
    res = outputs(det, K).losses_batched(*cuda(rows_all), with_grads=True)
    assert_stats(res["sums"], stats)
    assert int(logits.argmax(1)[2]) == 1  # the oracle's torch.argmax takes the first NaN


@pytest.mark.gpu
@pytest.mark.parametrize("K", [20, 80, 1000])
def test_out_of_range_labels(det, O, K):
    """Labels outside [0, K]: counted in sums[6], zero gradient rows, the rest as the oracle with M as denominator."""
    M = 77
    rows = list(make_rows(M, K, 11, False, 0.5))
    bad = torch.zeros(M, dtype=torch.bool)
    bad[[0, 5, 31, 32, 76]] = True
    rows[3] = rows[3].clone()
    rows[3][[0, 5, 31, 32, 76]] = torch.tensor([-1, K + 1, 1000000, -7, K + 2])
    want, stats, wgl, wgd = oracle(O, rows, K)
    res = outputs(det, K).losses_batched(*cuda(rows), with_grads=True)
    assert_stats(res["sums"], stats, bad=5)
    torch.testing.assert_close(res["loss_cls"].cpu(), want["loss_cls"].detach(), rtol=1e-5, atol=0.0)
    torch.testing.assert_close(res["loss_box_reg"].cpu(), want["loss_box_reg"].detach(), rtol=1e-5, atol=0.0)
    gl, gd = res["grad_logits"].cpu(), res["grad_deltas"].cpu()
    assert not bool(gl[bad].any()) and not bool(gd[bad].any())
    torch.testing.assert_close(gl, wgl, rtol=1e-5, atol=1e-6 / M)
    torch.testing.assert_close(gd, wgd, rtol=1e-5, atol=1e-6 / M)


@pytest.mark.gpu
def test_empty_batch(det):
    """M = 0: both losses 0, empty gradients, and the entry reads no input pointer (NULL inputs are accepted)."""
    K = 80
    fr = outputs(det, K)
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
    lg, dl = z(0, K + 1).requires_grad_(True), z(0, 4 * K).requires_grad_(True)
    res = fr.losses_batched(lg, dl, z(0, 4), z(0, dt=torch.int64), z(0, 4))
    (res["loss_cls"] + res["loss_box_reg"]).backward()
    assert res["sums"].cpu().tolist() == [0.0] * 8
    assert lg.grad.shape == (0, K + 1) and dl.grad.shape == (0, 4 * K)
    fused = fr.losses_batched(lg.detach(), dl.detach(), z(0, 4), z(0, dt=torch.int64), z(0, 4), with_grads=True)
    assert fused["grad_logits"].shape == (0, K + 1) and float(fused["loss_box_reg"]) == 0.0
    from det_b200 import _native as N
    sums = torch.full((8,), 5.0, device="cuda")
    rc = N.fn("det_fast_rcnn_loss_typed")(None, None, 0, None, None, None, 0, K, 0, *WEIGHTS, CLAMP, 0, 0.0, 1.0, 1.0,
                                          None, N.ptr(N.accumulators("cuda")), N.ptr(sums), None, None, N.stream())
    assert rc == 0 and sums.cpu().tolist() == [0.0] * 8
    # losses() on an empty proposal list
    out = fr.losses((lg, dl), [])
    assert float(out["loss_cls"].detach()) == 0.0 and float(out["loss_box_reg"].detach()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("agnostic", [False, True])
@pytest.mark.parametrize("K", [80, 130])
def test_16bit_rows(det, dtype, agnostic, K):
    """bf16 / fp16 rows: losses are the fp32 call's on .float(); gradients are the fp32 gradients .to(dtype), bit for
    bit, through both the fused launch and autograd's backward."""
    rows = cuda(make_rows(333, K, 21, agnostic, 0.4))
    lo, do = rows[0].to(dtype), rows[1].to(dtype)
    fr = outputs(det, K, agnostic)
    ref = fr.losses_batched(lo.float(), do.float(), *rows[2:], with_grads=True)
    got = fr.losses_batched(lo, do, *rows[2:], with_grads=True)
    assert got["grad_logits"].dtype == dtype and got["grad_deltas"].dtype == dtype
    assert torch.equal(got["grad_logits"], ref["grad_logits"].to(dtype))
    assert torch.equal(got["grad_deltas"], ref["grad_deltas"].to(dtype))
    torch.testing.assert_close(got["sums"][:2], ref["sums"][:2], rtol=1e-6, atol=0.0)
    assert torch.equal(got["sums"][2:], ref["sums"][2:])
    lg, dl = lo.clone().requires_grad_(True), do.clone().requires_grad_(True)
    res = fr.losses_batched(lg, dl, *rows[2:])
    (res["loss_cls"] + res["loss_box_reg"]).backward()
    assert lg.grad.dtype == dtype and torch.equal(lg.grad, got["grad_logits"]) and torch.equal(dl.grad, got["grad_deltas"])


@pytest.mark.gpu
def test_graph_replay_and_determinism(det):
    """losses_batched(with_grads=True) captured in a CUDA graph and replayed equals the eager call (gradients and
    counts bitwise, losses within summation order: 1024 CTA partial sums are added by atomics in arrival order); 26
    eager launches agree the same way."""
    K = 80
    rows = cuda(make_rows(16 * 512, K, 8, False, 0.25))
    fr = outputs(det, K)
    eager = fr.losses_batched(*rows, with_grads=True)
    for _ in range(25):
        again = fr.losses_batched(*rows, with_grads=True)
        assert torch.equal(again["grad_logits"], eager["grad_logits"])
        assert torch.equal(again["grad_deltas"], eager["grad_deltas"])
        assert torch.equal(again["sums"][2:], eager["sums"][2:])
        torch.testing.assert_close(again["sums"][:2], eager["sums"][:2], rtol=1e-5, atol=0.0)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fr.losses_batched(*rows, with_grads=True)  # warm-up: this stream's accumulators exist before the capture
    torch.cuda.current_stream().wait_stream(st)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        cap = fr.losses_batched(*rows, with_grads=True)
    for _ in range(2):
        for k in ("grad_logits", "grad_deltas", "sums"):
            cap[k].fill_(-3)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(cap["grad_logits"], eager["grad_logits"])
        assert torch.equal(cap["grad_deltas"], eager["grad_deltas"])
        assert torch.equal(cap["sums"][2:], eager["sums"][2:])
        torch.testing.assert_close(cap["sums"][:2], eager["sums"][:2], rtol=1e-5, atol=0.0)


@pytest.mark.gpu
def test_second_stage_training_step_end_to_end(det, O):
    """label_and_sample_proposals -> ROIPooler (ROIAlignV2, features requiring grad) -> Linear box head ->
    FastRCNNOutputs.losses -> backward, against the same graph with the oracle loss: the sampled proposals are fixed
    once so both arms see the same rows.  Feature and Linear-weight gradients within 1e-4 (the pooler's backward
    accumulates with atomics)."""
    g = gen(42)
    K, C, S = 20, 16, 7
    heads = det.ROIHeads(K, 128, 0.25, det.Matcher([0.5], [0, 1], allow_low_quality_matches=False), True)
    proposals, targets = [], []
    for P, G in [(300, 5), (200, 3), (100, 0)]:
        gb = torch.rand(G, 2, generator=g) * 400
        gb = torch.cat([gb, gb + 30 + torch.rand(G, 2, generator=g) * 150], 1)
        pb = torch.rand(P, 2, generator=g) * 400
        pb = torch.cat([pb, pb + 20 + torch.rand(P, 2, generator=g) * 150], 1)
        if G:
            pb[:3 * G] = gb.repeat(3, 1) + (torch.rand(3 * G, 4, generator=g) - 0.5) * 16
        p = det.Instances((600, 600))
        p.proposal_boxes = det.Boxes(pb.cuda())
        p.objectness_logits = torch.randn(P, generator=g).cuda()
        t = det.Instances((600, 600))
        t.gt_boxes = det.Boxes(gb.cuda())
        t.gt_classes = torch.randint(0, K, (G,), generator=g).cuda()
        proposals.append(p)
        targets.append(t)
    torch.manual_seed(0)
    sampled = heads.label_and_sample_proposals(proposals, targets)
    scales = [1 / 4, 1 / 8, 1 / 16, 1 / 32]
    feats0 = [torch.randn(3, C, 608 // int(1 / s), 608 // int(1 / s), generator=g).cuda() for s in scales]
    fc0 = torch.nn.Linear(C * S * S, 64)
    cls0, box0 = torch.nn.Linear(64, K + 1), torch.nn.Linear(64, 4 * K)
    pooler = det.ROIPooler(scales, 0, S, "ROIAlignV2")
    fr = outputs(det, K)

    def step(use_library):
        feats = [f.clone().requires_grad_(True) for f in feats0]
        fc, cls, box = [copy.deepcopy(m).cuda() for m in (fc0, cls0, box0)]
        x = pooler(feats, [p.proposal_boxes for p in sampled]).flatten(1)
        h = torch.relu(fc(x))
        logits, deltas = cls(h), box(h)
        if use_library:
            losses = fr.losses((logits, deltas), sampled)
        else:
            pb = torch.cat([p.proposal_boxes.tensor for p in sampled])
            gtc = torch.cat([p.gt_classes for p in sampled])
            gtb = torch.cat([(p.gt_boxes if p.has("gt_boxes") else p.proposal_boxes).tensor for p in sampled])
            losses, _ = O.fast_rcnn_losses(logits, deltas, pb, gtc, gtb, K, "smooth_l1", 0.0, WEIGHTS, CLAMP)
        (losses["loss_cls"] + losses["loss_box_reg"]).backward()
        return losses, [f.grad for f in feats], fc.weight.grad, cls.weight.grad, box.weight.grad

    got, want = step(True), step(False)
    assert int(fr.last_sums[2]) > 0, "the sampled batch has foreground rows"
    for k in ("loss_cls", "loss_box_reg"):
        torch.testing.assert_close(got[0][k].detach(), want[0][k].detach(), rtol=1e-5, atol=0.0)
    for a, b in zip(got[1] + list(got[2:]), want[1] + list(want[2:])):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-6 * float(b.abs().max()))


# ---------------------------------------------------------------------------------------------------- no GPU needed
def test_loss_type_is_validated():
    import det_b200
    fr = det_b200.FastRCNNOutputs(3, box_reg_loss_type="diou")
    with pytest.raises(ValueError):
        fr._loss_scales(4)
    assert det_b200.FastRCNNOutputs(3, loss_weight={"loss_cls": 2.0})._loss_scales(4) == (0, 0.5, 0.25)


def test_argument_checks_need_no_gpu():
    """Argument checks return the documented codes before any CUDA call."""
    from det_b200 import _native as N
    f = N.fn("det_fast_rcnn_loss_typed")
    one = ctypes.c_void_p(16)  # never dereferenced: every call below is rejected before a launch

    def call(m=8, k=80, dtype=0, loss_type=0, acc=one, sums=one, logits=one, gl=None, gd=None):
        return f(logits, one, dtype, one, one, one, m, k, 0, *WEIGHTS, CLAMP, loss_type, 0.0, 1.0, 1.0, None, acc, sums,
                 gl, gd, None)

    assert call(dtype=3) == -1                    # unknown head dtype
    assert call(loss_type=2) == -1                # unknown loss type
    assert call(acc=None) == -1 and call(sums=None) == -1
    assert call(logits=None) == -1                # null input with m > 0
    assert call(gl=one) == -1                     # one gradient without the other
    assert call(m=-1) == -1 and call(k=0) == -1
    assert call(k=4097) == -2                     # K > 4096
    assert call(m=1 << 24) == -2                  # M >= 2^24
    assert b"m < 2^24" in N.fn("det_last_error")()
