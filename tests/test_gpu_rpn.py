"""GPU parity: RPN decode from the conv layout, proposal selection (find_top_rpn_proposals) vs the oracle."""
import pytest
import torch

from tests.util import gen, rand_boxes, assert_boxes_close

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


def _heads(n, img, g, scale=1.0, a=3):
    """a: anchors per position, one count for every level or a sequence with one count per level"""
    per_level = [a] * len(STRIDES) if isinstance(a, int) else a
    obj = [torch.randn(n, k, img // s, img // s, generator=g) for s, k in zip(STRIDES, per_level)]
    dlt = [torch.randn(n, 4 * k, img // s, img // s, generator=g) * scale for s, k in zip(STRIDES, per_level)]
    return obj, dlt


def _oracle_decode(O, obj, dlt, img, weights=(1.0, 1.0, 1.0, 1.0), sizes=SIZES, ratios=RATIOS):
    ratios = ratios * len(sizes) if len(ratios) == 1 else ratios
    cells = [O.cell_anchors(s, r) for s, r in zip(sizes, ratios)]
    anchors = O.grid_anchors([(img // s, img // s) for s in STRIDES], STRIDES, cells, 0.0)
    lg, dl = zip(*[O.head_to_hwa(o, d) for o, d in zip(obj, dlt)])
    props = O.decode_proposals(anchors, list(dl), weights)
    return anchors, list(lg), list(dl), props


RPN_FLAT_MAX_A = 4  # kRpnFlatMaxA, csrc/box_ops.cu:278


def rpn_decode_launches(a, level_hw):
    """The launches det_rpn_decode makes (box_ops.cu:541-556, :521-528): one flat launch for the whole pyramid when
    a <= RPN_FLAT_MAX_A, else one det_rpn_decode_level launch per level, with 16-byte loads ("vec") when the level's
    planes are whole 16-byte tiles and scalar loads otherwise (aligned heads assumed, as torch allocates them)."""
    if a <= RPN_FLAT_MAX_A:
        return ["flat"]
    return ["vec" if (h * w) % 4 == 0 else "scalar" for h, w in level_hw]


_ANCHOR_SETS = {  # anchors per position: (sizes per level, ratios)
    1: (SIZES, [[1.0]]),
    2: (SIZES, [[0.5, 2.0]]),
    4: ([[s[0], s[0] * 1.5] for s in SIZES], [[0.5, 2.0]]),
    9: ([[s[0], s[0] * 1.26, s[0] * 1.59] for s in SIZES], RATIOS),
    (3, 6, 3, 3, 3): ([[32], [64, 90], [128], [256], [512]], RATIOS),
}


@pytest.mark.parametrize("img,a,weights", [
    pytest.param(448, 3, (1.0, 1.0, 1.0, 1.0), id="448"),
    pytest.param(224, 3, (1.0, 1.0, 1.0, 1.0), id="224"),
    pytest.param(224, 1, (10.0, 10.0, 5.0, 5.0), id="224-a1"),
    pytest.param(224, 2, (10.0, 10.0, 5.0, 5.0), id="224-a2"),
    pytest.param(448, 4, (10.0, 10.0, 5.0, 5.0), id="448-a4"),
    pytest.param(448, 9, (10.0, 10.0, 5.0, 5.0), id="448-a9"),
    pytest.param(448, (3, 6, 3, 3, 3), (10.0, 10.0, 5.0, 5.0), id="448-a3-6-3-3-3"),
])
def test_decode_heads_matches_oracle(det, O, img, a, weights):
    """a = 3 (the reference's anchors) and other anchor sets: a <= 4 decodes the pyramid in one flat launch, a = 9
    (three sizes x three ratios) falls back to one launch per level (vec and scalar forms).  Unequal anchor counts per
    level (a = 3, 6, 3, 3, 3): decode_heads calls det_rpn_decode_typed once per level.  With box weights (10, 10, 5, 5)
    some width / height deltas exceed scale_clamp."""
    sizes, ratios = _ANCHOR_SETS[a] if a != 3 else (SIZES, RATIOS)
    level_hw = [(img // s, img // s) for s in STRIDES]
    if isinstance(a, int):
        per_level = [a] * len(STRIDES)
        launches = rpn_decode_launches(a, level_hw)
        if a <= RPN_FLAT_MAX_A:
            assert launches == ["flat"]
        else:
            assert {"vec", "scalar"} <= set(launches)
    else:
        per_level = list(a)
        launches = [x for k, hw in zip(per_level, level_hw) for x in rpn_decode_launches(k, [hw])]
        assert launches == ["flat", "vec", "flat", "flat", "flat"]
    g = gen(img + (0 if a == 3 else 100 * sum(per_level) // len(per_level)))
    obj, dlt = _heads(3, img, g, 0.5 if weights[2] == 1.0 else 4.0, a)
    rpn = det.RegionProposalNetwork(STRIDES, sizes, ratios, box2box_weights=weights)
    if weights[2] != 1.0:
        for d in dlt:  # beyond scale_clamp (log(1000/16) = 4.14 after dividing by 5), both signs of dx / dy
            d[:, 2::4, ::3, ::2] = 30.0
            d[:, 3::4, 1::3, ::2] = 25.0
            d[:, 0::4, ::2, 1::3] *= -3.0
        assert any(float(d[:, 2::4].max()) / weights[2] > rpn.box2box_transform.scale_clamp for d in dlt)
    logits, boxes, lsz = rpn.decode_heads([o.cuda() for o in obj], [d.cuda() for d in dlt])
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, img, weights, sizes, ratios)
    assert lsz == [x.shape[0] for x in anchors]
    assert sum(lsz) == sum(k * (img // s) ** 2 for k, s in zip(per_level, STRIDES))
    if img == 448 and a == 3:
        assert sum(lsz) == 50127
    assert torch.equal(logits.cpu(), torch.cat(lg, 1))          # pure layout change: bit-exact
    assert_boxes_close(boxes.cpu(), torch.cat(props, 1), rtol=1e-5)


def test_reference_signature_decode_proposals(det, O):
    g = gen(1)
    obj, dlt = _heads(2, 128, g)
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, 128, (10.0, 10.0, 5.0, 5.0))
    rpn = det.RegionProposalNetwork(STRIDES, SIZES, RATIOS, box2box_weights=(10.0, 10.0, 5.0, 5.0))
    got = rpn._decode_proposals([det.Boxes(a.cuda()) for a in anchors], [d.cuda() for d in dl])
    for a, b in zip(got, props):
        assert_boxes_close(a.cpu(), b, rtol=1e-5)


@pytest.mark.parametrize("img,pre,post,training", [(448, 12000, 2000, False), (448, 6000, 1000, True),
                                                   (128, 12000, 2000, False), (64, 50, 20, False)])
def test_find_top_rpn_proposals_matches_oracle(det, O, img, pre, post, training):
    """Kept boxes/logits and counts bit-exact on identical inputs (the proposals fed to both sides are the same)."""
    g = gen(img + pre)
    n = 3
    obj, dlt = _heads(n, img, g, 0.3)
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, img)
    sizes = [(img, img), (img - 17, img), (img, img - 40)]
    want = O.find_top_rpn_proposals(props, lg, sizes, 0.7, pre, post, 0.0, training)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, 0.7, pre, post, 0.0,
                                     training)
    assert len(got) == n
    for i in range(n):
        wb, ws = want[i]
        assert len(got[i]) == wb.shape[0], (i, len(got[i]), wb.shape[0])
        assert torch.equal(got[i].objectness_logits.cpu(), ws)
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), wb)
        assert got[i].image_size == sizes[i]


def test_find_top_rpn_proposals_min_size_and_nonfinite(det, O):
    g = gen(77)
    obj, dlt = _heads(2, 128, g, 0.3)
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, 128)
    props[0][0, 5, 2] = float("inf")
    lg[1][1, 7] = float("nan")
    sizes = [(128, 128), (100, 128)]
    want = O.find_top_rpn_proposals([p.clone() for p in props], lg, sizes, 0.7, 1000, 300, 8.0, False)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, 0.7, 1000, 300, 8.0, False)
    for i in range(2):
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), want[i][0])
        assert torch.equal(got[i].objectness_logits.cpu(), want[i][1])
    with pytest.raises(FloatingPointError):
        det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, 0.7, 1000, 300, 8.0, True)


def test_forward_eval_from_heads(det, O):
    g = gen(9)
    obj, dlt = _heads(2, 224, g, 0.3)
    rpn = det.RegionProposalNetwork(STRIDES, SIZES, RATIOS).eval()
    sizes = [(224, 224), (200, 210)]
    props, losses = rpn.forward(sizes, head_outputs=([o.cuda() for o in obj], [d.cuda() for d in dlt]))
    assert losses == {}
    # oracle fed with the GPU's own decoded proposals (identical inputs to the selection stage)
    logits, boxes, lsz = rpn.decode_heads([o.cuda() for o in obj], [d.cuda() for d in dlt])
    pl = list(torch.split(boxes.cpu(), lsz, dim=1))
    ll = list(torch.split(logits.cpu(), lsz, dim=1))
    want = O.find_top_rpn_proposals(pl, ll, sizes, 0.7, 12000, 2000, 0.0, False)
    for i in range(2):
        assert torch.equal(props[i].proposal_boxes.tensor.cpu(), want[i][0])
        assert torch.equal(props[i].objectness_logits.cpu(), want[i][1])


@pytest.mark.parametrize("nms_thresh,pre,post", [(0.7, 2000, 300), (0.05, 2000, 300), (0.3, 4000, 1000), (0.7, 1000, 50)])
def test_find_top_rpn_proposals_tier_cut(det, O, nms_thresh, pre, post):
    """post_nms_topk << candidates: the per-level sweeps first run above a global score cut (exact); with a low NMS
    threshold the cut falls short and the full segments are swept in a second pass."""
    g = gen(int(nms_thresh * 100) + post)
    n = 3
    obj, dlt = _heads(n, 448, g, 0.3)
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, 448)
    sizes = [(448, 448), (400, 448), (448, 300)]
    want = O.find_top_rpn_proposals(props, lg, sizes, nms_thresh, pre, post, 0.0, False)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, nms_thresh, pre, post,
                                     0.0, False)
    for i in range(n):
        wb, ws = want[i]
        assert len(got[i]) == wb.shape[0], (i, len(got[i]), wb.shape[0])
        assert torch.equal(got[i].objectness_logits.cpu(), ws)
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), wb)


def test_find_top_rpn_proposals_equal_logits_straddle_the_topk_cut(det, O):
    """Quantised logits: the per-level radix select has to go on into the index bits (stable order, lower index first)."""
    g = gen(123)
    n = 2
    obj, dlt = _heads(n, 224, g, 0.3)
    obj = [(o * 2).round() / 2 for o in obj]
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, 224)
    sizes = [(224, 224), (200, 224)]
    for pre, post in ((100, 40), (700, 300), (3000, 1000)):
        want = O.find_top_rpn_proposals(props, lg, sizes, 0.7, pre, post, 0.0, False)
        got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, 0.7, pre, post, 0.0,
                                         False)
        for i in range(n):
            assert torch.equal(got[i].objectness_logits.cpu(), want[i][1])
            assert torch.equal(got[i].proposal_boxes.tensor.cpu(), want[i][0])


@pytest.mark.parametrize("seed", list(range(int(__import__("os").environ.get("DET_STRESS_SEEDS", "12")))))
def test_find_top_rpn_proposals_stress(det, O, seed):
    """Random proposal-selection problems: pyramid size, delta scale (tiny to image-sized boxes), pre/post top-k around the
    level sizes, NMS threshold, min box size, ragged image sizes, quantised logits (ties at the cuts) and an occasional
    non-finite proposal in eval mode: kept boxes, logits and counts bit-exact on identical inputs."""
    g = gen(13000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    rf = lambda lo, hi: float(torch.rand(1, generator=g)) * (hi - lo) + lo
    img = 64 * ri(1, 5)
    n = ri(1, 4)
    obj, dlt = _heads(n, img, g, rf(0.05, 1.5))
    if ri(0, 2) == 0:
        obj = [(o * 2).round() / 2 for o in obj]
    anchors, lg, dl, props = _oracle_decode(O, obj, dlt, img)
    if ri(0, 3) == 0:
        props[ri(0, len(props) - 1)][0, 0, ri(0, 3)] = float("inf")
    pre = [5, 60, 1000, 12000][ri(0, 3)]
    post = [1, 20, 300, 2000][ri(0, 3)]
    thr = rf(0.3, 0.9)
    min_size = [0.0, 0.0, 4.0, 20.0][ri(0, 3)]
    sizes = [(img - ri(0, 30), img - ri(0, 30)) for _ in range(n)]
    want = O.find_top_rpn_proposals([p.clone() for p in props], lg, sizes, thr, pre, post, min_size, False)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lg], sizes, thr, pre, post, min_size, False)
    for i in range(n):
        wb, ws = want[i]
        assert len(got[i]) == wb.shape[0], (i, len(got[i]), wb.shape[0])
        assert torch.equal(got[i].objectness_logits.cpu(), ws), i
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), wb), i

