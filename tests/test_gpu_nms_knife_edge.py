"""Knife-edge IoU parity for every NMS route: box pairs whose fp32 IoU lands one ulp either side of the threshold.

Every kept index the library returns depends on common.cuh nms_suppresses: "kept box a suppresses box b" iff the fp32
quotient inter / (area_a + area_b - inter) exceeds the DOUBLE threshold, as torchvision's CPU kernel decides it.  The
predicate compares with thr_f = float_threshold_below(thr), decides most pairs by two division-free guards
(inter > fl(t * 1.000001f), inter < fl(t * 0.999999f) with t = fl(thr_f * denom)) and takes the IEEE quotient only in
the band between them.  Random boxes essentially never land within ~1.5e-6 relative of the threshold, so the inputs
here are BUILT there: a partner of box a whose real IoU is exactly thr, one coordinate stepped by a few ulps, kept when
its fp32 IoU is prev(thr_f), thr_f or next(thr_f), or its intersection sits within a few ulps of a guard.  Every GPU
test counts, on the exact boxes the kernel compared (the boxes passed in, the offset trick's shifted boxes, or the
kernel's own decoded boxes), how many pairs are on the edge (`census`) and asserts that count before it compares the
kept indices with the C oracle (oracle/nms_ref.c, the plain formula) bit for bit.

The first part needs no GPU: the fp32 reference, the census and the generators, checked against the oracle."""
import math

import numpy as np
import pytest
import torch

F32 = np.float32
THRESHOLDS = (0.5, 0.7, 0.3, 0.45, 0.6, 0.05, 0.9, 0.75)
GUARD_HI, GUARD_LO = F32(1.000001), F32(0.999999)   # the guard factors of nms_suppresses (common.cuh)


# ---------------------------------------------------------------------------------------------------------------------
# fp32 reference (numpy float32: one IEEE operation at a time; the library is built with -fmad=false)
# ---------------------------------------------------------------------------------------------------------------------
def _ord(x):
    """float32 -> integer that orders like the float (+0 and -0 both 0): adjacent floats differ by 1."""
    i = np.asarray(x, dtype=F32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7FFFFFFF), i)


def _unord(o):
    o = np.asarray(o, dtype=np.int64)
    u = np.where(o < 0, (-o) | 0x80000000, o).astype(np.uint32)
    return u.view(F32)


def ulp_step(x, k):
    """x moved by k ulps (k > 0 towards +inf): np.nextafter applied k times."""
    return _unord(_ord(x) + np.asarray(k, dtype=np.int64))


def thr_below(thr):
    """common.cuh float_threshold_below: the largest float f with (double)f <= thr."""
    f = F32(thr)
    if float(f) > thr:
        f = np.nextafter(f, F32(-np.inf), dtype=F32)
    return F32(f)


def _max_std(a, b):  # std::max: (a < b) ? b : a
    return np.where(a < b, b, a).astype(F32)


def _min_std(a, b):  # std::min: (b < a) ? b : a
    return np.where(b < a, b, a).astype(F32)


def _inter_denom(a, b):
    a, b = np.asarray(a, dtype=F32), np.asarray(b, dtype=F32)
    with np.errstate(all="ignore"):
        xx1, yy1 = _max_std(a[..., 0], b[..., 0]), _max_std(a[..., 1], b[..., 1])
        xx2, yy2 = _min_std(a[..., 2], b[..., 2]), _min_std(a[..., 3], b[..., 3])
        w, h = _max_std(F32(0), xx2 - xx1), _max_std(F32(0), yy2 - yy1)
        inter = w * h
        area_a = (a[..., 2] - a[..., 0]) * (a[..., 3] - a[..., 1])
        area_b = (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])
        denom = (area_a + area_b) - inter
    return inter, denom


def ovr32(a, b):
    """fp32 IoU of box a (kept) and box b in oracle/nms_ref.c's operation order."""
    inter, denom = _inter_denom(a, b)
    with np.errstate(all="ignore"):
        return inter / denom


def suppresses(a, b, thr):
    """The oracle's decision for one pair: (double)fp32 IoU > the double threshold."""
    return float(ovr32(a, b)) > thr


def predicate(a, b, thr_f, hi=GUARD_HI, lo=GUARD_LO):
    """A restatement of nms_suppresses (NONAN = false) with its guard factors as parameters."""
    inter, denom = _inter_denom(a, b)
    thr_f = F32(thr_f)
    with np.errstate(all="ignore"):
        t = thr_f * denom
        guarded = (thr_f > F32(1e-30)) & (t > F32(1e-30)) & (t < F32(1e30))
        up = guarded & (inter > t * F32(hi))
        down = guarded & (inter < t * F32(lo))
        exact = (inter / denom) > thr_f
    zero = (thr_f < 0) & (denom == denom) & (denom != 0)
    return np.where(inter == 0, zero, np.where(up, True, np.where(down, False, exact)))


# ---------------------------------------------------------------------------------------------------------------------
# census: how many pairs of a box set sit on the predicate's decision boundary
# ---------------------------------------------------------------------------------------------------------------------
CENSUS_KEYS = ("prev", "eq", "next", "band", "hi_edge", "lo_edge", "guard", "range")


def _pair_census(a, b, thr):
    """Counts for the pairs (a[k], b[k]); see census()."""
    thr_f = thr_below(thr)
    inter, denom = _inter_denom(a, b)
    with np.errstate(all="ignore"):
        o = inter / denom
        t = thr_f * denom
        thi, tlo = t * GUARD_HI, t * GUARD_LO
    live = (inter != 0) & np.isfinite(inter) & np.isfinite(denom)
    oi = _ord(np.where(np.isfinite(o), o, F32(0)))
    d = oi - _ord(thr_f)
    edge = lambda g: live & np.isfinite(g) & (np.abs(_ord(inter) - _ord(np.where(np.isfinite(g), g, F32(0)))) <= 4)
    plain = o.astype(np.float64) > thr
    narrowed = predicate(a, b, thr_f, hi=F32(1.0))
    return {"prev": int((live & (d == -1)).sum()), "eq": int((live & (d == 0)).sum()),
            "next": int((live & (d == 1)).sum()),
            "band": int((live & (inter >= tlo) & (inter <= thi)).sum()),
            "hi_edge": int(edge(thi).sum()), "lo_edge": int(edge(tlo).sum()),
            "guard": int((live & (narrowed != plain)).sum()),
            "range": int((live & ((t <= F32(1e-30)) | (t >= F32(1e30)))).sum())}


def census(boxes, thr, groups=None, chunk=256):
    """Edge counts over every unordered pair of `boxes` (n, 4) fp32 (pairs of different `groups` are skipped: boxes
    that NMS never compares, e.g. of different categories):
      prev / eq / next   fp32 IoU == prev(thr_f) / thr_f / next(thr_f)
      band               inter inside the guard band [fl(t * 0.999999f), fl(t * 1.000001f)], t = fl(thr_f * denom)
      hi_edge / lo_edge  inter within 4 ulps of the upper / lower guard
      guard              nms_suppresses with its upper guard narrowed to 1.0f disagrees with the plain formula
      range              t outside (1e-30, 1e30): the guards are skipped, the exact division decides"""
    b = np.ascontiguousarray(np.asarray(boxes, dtype=F32).reshape(-1, 4))
    g = None if groups is None else np.asarray(groups).reshape(-1)
    n = b.shape[0]
    tot = dict.fromkeys(CENSUS_KEYS, 0)
    for s in range(0, n, chunk):
        i = np.arange(s, min(n, s + chunk))
        ii, jj = np.nonzero(np.arange(n)[None, :] > i[:, None])
        ii = i[ii]
        # only pairs whose boxes can intersect (x and y ranges overlap, NaN kept) are worth the fp32 evaluation
        bi, bj = b[ii], b[jj]
        with np.errstate(invalid="ignore"):
            sep = (bi[:, 2] < bj[:, 0]) | (bj[:, 2] < bi[:, 0]) | (bi[:, 3] < bj[:, 1]) | (bj[:, 3] < bi[:, 1])
        keep = ~sep
        if g is not None:
            keep &= g[ii] == g[jj]
        c = _pair_census(bi[keep], bj[keep], thr)
        for k in CENSUS_KEYS:
            tot[k] += c[k]
    return tot


def assert_census(c, *need, least=1):
    """Each named count of census `c` is at least `least`."""
    low = {k: c[k] for k in need if c[k] < least}
    assert not low, f"too few knife-edge pairs {low} (census {c})"


# ---------------------------------------------------------------------------------------------------------------------
# generators: box a and a partner b with real IoU exactly thr, one coordinate of b stepped by up to +-40 ulps
# ---------------------------------------------------------------------------------------------------------------------
KSTEP = 40
# magnitude families: (x base, y base, pitch, side range).  Pair p sits in its own cell of a grid of the given pitch,
# so that pairs never meet; sides are drawn from the range (thin: width 1e4 x height)
FAMILIES = {
    "unit":     (20.0, 20.0, 400.0, (16.0, 180.0)),
    "near0":    (-0.3, -0.3, 0.02, (1e-3, 8e-3)),
    "neg":      (-500.0, -500.0, -400.0, (16.0, 180.0)),
    "e4":       (1e4, 1e4, 400.0, (16.0, 180.0)),
    "neg_e4":   (-1.2e4, -1.2e4, -400.0, (16.0, 180.0)),
    "e6":       (1e6, 1e6, 500.0, (40.0, 220.0)),
    "neg_e6":   (-1.01e6, -1.01e6, -500.0, (40.0, 220.0)),
    "thin":     (10.0, -50.0, -0.1, (0.01, 0.04)),     # width = 1e4 x height, one column of cells going down
    "thin_g":   (10.0, -200.0, -0.1, (0.01, 0.04)),   # a second column: the long search for guard pairs
    "e10":      (1e10, 1e10, 4e8, (4e7, 2e8)),
    "e14":      (1e14, 1e14, 4e12, (4e11, 2e12)),
    "e15":      (2e15, 2e15, 4e13, (4e12, 2e13)),      # above the spatial index's 1e15 cut-off
    "origin":   (0.0, 0.0, 0.0, (16.0, 180.0)),        # every cell at the origin (second-stage boxes, part 3)
}
DEFAULT_FAMILIES = ("unit", "near0", "neg", "e4", "neg_e4", "e6", "neg_e6", "thin")
MAX_CELLS = 400   # per family except "thin": keeps the families' regions apart
GEOMETRIES = ("nested", "corner", "shift")


def _cells(family, n, rng):
    """Lower-left corners and sides of n boxes of a magnitude family (a name of FAMILIES or such a tuple), one per cell
    of a grid (a negative pitch lays the grid out towards -inf), so that boxes of different cells never meet."""
    x0, y0, pitch, (lo, hi) = FAMILIES[family] if isinstance(family, str) else family
    k = np.arange(n)
    if family in ("thin", "thin_g"):
        h = rng.uniform(lo, hi, n)
        return np.full(n, x0), y0 + k * pitch, h * 1e4, h
    assert n <= MAX_CELLS
    cols = 20
    w, h = rng.uniform(lo, hi, n), rng.uniform(lo, hi, n)
    x, y = x0 + (k % cols) * pitch, y0 + (k // cols) * pitch
    if family == "near0":   # straddle zero: coordinates of both signs and magnitudes down to the side length
        x, y = x - cols * pitch / 2, y - cols * pitch / 2
    return x, y, w, h


def _base_pairs(geometry, thr, x, y, w, h):
    """(a, b0, stepped coordinates): b0 has real IoU thr with a before rounding."""
    a = np.stack([x, y, x + w, y + h], 1)
    if geometry == "nested":     # b shares a's y-range and left edge: IoU = b.w / a.w
        b = np.stack([x, y, x + thr * w, y + h], 1)
        return a.astype(F32), b.astype(F32), (2,)
    if geometry == "corner":     # equal boxes shifted diagonally by (1-s) of a side: IoU = s^2 / (2 - s^2)
        s = math.sqrt(2 * thr / (1 + thr))
        b = np.stack([x + (1 - s) * w, y + (1 - s) * h, x + (1 - s) * w + w, y + (1 - s) * h + h], 1)
        return a.astype(F32), b.astype(F32), (0, 1)
    if geometry == "shift":      # equal boxes shifted in x by d: IoU = (w - d) / (w + d)
        d = w * (1 - thr) / (1 + thr)
        b = np.stack([x + d, y, x + d + w, y + h], 1)
        return a.astype(F32), b.astype(F32), (0, 2)
    raise AssertionError(geometry)


def _classify(a, b, thr):
    """Per candidate pair: the census class it belongs to, or ''.  Where several apply, the rarer wins: guard over
    prev / eq / next over the guard-boundary classes."""
    thr_f = thr_below(thr)
    inter, denom = _inter_denom(a, b)
    with np.errstate(all="ignore"):
        o = inter / denom
        t = thr_f * denom
        thi, tlo = t * GUARD_HI, t * GUARD_LO
    d = _ord(o) - _ord(thr_f)
    plain = o.astype(np.float64) > thr
    guard = predicate(a, b, thr_f, hi=F32(1.0)) != plain
    out = np.full(inter.shape, "", dtype=object)
    for name, m in (("lo_edge", np.abs(_ord(inter) - _ord(tlo)) <= 2), ("hi_edge", np.abs(_ord(inter) - _ord(thi)) <= 2),
                    ("next", d == 1), ("eq", d == 0), ("prev", d == -1), ("guard", guard)):
        out[m & (inter > 0)] = name
    return out


CLASS_ORDER = ("guard", "prev", "eq", "next", "hi_edge", "lo_edge")


def edge_pairs(thr, n, family="unit", seed=0, geometries=GEOMETRIES, cells=None, only=None, transform=None):
    """Up to n pairs (a, b) (each (n, 4) fp32) of one magnitude family, laid out so that no two pairs meet; pair p has
    geometry geometries[p % len] and aims at class CLASS_ORDER[1 + p % 5] -- guard-distinguishing pairs are taken
    wherever the ulp search meets one -- falling back to any edge class.  `cells` (default n) cells are searched;
    `only` restricts the classes taken; with `transform` the classes are those of transform(a), transform(b) (the
    boxes a kernel derives from the ones passed in).  Returns (a, b, classes)."""
    rng = np.random.default_rng(seed)
    nc = n if cells is None else cells
    x, y, w, h = _cells(family, nc, rng)
    ks = np.arange(-KSTEP, KSTEP + 1)
    a = np.zeros((nc, 4), F32)
    B = np.zeros((nc, ks.size, 4), F32)
    for gi, geo in enumerate(geometries):
        sel = np.arange(nc) % len(geometries) == gi
        ag, bg, coords = _base_pairs(geo, thr, x[sel], y[sel], w[sel], h[sel])
        Bg = np.repeat(bg[:, None, :], ks.size, 1)
        for c in coords:
            Bg[:, :, c] = ulp_step(Bg[:, :, c], ks[None, :])
        a[sel], B[sel] = ag, Bg
    A = np.repeat(a[:, None, :], ks.size, 1)
    cls = _classify(A, B, thr) if transform is None else _classify(transform(A), transform(B), thr)
    keep_a, keep_b, got = [], [], []
    for p in range(nc):
        if len(got) == n:
            break
        row = cls[p]
        for c in ("guard", CLASS_ORDER[1 + p % 5]) + CLASS_ORDER:
            if only is not None and c not in only:
                continue
            hit = np.nonzero(row == c)[0]
            if hit.size:
                keep_a.append(a[p]); keep_b.append(B[p, hit[rng.integers(hit.size)]]); got.append(c)
                break
    if not got:
        return np.zeros((0, 4), F32), np.zeros((0, 4), F32), []
    return np.stack(keep_a).astype(F32), np.stack(keep_b).astype(F32), got


def edge_boxes(thr, n_per, families=DEFAULT_FAMILIES, seed=0):
    """Edge pairs of several families (disjoint regions of the plane), interleaved a0, b0, a1, b1, ... as (2P, 4)."""
    boxes = []
    for fi, fam in enumerate(families):
        a, b, _ = edge_pairs(thr, n_per, fam, seed=seed * 100 + fi)
        boxes.append(np.stack([a, b], 1).reshape(-1, 4))
    return np.concatenate(boxes, 0)


def guard_boxes(thr, n, seed=0):
    """Up to n guard-distinguishing pairs (see census), from a long search of thin boxes, as (2P, 4)."""
    a, b, _ = edge_pairs(thr, n, "thin_g", seed=seed, cells=6000, only=("guard",))
    return np.stack([a, b], 1).reshape(-1, 4)


def widening_pairs(n, mag, x0, y0, seed=0):
    """Pairs that only the spatial index's widening m keeps correct: a suppresses b at 0.5 (fp32 IoU > 0.5) although
    the rounded centre fl(0.5 * (a.x1 + a.x2)) lies one ulp right of b's right edge.  b = a's left half with
    b.x2 = prev(centre), both sharing a's y-range; a's left edge at x0 + ~mag, width and height are searched.  Pair p
    sits in its own row from y0 + p * step (step a power of two >= 64 mag, y0 a multiple of it), heights on a grid
    coarse enough that y + height is exact: every row has the heights of the search.  Returns (2P, 4)."""
    rng = np.random.default_rng(seed)
    m = 30000
    step = 2.0 ** math.ceil(math.log2(64 * mag))
    assert y0 % step == 0
    u = float(np.spacing(F32(abs(y0) + (n + 1) * step)))
    x1 = (x0 + mag * rng.uniform(1, 2, m)).astype(F32)
    x2 = (x1 + mag * rng.uniform(0.3, 3, m)).astype(F32)
    hgt = np.maximum(np.round(mag * rng.uniform(0.5, 50, m) / u), 1) * u
    a = np.stack([x1, np.zeros(m), x2, hgt], 1).astype(F32)
    centre = F32(0.5) * (a[:, 0] + a[:, 2])
    b = a.copy()
    b[:, 2] = ulp_step(centre, -1)
    hit = np.nonzero((ovr32(a, b).astype(np.float64) > 0.5) & (centre > b[:, 2]))[0][:n]
    a, b = a[hit], b[hit]
    y = (y0 + np.arange(hit.size) * step).astype(F32)
    for t in (a, b):
        t[:, 1], t[:, 3] = y, (y + t[:, 3]).astype(F32)
    assert np.array_equal(b[:, 3] - b[:, 1], hgt[hit].astype(F32))
    return np.stack([a, b], 1).reshape(-1, 4)


def pad_boxes(family, n, rng):
    """n ordinary random boxes of a family's magnitude, in a region beside its grid of edge pairs."""
    x0, y0, pitch, (lo, hi) = FAMILIES[family]
    if family.startswith("thin"):
        x0, pitch = x0 + 2e4, 400.0
    x = x0 + 30 * pitch + rng.uniform(0, 15, n) * pitch
    y = y0 + rng.uniform(0, 15, n) * pitch
    w, h = rng.uniform(lo, hi, n) * 2, rng.uniform(lo, hi, n) * 2
    return np.stack([x, y, x + w, y + h], 1).astype(F32)


def distinct_scores(n, rng):
    return ((rng.permutation(n) + 0.5) / n).astype(F32)


# ---------------------------------------------------------------------------------------------------------------------
# part 1: the reference, the census and the generators (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def O():
    from oracle import ref_torch
    return ref_torch


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_thr_below_is_the_largest_float_not_above(thr):
    f = thr_below(thr)
    assert float(f) <= thr < float(np.nextafter(f, F32(np.inf), dtype=F32))
    v = ulp_step(f, np.arange(-3, 4))
    assert np.array_equal(v.astype(np.float64) > thr, v > f)


@pytest.mark.parametrize("thr", THRESHOLDS)
@pytest.mark.parametrize("family", DEFAULT_FAMILIES)
def test_generator_reaches_every_ulp_offset(thr, family):
    """Each family, at each threshold, yields pairs at prev(thr_f), thr_f and next(thr_f) (the coarse e6 families
    step IoU by several ulps, and at 0.05 the others meet the edge rarely: there, at least one of the three) and
    inside the guard band."""
    a, b, got = edge_pairs(thr, 400, family, seed=3)
    c = census(np.stack([a, b], 1).reshape(-1, 4), thr)
    hits = [k for k in ("prev", "eq", "next") if c[k] > 0]
    assert len(hits) >= (3 if family in ("unit", "neg", "thin") else 1), c
    assert_census(c, "band", least=len(got) // 2)


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_generator_reaches_the_guard_boundaries(thr):
    """All families together: every ulp offset and both guard boundaries, many times over."""
    c = census(edge_boxes(thr, 200, seed=4), thr)
    assert_census(c, "prev", "eq", "next", "band", "hi_edge", "lo_edge", least=10)


@pytest.mark.parametrize("thr,least", [(0.3, 24), (0.05, 12), (0.7, 12), (0.6, 12)])
def test_guard_distinguishing_pairs_exist(thr, least):
    """Pairs on which the upper guard narrowed to 1.0f decides wrongly: the ones a narrowed band would break."""
    bx = guard_boxes(thr, 40)
    a, b = bx[0::2], bx[1::2]
    c = census(bx, thr)
    assert c["guard"] >= least, c
    thr_f = thr_below(thr)
    plain = ovr32(a, b).astype(np.float64) > thr
    assert np.array_equal(predicate(a, b, thr_f), plain)   # the real guards agree with the plain formula
    assert not np.array_equal(predicate(a, b, thr_f, hi=F32(1.0)), plain)


def test_widening_pairs_need_the_widening():
    for mag in (1e-3, 1.0, 1e4, 1e6, 1e10, 1e14):
        bx = widening_pairs(8, mag, 0.0, 0.0, seed=int(math.log10(mag) + 10))
        assert bx.shape[0] == 16, mag
        a, b = bx[0::2], bx[1::2]
        assert (ovr32(a, b).astype(np.float64) > 0.5).all()
        centre = F32(0.5) * (a[:, 0] + a[:, 2])
        assert (centre > b[:, 2]).all() and (ulp_step(centre, -1) == b[:, 2]).all()


def test_range_edges_take_the_exact_path():
    """t = thr_f * denom near 1e-30 (sides ~1e-15) and near 1e30 (sides ~1e15): the guards are skipped."""
    thr = 0.5
    tiny = np.array([[0, 0, 2e-15, 1e-15], [0, 0, 1e-15, 1e-15]], F32)
    huge = np.array([[0, 0, 2.2e15, 1e15], [0, 0, 1.1e15, 1e15]], F32)
    for bx in (tiny, huge):
        c = census(bx, thr)
        assert c["range"] == 1, c
        assert predicate(bx[0], bx[1], thr_below(thr)) == suppresses(bx[0], bx[1], thr)


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_suppresses_agrees_with_the_oracle_on_two_boxes(O, thr):
    """Two-box NMS of the C oracle: box 1 survives iff the reference here says box 0 does not suppress it."""
    bx = np.concatenate([edge_boxes(thr, 12, seed=5), guard_boxes(thr, 4)], 0)
    wide = np.concatenate([bx, widening_pairs(2, 1.0, 0.0, 0.0)], 0)
    s = torch.tensor([1.0, 0.5])
    for k in range(0, wide.shape[0], 2):
        a, b = wide[k], wide[k + 1]
        got = O.nms(torch.from_numpy(wide[k:k + 2].copy()), s, thr).tolist()
        assert got == ([0] if suppresses(a, b, thr) else [0, 1]), (a, b)
        assert bool(predicate(a, b, thr_below(thr))) == suppresses(a, b, thr)


# ---------------------------------------------------------------------------------------------------------------------
# part 2: det_nms_batched (nms_images / batched_nms / nms), bit-exact against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def det():
    import det_b200
    return det_b200


def knife_image(thr, n, ncat, seed, n_per=40, pad_family="unit"):
    """(boxes (n, 4), scores (n,), categories (n,)): edge pairs of every family plus guard pairs, both boxes of a pair in
    one category, the rest ordinary boxes far away.  Pairs get the best scores (they survive any top-k cut)."""
    rng = np.random.default_rng(seed)
    bx = np.concatenate([edge_boxes(thr, n_per, seed=seed), guard_boxes(thr, 30, seed=seed)], 0)
    assert bx.shape[0] <= n
    pc = np.repeat(rng.integers(0, ncat, bx.shape[0] // 2), 2)
    pad = pad_boxes(pad_family, n - bx.shape[0], rng)
    boxes = np.concatenate([bx, pad], 0)
    cats = np.concatenate([pc, rng.integers(0, ncat, pad.shape[0])])
    s = distinct_scores(n, rng)
    s = np.concatenate([np.sort(s)[::-1][:bx.shape[0]][rng.permutation(bx.shape[0])], np.sort(s)[::-1][bx.shape[0]:]])
    perm = rng.permutation(n)   # pairs spread over the image's rows
    return boxes[perm], s[perm].astype(F32), cats[perm]


def _with_nan(boxes, scores, cats):
    """The image plus one box with a NaN coordinate, far from everything: the NaN-safe predicate (NONAN = false)."""
    nb = np.array([[-9e5, -9e5, np.nan, -8.9e5]], F32)
    return (np.concatenate([boxes, nb]), np.concatenate([scores, F32([0.123457])]),
            np.concatenate([cats, cats[:1]]))


def _check_images(det, O, imgs, thr, max_out=None, mode=0):
    """nms_images over a padded batch of (boxes, scores, cats) images against the oracle's batched_nms per image."""
    n = len(imgs)
    m = max(b.shape[0] for b, _, _ in imgs)
    B = torch.zeros(n, m, 4)
    S = torch.zeros(n, m)
    C = torch.zeros(n, m, dtype=torch.int64)
    for i, (b, s, c) in enumerate(imgs):
        B[i, :b.shape[0]], S[i, :b.shape[0]], C[i, :b.shape[0]] = torch.from_numpy(b), torch.from_numpy(s), torch.from_numpy(c)
    counts = torch.tensor([b.shape[0] for b, _, _ in imgs], dtype=torch.int32)
    keep, kc = det.nms_images(B.cuda(), S.cuda(), C.cuda(), counts.cuda(), thr, max_out=max_out, mode=mode)
    keep, kc = keep.cpu(), kc.cpu()
    for i in range(n):
        k = int(counts[i])
        if mode == 1:
            want = _per_category(O, B[i, :k], S[i, :k], C[i, :k], thr)
        elif mode == 2:
            want = _offset_trick(O, B[i, :k], S[i, :k], C[i, :k], thr)
        else:
            want = O.batched_nms(B[i, :k], S[i, :k], C[i, :k], thr)
        if max_out is not None:
            want = want[:max_out]
        assert int(kc[i]) == want.numel(), (i, int(kc[i]), want.numel())
        assert torch.equal(keep[i, :want.numel()], want), i


def _per_category(O, b, s, c, thr):
    hit = torch.zeros(b.shape[0], dtype=torch.bool)
    for cat in torch.unique(c):
        mem = torch.nonzero(c == cat, as_tuple=True)[0]
        hit[mem[O.nms(b[mem], s[mem], thr)]] = True
    kept = torch.nonzero(hit, as_tuple=True)[0]
    return kept[O.stable_desc_order(s[kept])]


def shifted(boxes, cats):
    """torchvision's offset trick in fp32: box + category * (max coordinate + 1)."""
    b = torch.from_numpy(np.ascontiguousarray(boxes, dtype=F32))
    span = b.max() + torch.tensor(1).to(b)
    return (b + (torch.from_numpy(np.asarray(cats)).to(b) * span)[:, None]).numpy()


def _offset_trick(O, b, s, c, thr):
    return O.nms(torch.from_numpy(shifted(b.numpy(), c.numpy())), s, thr)


# route: (boxes per image, categories, max_out, mode): the path det_nms_batched takes for the pairs' segments
ROUTES = {
    "small_trick": (900, 4, None, 0),        # nms_small_kernel, <= 1000 boxes: offset trick
    "small_percat": (1500, 3, None, 0),      # nms_small_kernel, per category
    "warp": (4600, 24, None, 1),             # large path, segments <= 256: warp sweep
    "cta": (6000, 3, None, 1),               # large path, segments 257..4096: CTA sweep (spatial index at thr_f >= 0.5)
    "huge": (6000, 1, None, 1),              # one segment > 4096: cooperative sweep
    "topk": (6000, 3, 100, 0),               # max_out << boxes: top-k tier (pairs hold the best scores)
}
GPU_THRESHOLDS = (0.5, 0.7, 0.3, 0.6, 0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("nan", [False, True])
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("thr", GPU_THRESHOLDS)
def test_nms_images_knife_edge_routes(det, O, thr, route, nan):
    n, ncat, max_out, mode = ROUTES[route]
    b, s, c = knife_image(thr, n, ncat, seed=11)
    if nan:
        b, s, c = _with_nan(b, s, c)
        if route == "small_trick":   # a NaN coordinate makes the trick's span NaN: compare per category instead
            route, mode = "small_percat", 1
    seg = np.bincount(c, minlength=ncat)
    if route == "warp":
        assert seg.max() <= 256 and b.shape[0] > 4096
    elif route == "cta":
        assert 256 < seg.min() and seg.max() <= 4096
    elif route == "huge":
        assert seg.max() > 4096
    cen = census(shifted(b, c), thr) if route == "small_trick" else census(b, thr, groups=c)
    assert_census(cen, "prev", "eq", "next", "band", "hi_edge", "lo_edge")
    if thr in (0.3, 0.05, 0.6, 0.7):
        assert_census(cen, "guard")
    # a second image with a different draw rides along (images of a batch are independent)
    b2, s2, c2 = knife_image(thr, n - 37, ncat, seed=12)
    _check_images(det, O, [(b, s, c), (b2, s2, c2)], thr, max_out, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("thr", GPU_THRESHOLDS)
def test_batched_nms_and_nms_knife_edge(det, O, thr):
    """The single-image wrappers: batched_nms (small image, offset trick) and nms (one category)."""
    b, s, c = knife_image(thr, 800, 3, seed=21)
    sc = census(shifted(b, c), thr)
    assert_census(sc, "band")
    assert sc["prev"] + sc["eq"] + sc["next"] > 0, sc
    bt, st, ct = torch.from_numpy(b), torch.from_numpy(s), torch.from_numpy(c)
    assert torch.equal(det.batched_nms(bt.cuda(), st.cuda(), ct.cuda(), thr).cpu(), O.batched_nms(bt, st, ct, thr))
    assert_census(census(b, thr), "prev", "eq", "next", "band", "guard" if thr != 0.5 else "band")
    assert torch.equal(det.nms(bt.cuda(), st.cuda(), thr).cpu(), O.nms(bt, st, thr))


# ---- offset trick: pairs on the edge after the shift, and pairs on the edge before it --------------------------------
SPAN_MAX = 2e4   # the image's largest coordinate (held by one box): span = 20001


def trick_image(thr, n, seed):
    """Categories 0..3.  Pairs on the edge in raw coordinates (negative families only in category 0, which is not
    moved, so that no shifted box reaches another category), and pairs built on the edge in SHIFTED coordinates:
    X in [off, 2 off), raw x = X - off exactly (Sterbenz), so fl(x + off) == X.  Returns boxes, scores, cats and the
    rows of the shifted-space pairs."""
    rng = np.random.default_rng(seed)
    span = F32(SPAN_MAX + 1)
    raw_fam = ("unit", "near0", "neg", "e4", "neg_e4", "thin")
    parts, cats = [], []
    for fi, fam in enumerate(raw_fam):
        a, b, _ = edge_pairs(thr, 30, fam, seed=seed + fi)
        bx = np.stack([a, b], 1).reshape(-1, 4)
        parts.append(bx)
        cats.append(np.zeros(bx.shape[0], np.int64) if fam.startswith("neg") or fam == "near0"
                    else np.repeat(rng.integers(0, 4, bx.shape[0] // 2), 2))
    first_shift = sum(p.shape[0] for p in parts)
    for cat in (1, 2, 3):
        off = F32(cat) * span
        a, b, _ = edge_pairs(thr, 30, (float(off) + 200.0, float(off) + 200.0, 400.0, (16.0, 180.0)), seed=seed + 10 * cat)
        bx = np.stack([a, b], 1).reshape(-1, 4)
        raw = (bx - off).astype(F32)
        assert np.array_equal((raw + off).astype(F32), bx)
        parts.append(raw)
        cats.append(np.full(raw.shape[0], cat, np.int64))
    edge = np.concatenate(parts)
    ce = np.concatenate(cats)
    nshift = edge.shape[0] - first_shift
    top = np.array([[SPAN_MAX - 10, SPAN_MAX - 10, SPAN_MAX, SPAN_MAX]], F32)
    pad = pad_boxes("unit", n - edge.shape[0] - 1, rng)
    pad = pad[(pad < SPAN_MAX - 20).all(1)]
    boxes = np.concatenate([edge, top, pad]).astype(F32)
    cats_all = np.concatenate([ce, [0], rng.integers(0, 4, pad.shape[0])])
    assert boxes.max() == SPAN_MAX
    return boxes, distinct_scores(boxes.shape[0], rng), cats_all, np.arange(first_shift, first_shift + nshift)


@pytest.mark.gpu
@pytest.mark.parametrize("n,mode", [(1000, 0), (1000, 2), (2500, 2), (6000, 2)])
@pytest.mark.parametrize("thr", GPU_THRESHOLDS)
def test_offset_trick_knife_edge(det, O, thr, n, mode):
    """The trick on small (nms_small_kernel) and large images, automatic and forced.  No NaN variant: a NaN coordinate
    makes the span, and so every shifted box, NaN (the NaN-safe predicate is covered per category above)."""
    b, s, c, srows = trick_image(thr, n, seed=31)
    sh = shifted(b, c)
    before = census(b[:srows[0]], thr, groups=c[:srows[0]])   # raw pairs, compared within their category
    after = census(sh[srows], thr)                              # pairs built in shifted coordinates
    assert_census(before, "prev", "eq", "next", "band")
    assert_census(after, "band")
    assert after["prev"] + after["eq"] + after["next"] > 0, after
    assert_census(census(sh, thr), "prev", "eq", "next", "band")   # what the trick's one NMS compares
    _check_images(det, O, [(b, s, c)], thr, None, mode)


# ---- spatial index (nms_large.cuh large_bin_segments_kernel): CTA-class segments at thr_f >= 0.5 ----------------------
INDEX_MAX_ROUNDS = 48   # kBinRounds


def index_rounds(boxes, scores, thr):
    """Decision rounds large_bin_segments_kernel needs for one segment (step 4, evaluated synchronously: an upper
    bound of the kernel's count): a box with no better-scored suppressor is kept at once; then, per round, an
    undecided box dies if one of its suppressors is kept and is kept once all of them are dead."""
    n = boxes.shape[0]
    order = np.argsort(-scores, kind="stable")
    rank = np.empty(n, np.int64)
    rank[order] = np.arange(n)
    sup = [[] for _ in range(n)]
    for s in range(0, n, 256):
        i = np.arange(s, min(n, s + 256))
        bi, bj = boxes[i][:, None, :], boxes[None, :, :]
        meet = ~((bi[..., 2] < bj[..., 0]) | (bj[..., 2] < bi[..., 0]) | (bi[..., 3] < bj[..., 1]) | (bj[..., 3] < bi[..., 1]))
        ii, jj = np.nonzero(meet & (rank[None, :] < rank[i][:, None]))
        ii = i[ii]
        hit = ovr32(boxes[jj], boxes[ii]).astype(np.float64) > thr
        for a, b in zip(jj[hit], ii[hit]):
            sup[b].append(a)
    state = np.array([0 if sup[q] else 2 for q in range(n)])
    rounds = 0
    while (state == 0).any():
        rounds += 1
        new = state.copy()
        for q in np.nonzero(state == 0)[0]:
            st = state[sup[q]]
            new[q] = 1 if (st == 2).any() else (2 if (st == 1).all() else 0)
        state = new
        if rounds > INDEX_MAX_ROUNDS:
            break
    return rounds


def index_takes(boxes, scores, thr):
    """The criterion under which large_bin_segments_kernel decides a segment (nms_large.cuh:566-577, :677, :957): a
    segment of 257..4096 boxes, thr_f >= 0.5, every coordinate finite, every area 0 or inside [1e-30, 1e30],
    1e-20 < largest |coordinate| < 1e15, and a dependency chain of at most kBinRounds rounds."""
    area = (boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1])
    amax = float(np.abs(boxes).max())
    return (257 <= boxes.shape[0] <= 4096 and thr_below(thr) >= F32(0.5) and bool(np.isfinite(boxes).all())
            and not bool(((area > 0) & (area < F32(1e-30))).any()) and not bool((area > F32(1e30)).any())
            and 1e-20 < amax < 1e15 and index_rounds(boxes, scores, thr) <= INDEX_MAX_ROUNDS)


# (family of the edge pairs, magnitude and left edge of the widening pairs, segment length); one category each
INDEX_SEGMENTS = [("near0", 1e-3, 0.0, 300), ("unit", 1.0, 0.0, 700), ("e4", 1e3, 0.0, 1300),
                  ("e6", 1e5, 0.0, 2100), ("e10", 1e9, 0.0, 900), ("e14", 1e12, 0.0, 3000),
                  ("e15", None, None, 400)]   # above the 1e15 cut-off: the CTA sweep decides it


def index_image(thr, seed):
    rng = np.random.default_rng(seed)
    boxes, scores, cats, pairs = [], [], [], []
    for cat, (fam, mag, x0w, length) in enumerate(INDEX_SEGMENTS):
        a, b, _ = edge_pairs(thr, 60, fam, seed=seed + cat)
        half_a, half_b, _ = edge_pairs(0.5, 30, fam, seed=seed + 50 + cat, geometries=("nested",)) \
            if thr != 0.5 else (a[:0], b[:0], None)
        bx = [np.stack([a, b], 1).reshape(-1, 4)]
        if half_a.shape[0]:   # near-half containment (IoU around 0.5) in a second grid beside the first
            sh = F32(FAMILIES[fam][2] * 60)
            hb = np.stack([half_a, half_b], 1).reshape(-1, 4).copy()
            hb[:, 1::2] = (hb[:, 1::2] + sh).astype(F32)
            bx.append(hb)
        if mag is not None:
            bx.append(widening_pairs(8, mag, x0w, 0.0, seed=seed + 90 + cat))
            assert bx[-1].shape[0] == 16, fam
        if fam == "unit":   # guard-distinguishing pairs (thin boxes below the unit grid)
            bx.append(guard_boxes(thr, 20, seed=seed))
        bx = np.concatenate(bx).astype(F32)
        pad = pad_boxes(fam, length - bx.shape[0], rng)
        seg = np.concatenate([bx, pad])
        sc = distinct_scores(length, rng)
        pa, pb = np.arange(0, bx.shape[0], 2), np.arange(1, bx.shape[0], 2)
        hi, lo = np.maximum(sc[pa], sc[pb]), np.minimum(sc[pa], sc[pb])
        sc[pa], sc[pb] = hi, lo   # box a of every pair outranks its partner (the widening pairs need a to be kept)
        boxes.append(seg); scores.append(sc); cats.append(np.full(length, cat, np.int64))
        pairs.append(bx.shape[0])
    return boxes, scores, cats, pairs


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.5, 0.5 + 1e-12, 0.6, 0.7, 0.9])
def test_spatial_index_knife_edge(det, O, thr):
    """Segments of one image at magnitudes from 1e-3 to 1e14 (and one above the 1e15 cut-off), each holding edge pairs,
    near-half-containment pairs and pairs that only the index's widening m keeps correct, padded with ordinary boxes."""
    boxes, scores, cats, _ = index_image(thr, seed=41)
    for k, (b, s) in enumerate(zip(boxes, scores)):
        fam, mag = INDEX_SEGMENTS[k][:2]
        assert index_takes(b, s, thr) == (fam != "e15"), fam
        c = census(b, thr)
        assert_census(c, "band")
        assert c["prev"] + c["eq"] + c["next"] > 0, (fam, c)
        if mag is not None:   # 8 widening pairs: a suppresses b although a's rounded centre lies outside b
            a_, b_ = b[:-1], b[1:]
            centre = F32(0.5) * (a_[:, 0] + a_[:, 2])
            wide = (ovr32(a_, b_).astype(np.float64) > 0.5) & (centre > b_[:, 2]) & (a_[:, 0] == b_[:, 0]) \
                & (a_[:, 1] == b_[:, 1]) & (a_[:, 3] == b_[:, 3]) & (s[:-1] > s[1:])
            assert int(wide.sum()) >= 8, fam
    allb = np.concatenate(boxes)
    c = census(allb, thr, groups=np.concatenate(cats))
    assert_census(c, "prev", "eq", "next", "band", "hi_edge", "lo_edge")
    if thr in (0.6, 0.7):
        assert_census(c, "guard")
    half = census(allb, 0.5, groups=np.concatenate(cats))   # near-half containment: IoU around 1/2
    assert_census(half, "prev", "eq", "next")
    img = (allb, np.concatenate(scores), np.concatenate(cats))
    assert img[0].shape[0] > 4096   # the large path, where the index lives
    _check_images(det, O, [img], thr, None, 1)
    _check_images(det, O, [img, _with_nan(*img)], thr, None, 1)   # NaN: that image goes to the sweep, the other not


# ---------------------------------------------------------------------------------------------------------------------
# part 3: the other routes -- RPN proposals, second-stage detection (list NMS and det_nms_batched)
# ---------------------------------------------------------------------------------------------------------------------
def _rank_pairs_first(n_pairs_rows, n, rng):
    """Distinct scores with the first n_pairs_rows rows (pairs, box a first) above every other row, a above b."""
    s = np.sort(distinct_scores(n, rng))[::-1].copy()
    top = s[:n_pairs_rows].reshape(-1, 2)[rng.permutation(n_pairs_rows // 2)].reshape(-1)
    return np.concatenate([top, s[n_pairs_rows:][rng.permutation(n - n_pairs_rows)]]).astype(F32)


def rpn_level(thr, families, n, seed, widening=False):
    """One pyramid level of decoded proposals (inside a 30000 x 30000 image, so that clipping changes nothing) and
    logits: edge pairs (and widening pairs) with the best logits, then ordinary boxes."""
    rng = np.random.default_rng(seed)
    bx = [np.stack(edge_pairs(thr, 40, fam, seed=seed + k)[:2], 1).reshape(-1, 4) for k, fam in enumerate(families)]
    if widening:
        bx.append(widening_pairs(8, 1.0, 0.0, 0.0, seed=seed))
    bx = np.concatenate(bx)
    pad = pad_boxes(families[0], n - bx.shape[0], rng)
    boxes = np.concatenate([bx, pad]).astype(F32)
    assert boxes.min() >= 0 and boxes.max() <= 30000
    logits = (_rank_pairs_first(bx.shape[0], n, rng) * 8 - 4).astype(F32)
    perm = rng.permutation(n)
    return boxes[perm], logits[perm]


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.7, 0.5, 0.3])
def test_rpn_proposals_knife_edge(det, thr):
    """find_top_rpn_proposals on decoded boxes: a level of 5000 cut to pre_nms_topk = 3000 (a CTA-class segment: the
    spatial index at thr >= 0.5), a level of 200 (a short segment, riding in the index kernel) and one of 1000; the
    edge pairs hold the best logits, so they survive the per-level top-k.  Boxes, logits and counts bit-exact."""
    from oracle import ref_torch as R
    pre, post = 3000, 10000
    spec = [(("unit",), 5000, True), (("e4",), 200, False), (("unit", "e4"), 1000, False)]
    sizes = [(30000, 30000), (30000, 29000)]
    props, lgs, total = [], [], dict.fromkeys(CENSUS_KEYS, 0)
    for lvl, (fams, n, wide) in enumerate(spec):
        per_img = [rpn_level(thr, fams, n, seed=100 * lvl + i, widening=wide) for i in range(len(sizes))]
        b = np.stack([p[0] for p in per_img])
        l = np.stack([p[1] for p in per_img])
        for i in range(len(sizes)):   # census on what the level's NMS sees: its top-`pre` boxes
            top = np.argsort(-l[i], kind="stable")[:min(pre, n)]
            c = census(b[i, top], thr)
            for k in CENSUS_KEYS:
                total[k] += c[k]
        props.append(torch.from_numpy(b))
        lgs.append(torch.from_numpy(l))
    assert_census(total, "prev", "eq", "next", "band")
    want = R.find_top_rpn_proposals([p.clone() for p in props], lgs, sizes, thr, pre, post, 0.0, False)
    got = det.find_top_rpn_proposals([p.cuda() for p in props], [l.cuda() for l in lgs], sizes, thr, pre, post, 0.0,
                                     False)
    for i in range(len(sizes)):
        wb, ws = want[i]
        assert len(got[i]) == wb.shape[0], (i, len(got[i]), wb.shape[0])
        assert torch.equal(got[i].objectness_logits.cpu(), ws), i
        assert torch.equal(got[i].proposal_boxes.tensor.cpu(), wb), i


def zero_delta_decode(p):
    """Box2BoxTransform.apply_deltas with zero deltas (common.cuh decode_delta): what the second stage makes of a
    proposal.  Exact for a box with a corner at the origin; elsewhere it may move a corner by an ulp."""
    p = np.asarray(p, dtype=F32)
    w, h = p[..., 2] - p[..., 0], p[..., 3] - p[..., 1]
    cx, cy = p[..., 0] + F32(0.5) * w, p[..., 1] + F32(0.5) * h
    pcx, pcy = F32(0) * w + cx, F32(0) * h + cy
    pw, ph = F32(1) * w, F32(1) * h
    return np.stack([pcx - F32(0.5) * pw, pcy - F32(0.5) * ph, pcx + F32(0.5) * pw, pcy + F32(0.5) * ph], -1)


@pytest.mark.gpu
@pytest.mark.parametrize("body", ["fast", "general"])
@pytest.mark.parametrize("thr", [0.5, 0.7, 0.3, 0.05])
def test_roi_detect_list_nms_knife_edge(det, thr, body):
    """FastRCNNOutputs.inference_batched (det_roi_detect_typed: list NMS) with zero deltas, so that every detection box
    is its proposal decoded: pairs built on the edge AFTER the decode.  fast: one pair per class (the fast form);
    general: every pair in one class (more than 200 candidates in a category bucket: the general body).  Per-category
    NMS (mode 1).  The census runs on the decoded boxes, checked bit for bit against the kernel's kept boxes."""
    from tests.test_gpu_roi_detect import check_against_oracle, run
    from tests import fast_rcnn_oracle as FO
    npair = 110
    a, b, _ = edge_pairs(thr, npair, "origin", seed=7, geometries=("nested",), transform=zero_delta_decode)
    assert a.shape[0] >= 100
    npair = a.shape[0]
    props = np.stack([a, b], 1).reshape(-1, 4)
    rows = props.shape[0]
    K = npair if body == "fast" else 2
    cls = np.repeat(np.arange(npair) % K if body == "fast" else np.zeros(npair, np.int64), 2)
    rng = np.random.default_rng(3)
    logits = np.full((rows, K + 1), -8.0, F32)
    logits[np.arange(rows), cls] = _rank_pairs_first(rows, rows, rng) * 4 + 4   # box a of a pair outranks b
    dec = zero_delta_decode(props)
    cen = census(dec, thr, groups=cls)
    assert_census(cen, "prev", "eq", "next", "band")
    counts, sizes = [rows], [(400, 400)]
    lg, dl, pr = torch.from_numpy(logits), torch.zeros(rows, 4 * K), torch.from_numpy(props)
    r = run(det, K, lg, dl, pr, counts, sizes, thr=0.05, iou=thr, topk=-1, mode=1)
    assert int(r["overflow"].item()) == 0
    cnt = check_against_oracle(FO, r, lg, dl, pr, counts, sizes, 0.05, thr, -1, 1)
    k = int(cnt[0])
    kept_rows = (r["idx"][0, :k] // K).cpu().numpy()
    assert np.array_equal(r["boxes"][0, :k].cpu().numpy().view(np.int32), dec[kept_rows].view(np.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.5, 0.7, 0.3, 0.05])
def test_fast_rcnn_inference_decoded_knife_edge(det, thr):
    """fast_rcnn_inference on boxes and probabilities the caller decoded (det_nms_batched behind it, offset trick
    for this image size): edge pairs of non-negative coordinates inside the frame, each pair in one class.  The census
    runs on the boxes the trick compares: shifted by class * (largest coordinate + 1)."""
    from tests import fast_rcnn_oracle as FO
    rng = np.random.default_rng(5)
    bx = edge_boxes(thr, 200, families=("unit", "e4"), seed=9)
    K, rows = 3, bx.shape[0]
    cls = np.repeat(np.where(np.arange(rows // 2) % 2 == 0, 0, rng.integers(1, K, rows // 2)), 2)   # class 0: no shift
    boxes = np.tile(bx, (1, K))
    probs = np.full((rows, K + 1), 0.001, F32)
    probs[np.arange(rows), cls] = _rank_pairs_first(rows, rows, rng) * 0.5 + 0.4
    assert_census(census(bx, thr, groups=cls), "prev", "eq", "next", "band")
    assert rows <= 1000   # the candidates go through the offset trick: census on the shifted boxes as well
    assert_census(census(shifted(bx, cls), thr), "prev", "eq", "next", "band")
    size = (40000, 40000)
    bt, pt = torch.from_numpy(boxes), torch.from_numpy(probs)
    results, kept = det.fast_rcnn_inference([bt.cuda()], [pt.cuda()], [size], 0.05, thr, -1)
    wi, wb, ws, wc = FO.fast_rcnn_select_single_image(pt, bt.reshape(rows, K, 4), torch.ones(rows, dtype=torch.bool),
                                                      0.05, thr, -1)
    assert len(results[0]) == wi.numel()
    assert torch.equal(kept[0].cpu(), wi // K) and torch.equal(results[0].pred_classes.cpu(), wc)
    assert torch.equal(results[0].pred_boxes.tensor.cpu(), wb) and torch.equal(results[0].scores.cpu(), ws)


def _yolo_edge_logits(thr, row, col, want, salt, u):
    """Logits (tw, th) of predictor 0 of cell (row, col) of the 448 x 448, 7 x 7 grid (priors 64 and 192, x = y = 0;
    predictor 1 has logits u = (tw1, th1)) whose box and predictor 1's box have an fp32 IoU of class `want`, aimed with
    torch's fp32 decode on the CPU (exp(t) * prior, centre +- half the side; both sides are searched, since one side's
    rounding alone skips IoU values); the census then checks the kernel's own boxes.  The `salt`-th hit is taken."""
    t0 = F32(math.log(3 * math.sqrt(thr)) + 0.5 * (u[0] + u[1]))
    tw, th = np.meshgrid(ulp_step(t0, np.arange(-30, 31)), ulp_step(t0, np.arange(-30, 31)))
    tw, th = torch.from_numpy(tw.reshape(-1)), torch.from_numpy(th.reshape(-1))
    cx, cy = (0.5 + col) * 64.0, (0.5 + row) * 64.0

    def box(w, h):
        return torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], -1).numpy()
    b0 = box(torch.exp(tw) * 64.0, torch.exp(th) * 64.0)
    u = torch.tensor(u, dtype=torch.float32)
    b1 = np.repeat(box(torch.exp(u[0:1]) * 192.0, torch.exp(u[1:2]) * 192.0), b0.shape[0], 0)
    cls = _classify(b1, b0, thr)
    hit = np.nonzero(cls == want)[0]
    if hit.size == 0:
        hit = np.nonzero(cls != "")[0]
    j = hit[salt % hit.size]
    return float(tw[j]), float(th[j])


# ---- fused YOLO decode + NMS (yolo_fast.cuh fast path, and the generic kernel with clip=False) --------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("thr", [0.5, 0.7, 0.3])
def test_yolo_fused_knife_edge(det, thr, clip):
    """Logits x = y = 0 put both predictors of a cell on the same centre (sigmoid(0) is exactly 0.5), so their boxes
    are concentric and IoU = w0 h0 / w1 h1.  Predictor 1 gets small random tw, th; predictor 0 gets tw, th within 30
    ulps of the values that give real IoU thr (priors 64 vs 192), aimed at the three ulp offsets.  Only
    cells three apart are active, so different cells never meet.  The census runs on the kernel's own decoded boxes
    (return_dense); kept flat ids and counts bit-exact against the oracle's selection on those boxes and scores."""
    from oracle import ref_torch as R
    S, B, C, n = 7, 2, 20, 48
    yh = det.YoloGridHead(S, B, C, (448, 448), clip=clip)
    head = torch.full((n, S, S, B * 5 + C), -10.0)
    head[..., 0:2] = 0.0
    head[..., 5:7] = 0.0
    head[..., 2:4] = 0.0
    head[..., 7:9] = 0.0
    cells = [(1, 1), (1, 4), (4, 1), (4, 4), (1, 6) if not clip else (6, 6)]
    rng = np.random.default_rng(17)
    k = 0
    for i in range(n):
        for (r, c) in cells:
            u = [float(F32(v)) for v in rng.uniform(-0.1, 0.1, 2)]   # predictor 1: tw, th
            tw, th = _yolo_edge_logits(thr, r, c, ("prev", "eq", "next")[k % 3], k, u)
            k += 1
            head[i, r, c, 2], head[i, r, c, 3] = tw, th             # predictor 0
            head[i, r, c, 7], head[i, r, c, 8] = u[0], u[1]
            head[i, r, c, 4] = 3.0 + float(rng.uniform(0, 1))        # confidences: both predictors pass 0.25
            head[i, r, c, 9] = 3.0 + float(rng.uniform(0, 1))
            head[i, r, c, B * 5 + int(rng.integers(0, C))] = 4.0     # one class per cell
    r = yh.detect(head.cuda(), 0.25, thr, return_dense=True)
    gb, gs = r["dense_boxes"].cpu(), r["dense_scores"].cpu()
    bx = gb.numpy().reshape(n, S * S, B, 4)
    tot = dict.fromkeys(CENSUS_KEYS, 0)
    for i in range(n):
        for (rr, cc) in cells:
            c = census(bx[i, rr * S + cc], thr)
            for key in CENSUS_KEYS:
                tot[key] += c[key]
    assert_census(tot, "prev", "eq", "next", "band")
    for i in range(n):
        want, _, _, _ = R.yolo_select_nms(gb[i], gs[i], 0.25, thr)
        kk = int(r["count"][i])
        assert kk == want.numel() and torch.equal(r["flat"][i, :kk].cpu(), want), i


# ---- det_dense_detect (DenseAnchorHead.detect_thresholded: fused decode + list NMS) ------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("gate", [True, False])
@pytest.mark.parametrize("thr", [0.5, 0.7, 0.3])
def test_dense_detect_knife_edge(det, thr, gate):
    """The YOLO construction on a dense anchor head: one 8 x 8 level of stride 64, anchors 64 and 192, tx = ty = 0 so
    that the two anchors of a cell decode to concentric boxes, tw, th of anchor 0 aimed at the edge, of anchor 1
    small and random; active cells three apart, every candidate of class 0 (so the offset trick this candidate count
    selects moves nothing).  The census runs on the boxes decode() returns: the kernel's own values."""
    from tests.test_gpu_dense_detect import check_against_oracle
    A, C, H, n = 2, 4, 8, 24
    dh = det.DenseAnchorHead([64], [[[64.0, 64.0], [192.0, 192.0]]], C)
    head = torch.zeros(n, A, 5 + C, H, H)
    head[:, :, 4] = -10.0
    cells = [(r, c) for r in (1, 4, 7) for c in (1, 4, 7)]
    rng = np.random.default_rng(23)
    k = 0
    for i in range(n):
        for (r, c) in cells:
            u = [float(F32(v)) for v in rng.uniform(-0.1, 0.1, 2)]
            tw, th = _yolo_edge_logits(thr, r, c, ("prev", "eq", "next")[k % 3], k, u)
            k += 1
            head[i, 0, 2, r, c], head[i, 0, 3, r, c] = tw, th
            head[i, 1, 2, r, c], head[i, 1, 3, r, c] = u[0], u[1]
            head[i, :, 4, r, c] = torch.from_numpy(rng.uniform(3.0, 4.0, 2).astype(F32))
            head[i, :, 5, r, c] = 4.0
    heads = [head.reshape(n, A * (5 + C), H, H).cuda()]
    assert dh.fused_ok(heads)
    boxes = dh.decode(heads)[0].cpu().numpy().reshape(n, H, H, A, 4)
    tot = dict.fromkeys(CENSUS_KEYS, 0)
    for i in range(n):
        for (r, c) in cells:
            cen = census(boxes[i, r, c], thr)
            for key in CENSUS_KEYS:
                tot[key] += cen[key]
    assert_census(tot, "prev", "eq", "next", "band")
    r = dh.detect_thresholded(heads, 0.25, thr, max_det=300, cand_cap=1024, gate=gate, check=False)
    assert int(r["overflow"].item()) == 0
    from oracle import ref_torch as R
    check_against_oracle(dh, R, heads, r, 0.25, thr, 300)
