// Training side for GRID anchors (subsystem 4a on the layout AnchorGenerator really produces): IoU target assignment in
// one streaming pass, plus the sampled (sparse) loss forward + backward that reads the head where it lies (NCHW).
//
// Reference behaviour reproduced (paths relative to the reference root):
//   python/src/models/modules/anchor_generators.py:158-179   anchors of a level = shifts (h, w) + cell anchors, order (h, w, a)
//   python/src/models/rpn.py:161-168                           per image: pairwise_iou(gt, anchors) -> Matcher
//   python/src/models/components/matcher.py:53-120             column max / argmax, threshold buckets, low-quality promotion
//   python/src/models/rpn.py:187-244, components/box_regression.py:128-168   losses on the sampled anchors
//
// What the grid buys (the generic kernels of assign_loss.cu brute-force every anchor against every gt box, cull by the
// bounding box of 128 CONSECUTIVE anchors -- a 170-pixel strip of one feature-map row -- and need a second pass for the
// low-quality rule):
//   * match_rowmax_kernel (gt-centric): the anchors that can overlap a gt box form a closed-form (y, x) window per level
//     and cell anchor, so the row maximum of `pairwise_iou` is evaluated on that window only, and a whole (level, cell
//     anchor) is skipped once min(area)/max(area) -- an upper bound of its IoUs -- is below the running maximum.
//   * match_grid_kernel (anchor-centric): a warp owns an 8 x 4 TILE of positions (all A anchors of a position in one
//     lane); its bounding box is compact in both directions, so about half as many (gt, tile) pairs survive the cull as
//     with row strips.  The row maxima are already final, hence the low-quality promotion `IoU == row max`
//     (matcher.py:110-120, exact fp32 equality of the SAME pair_iou evaluation) is decided in the same pass: labels and
//     matched indices are written once, and there is no per-warp reduction, no atomic on row maxima and no second pass.
//     The kernel also counts positives / ignored anchors per image and lists the positives, which lets the sampler and
//     the loss work on O(sampled) instead of O(R) data.
// Anchor coordinates are always READ from the caller's (R, 4) table (802 KB, L2-resident): every IoU is the same fp32
// expression on the same bits as in the generic kernels, the grid layout only organises the work.
#include "common.cuh"
#include "peer.cuh"
#include "assign.cuh"

namespace det {

constexpr int kGridMaxLevels = 8;
constexpr int kTileW = 8, kTileH = 4;  // positions per warp tile (8 wide x 4 tall = one lane per position)
constexpr int kGridWarps = 8;          // warps (tiles) per CTA

struct GridLevelDev {
    int h, w, stride, tiles_x;
    int first_tile;
    int64_t first_row;
};
struct GridLayoutDev {
    GridLevelDev lv[kGridMaxLevels];
    int nlev, a, tiles_total;
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- K1: one warp per gt box: (1) marks the tiles of its image the box can overlap (bit `t` of mask[img][tile] for the
// image's t-th box, t < 32), (2) the row maximum of pairwise_iou(gt, anchors).
// stats (4 int32 per image: #positives, #ignored, 2 spare) are zeroed here for match_grid_kernel, which follows on the
// same stream; flags / mask are zeroed by the host's memset before the launch.
constexpr int kFlagPromoteAll = 1;  // some gt of the image has row maximum 0: `Q == rowmax` holds for EVERY anchor
constexpr int kFlagManyGt = 2;      // more than 32 gt boxes: the tile masks do not cover the image, cull on the fly

__device__ __forceinline__ int gt_image(const int32_t* __restrict__ gt_off, int n, int t) {
    int lo = 0, hi = n;  // the image with gt_off[img] <= t < gt_off[img + 1] (empty images are skipped by construction)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (gt_off[mid] <= t) lo = mid; else hi = mid;
    }
    return lo;
}

// positions x in [0, w) whose anchor [a_lo + x s, a_hi + x s] can reach the interval (g_lo, g_hi), one position of margin
__device__ __forceinline__ void reach_window(float g_lo, float g_hi, float a_lo, float a_hi, float s, int w, int& lo, int& hi) {
    const float f_lo = floorf((g_lo - a_hi) / s) - 1.0f, f_hi = ceilf((g_hi - a_lo) / s) + 1.0f;
    lo = (int)fminf(fmaxf(f_lo, 0.0f), (float)w);
    hi = (int)fmaxf(fminf(f_hi, (float)(w - 1)), -1.0f);
}

// positions whose overlap with (g_lo, g_hi) along one axis can be the LARGEST: with centre offset d the overlap is
// min(a_len, g_len, (a_len + g_len)/2 - |d|): constant on the plateau |d| <= |g_len - a_len| / 2 and strictly smaller
// by at least one stride for every further position.  IoU grows with the overlap of either axis, so a row maximum (and
// every anchor that EQUALS it) lies on plateau x plateau.  floor / ceil already round outwards; one more position of margin
// absorbs the rounding of the quotient (anchor coordinates are x * stride + offset: exact in fp32 at these sizes).
__device__ __forceinline__ void plateau_window(float g_lo, float g_hi, float a_lo, float a_hi, float s, int w, int& lo, int& hi) {
    const float gc = 0.5f * (g_lo + g_hi), ac = 0.5f * (a_lo + a_hi);
    const float half = 0.5f * fabsf((g_hi - g_lo) - (a_hi - a_lo));
    const float f_lo = floorf((gc - ac - half) / s) - 1.0f, f_hi = ceilf((gc - ac + half) / s) + 1.0f;
    // A plateau that lies beyond the feature map (a gt box sticking out of the image) is clamped ONTO the map, not cut
    // away: the overlap falls off monotonically with the distance from the plateau, so the best position that exists is
    // the border one.
    lo = (int)fminf(fmaxf(f_lo, 0.0f), (float)(w - 1));
    hi = (int)fmaxf(fminf(f_hi, (float)(w - 1)), 0.0f);
}

__global__ void __launch_bounds__(128, 10)
match_rowmax_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, int n, int64_t sum_g,
                    const float4* __restrict__ anchors, GridLayoutDev lay, int want_rowmax, float* __restrict__ rowmax,
                    int32_t* __restrict__ flags, uint32_t* __restrict__ mask, int32_t* __restrict__ stats,
                    int stats_words) {
    const unsigned FULLMASK = 0xffffffffu;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (stats && tid < stats_words) stats[tid] = 0;
    const int64_t t = tid >> 5;
    if (t >= sum_g) return;
    const int lane = threadIdx.x & 31;
    const float4 gb = gt[t];
    const float ga = box_area(gb);
    const bool finite = isfinite(gb.x) && isfinite(gb.y) && isfinite(gb.z) && isfinite(gb.w);
    const int A = lay.a, P = lay.nlev * A;  // (level, cell anchor) pairs, P <= 32: lane p looks after pair p
    float4 ab0 = make_float4(0.f, 0.f, 0.f, 0.f);
    float bound = -1.0f;
    if (lane < P) {
        ab0 = anchors[lay.lv[lane / A].first_row + lane % A];  // the pair's anchor at position (0, 0)
        const float aa = box_area(ab0);
        // IoU <= min(area) / max(area); anything doubtful (degenerate or non-finite boxes) is never pruned
        bound = (finite && ga > 0.0f && aa > 0.0f && isfinite(aa)) ? fminf(ga, aa) / fmaxf(ga, aa) : INFINITY;
    }
    // ---- (1) tile marks
    const int img = gt_image(gt_off, n, (int)t);
    const int tl = (int)t - gt_off[img];
    if (!mask) {
        // sample-list-only assignment (assign_candidates_kernel follows): no tile kernel, no masks
    } else if (tl >= 32) {
        if (lane == 0 && tl == 32) atomicOr(&flags[img], kFlagManyGt);
    } else {
        for (int l = 0; l < lay.nlev; ++l) {
            const GridLevelDev L = lay.lv[l];
            // union of the level's cell anchors at position (0, 0)
            float ux1 = INFINITY, uy1 = INFINITY, ux2 = -INFINITY, uy2 = -INFINITY;
            for (int a = 0; a < A; ++a) {
                ux1 = fminf(ux1, __shfl_sync(FULLMASK, ab0.x, l * A + a)); uy1 = fminf(uy1, __shfl_sync(FULLMASK, ab0.y, l * A + a));
                ux2 = fmaxf(ux2, __shfl_sync(FULLMASK, ab0.z, l * A + a)); uy2 = fmaxf(uy2, __shfl_sync(FULLMASK, ab0.w, l * A + a));
            }
            int x_lo = 0, x_hi = L.w - 1, y_lo = 0, y_hi = L.h - 1;
            if (finite && isfinite(ux1) && isfinite(uy1) && isfinite(ux2) && isfinite(uy2)) {
                reach_window(gb.x, gb.z, ux1, ux2, (float)L.stride, L.w, x_lo, x_hi);
                reach_window(gb.y, gb.w, uy1, uy2, (float)L.stride, L.h, y_lo, y_hi);
            }
            if (x_lo > x_hi || y_lo > y_hi) continue;
            const int tx_lo = x_lo / kTileW, tx_n = x_hi / kTileW - tx_lo + 1;
            const int ty_lo = y_lo / kTileH, ty_n = y_hi / kTileH - ty_lo + 1;
            uint32_t* __restrict__ row = mask + (int64_t)img * lay.tiles_total + L.first_tile;
            for (int k = lane; k < tx_n * ty_n; k += 32)
                atomicOr(&row[(ty_lo + k / tx_n) * L.tiles_x + tx_lo + k % tx_n], 1u << tl);
        }
    }
    if (!want_rowmax) return;
    // ---- (2) row maximum.  Lane p prepares pair p's plateau window once (the divisions run side by side instead of one
    // pair after the other); the sweep below fetches the window of the pair it works on with shuffles.
    int wx_lo = 0, wx_hi = -1, wy_lo = 0, wy_hi = -1;
    if (lane < P) {
        const GridLevelDev Lp = lay.lv[lane / A];
        wx_hi = Lp.w - 1;
        wy_hi = Lp.h - 1;
        if (finite && ga > 0.0f && isfinite(ab0.x) && isfinite(ab0.y) && isfinite(ab0.z) && isfinite(ab0.w) &&
            ab0.z > ab0.x && ab0.w > ab0.y) {
            plateau_window(gb.x, gb.z, ab0.x, ab0.z, (float)Lp.stride, Lp.w, wx_lo, wx_hi);
            plateau_window(gb.y, gb.w, ab0.y, ab0.w, (float)Lp.stride, Lp.h, wy_lo, wy_hi);
        }
    }
    float best = 0.0f;
    unsigned pending = __ballot_sync(FULLMASK, lane < P);
    while (pending) {
        // the pending pair with the largest bound
        const float mine = ((pending >> lane) & 1u) ? bound : -1.0f;
        const float bmax = warp_max(mine);
        if (bmax * 1.0001f < best) break;  // no remaining pair can reach (let alone equal) the maximum found so far
        const int src = __ffs(__ballot_sync(FULLMASK, mine == bmax)) - 1;
        pending &= ~(1u << src);
        const int x_lo = __shfl_sync(FULLMASK, wx_lo, src), x_hi = __shfl_sync(FULLMASK, wx_hi, src);
        const int y_lo = __shfl_sync(FULLMASK, wy_lo, src), y_hi = __shfl_sync(FULLMASK, wy_hi, src);
        const GridLevelDev L = lay.lv[src / A];
        const int a = src % A;
        float v = 0.0f;
        // the lanes sweep the window as an 8 x 4 patch (no integer division, 32-bit row arithmetic: r < 2^31 / 16)
        const float4* __restrict__ lvl = anchors + L.first_row + a;
        const int lx = lane & 7, ly = lane >> 3;
        for (int y = y_lo + ly; y <= y_hi; y += 4) {
            const int rowbase = y * L.w;
            for (int x = x_lo + lx; x <= x_hi; x += 8) {
                const float4 ab = lvl[(rowbase + x) * A];
                v = fmaxf(v, pair_iou(gb, ga, ab, box_area(ab)));  // same expression as match_grid_kernel
            }
        }
        best = fmaxf(best, warp_max(v));
    }
    if (lane == 0) {
        rowmax[t] = best;
        if (best == 0.0f) atomicOr(&flags[img], kFlagPromoteAll);
    }
}

// ---- sample-list-only assignment ("lazy"): the training step needs the <= num_samples sampled anchors of an image, not
// the labels of all R.  Positives are found from the gt side -- an anchor is positive only if its IoU with SOME gt box g
// reaches the lowest threshold of a positive bucket, or equals g's row maximum -- on closed-form windows around g;
// negatives are drawn by the sampler, which labels the few hundred anchors its permutation walk visits on the fly.
// Every label comes from anchor_verdict(), the same arithmetic as match_grid_kernel.
// positions whose overlap with the gt along one axis can be at least ov_min (centre offset |d| <= (a_len + g_len)/2 - ov_min)
__device__ __forceinline__ void overlap_window(float g_lo, float g_hi, float a_lo, float a_hi, float ov_min, float s, int w,
                                               int& lo, int& hi) {
    const float gc = 0.5f * (g_lo + g_hi), ac = 0.5f * (a_lo + a_hi);
    const float half = 0.5f * ((g_hi - g_lo) + (a_hi - a_lo)) - ov_min;
    if (!(half >= 0.0f)) {
        lo = 0;
        hi = -1;
        return;
    }
    const float f_lo = floorf((gc - ac - half) / s) - 1.0f, f_hi = ceilf((gc - ac + half) / s) + 1.0f;
    lo = (int)fminf(fmaxf(f_lo, 0.0f), (float)w);
    hi = (int)fmaxf(fminf(f_hi, (float)(w - 1)), -1.0f);
}

// one warp per gt box (row maxima are final: match_rowmax_kernel ran before).  Appends the image's positives
// (anchor row | label << 24, matched gt) to pos_list / pos_gt; stats[img*4+0] counts them.  An anchor that several boxes
// nominate is emitted by the first of them only (Verdict::first_q).
constexpr int kCandWarps = 4;   // warps (gt boxes) per CTA of match_rowmax_kernel / assign_candidates_kernel: small CTAs even
                                // out the very different amounts of work per box
constexpr int kHitCap = 128;    // nominated anchors buffered per warp before their verdicts are evaluated

__global__ void __launch_bounds__(kCandWarps * 32, 10)
assign_candidates_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, int n, int64_t sum_g,
                         const float4* __restrict__ anchors, GridLayoutDev lay, MatchRule rule, float tau,
                         const float* __restrict__ rowmax, const int32_t* __restrict__ flags, int32_t* __restrict__ stats,
                         int32_t* __restrict__ pos_list, int32_t* __restrict__ pos_gt, int list_cap) {
    __shared__ int s_hits[kCandWarps][kHitCap];
    const unsigned FULLMASK = 0xffffffffu;
    const int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= sum_g) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int img = gt_image(gt_off, n, (int)t);
    if (rule.allow_lq && (flags[img] & kFlagPromoteAll)) return;  // every anchor is positive: the sampler's dense path
    const int g0 = gt_off[img], G = gt_off[img + 1] - g0, tl = (int)t - g0;
    const float4 gb = gt[t];
    const float ga = box_area(gb);
    const bool lq = rule.allow_lq != 0;
    const float rm = lq ? rowmax[t] : -1.0f;
    const bool finite = isfinite(gb.x) && isfinite(gb.y) && isfinite(gb.z) && isfinite(gb.w) && ga > 0.0f;
    const int A = lay.a, P = lay.nlev * A;
    // lane p prepares the window of (level, cell anchor) pair p: the positions whose IoU with this box can reach tau
    // or equal the row maximum (empty for most pairs).  All the divisions of the 15 pairs run side by side.
    int wx_lo = 0, wx_hi = -1, wy_lo = 0, wy_hi = -1;
    if (lane < P) {
        const GridLevelDev L = lay.lv[lane / A];
        const float4 a0 = anchors[L.first_row + lane % A];
        const float aa = box_area(a0);
        wx_hi = L.w - 1;
        wy_hi = L.h - 1;  // anything doubtful (degenerate or non-finite boxes) sweeps the whole level
        if (finite && aa > 0.0f && isfinite(aa) && a0.z > a0.x && a0.w > a0.y) {
            const float bound = fminf(ga, aa) / fmaxf(ga, aa) * 1.0001f;  // IoU <= min(area) / max(area)
            const bool by_tau = bound >= tau, by_rm = lq && bound >= rm;
            // IoU >= tau needs inter >= tau * max(area), hence an x overlap of at least that over the largest possible y
            // overlap min(a_h, g_h) (and vice versa); IoU == row max lies on the plateau windows (match_rowmax_kernel)
            const float need = tau * fmaxf(ga, aa) * 0.9999f;
            int xa = 0, xb = -1, ya = 0, yb = -1, xc = 0, xd = -1, yc = 0, yd = -1;
            if (by_tau) {
                overlap_window(gb.x, gb.z, a0.x, a0.z, need / fminf(a0.w - a0.y, gb.w - gb.y), (float)L.stride, L.w, xa, xb);
                overlap_window(gb.y, gb.w, a0.y, a0.w, need / fminf(a0.z - a0.x, gb.z - gb.x), (float)L.stride, L.h, ya, yb);
            }
            if (by_rm) {
                plateau_window(gb.x, gb.z, a0.x, a0.z, (float)L.stride, L.w, xc, xd);
                plateau_window(gb.y, gb.w, a0.y, a0.w, (float)L.stride, L.h, yc, yd);
            }
            const bool e1 = xa > xb || ya > yb, e2 = xc > xd || yc > yd;
            wx_lo = e1 ? xc : (e2 ? xa : min(xa, xc)); wx_hi = e1 ? xd : (e2 ? xb : max(xb, xd));
            wy_lo = e1 ? yc : (e2 ? ya : min(ya, yc)); wy_hi = e1 ? yd : (e2 ? yb : max(yb, yd));
            if (e1 && e2) {
                wx_lo = 0;
                wx_hi = -1;
            }
        }
    }
    // Nominated anchors (IoU >= tau or == row maximum) are only buffered during the sweep; their verdicts -- one loop
    // over all gt boxes of the image each -- are evaluated 32 at a time with every lane busy.
    int nh = 0;
    auto flush = [&]() {
        __syncwarp();
        for (int h0 = 0; h0 < nh; h0 += 32) {
            const bool has = h0 + lane < nh;
            bool emit = false;
            int packed = 0, mgt = 0;
            if (has) {
                const int row = s_hits[wid][h0 + lane];
                const Verdict vd = anchor_verdict(anchors[row], gt, rowmax, g0, G, tau, lq);
                const int lb = verdict_label(rule, vd, G);
                if (vd.first_q == tl && lb != 0 && lb != -1) {  // an anchor several boxes nominate: the first one emits
                    emit = true;
                    packed = row | ((int)(uint8_t)lb << 24);
                    mgt = vd.argmax;
                }
            }
            const unsigned em = __ballot_sync(FULLMASK, emit);
            if (em) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&stats[img * 4 + 0], __popc(em));
                base = __shfl_sync(FULLMASK, base, 0) + __popc(em & ((1u << lane) - 1u));
                if (emit && base < list_cap) {
                    pos_list[(int64_t)img * list_cap + base] = packed;
                    pos_gt[(int64_t)img * list_cap + base] = mgt;
                }
            }
        }
        __syncwarp();
        nh = 0;
    };
    const int lx = lane & 7, ly = lane >> 3;
    for (int p = 0; p < P; ++p) {
        const int x_lo = __shfl_sync(FULLMASK, wx_lo, p), x_hi = __shfl_sync(FULLMASK, wx_hi, p);
        const int y_lo = __shfl_sync(FULLMASK, wy_lo, p), y_hi = __shfl_sync(FULLMASK, wy_hi, p);
        if (x_lo > x_hi || y_lo > y_hi) continue;  // warp-uniform
        const GridLevelDev L = lay.lv[p / A];
        const int a = p % A;
        const int row_a = (int)L.first_row + a;
        const float4* __restrict__ lvl = anchors + row_a;
        for (int yy = y_lo; yy <= y_hi; yy += 4) {
            for (int xx = x_lo; xx <= x_hi; xx += 8) {
                const int y = yy + ly, x = xx + lx;
                bool hit = false;
                int row = 0;
                if (y <= y_hi && x <= x_hi) {
                    row = (y * L.w + x) * A;
                    const float4 ab = lvl[row];
                    const float v = pair_iou(gb, ga, ab, box_area(ab));
                    hit = v >= tau || (lq && v == rm);
                }
                const unsigned bal = __ballot_sync(FULLMASK, hit);
                if (bal) {
                    if (nh + __popc(bal) > kHitCap) flush();
                    if (hit) s_hits[wid][nh + __popc(bal & ((1u << lane) - 1u))] = row_a + row;
                    nh += __popc(bal);
                }
            }
        }
    }
    flush();
}

// ---- K2: labels + matched index of every anchor, one pass -------------------------------------------------------------
struct TileBox {
    float x1, y1, x2, y2;
};
__device__ __forceinline__ bool tile_culls(const TileBox& bb, const float4 g) {
    // true iff the gt box certainly has zero intersection with every anchor of the tile (NaN: never culled)
    return g.z <= bb.x1 || g.x >= bb.x2 || g.w <= bb.y1 || g.y >= bb.y2;
}

// one gt box against the A anchors of this lane.  Lanes without a position hold all-zero anchors: their IoUs are 0, which
// never beats the initial best and is never stored.  hits: bit a set iff some IoU of anchor a equalled its gt's row maximum.
template <int A>
__device__ __forceinline__ void match_one(const float4 gb, float rm, int t, const float4 (&ab)[A], const float (&aa)[A],
                                          float (&best)[A], int (&bidx)[A], unsigned& hits) {
    const float ga = box_area(gb);
#pragma unroll
    for (int a = 0; a < A; ++a) {
        // pairwise_iou(gt, anchors): boxes1 = gt, boxes2 = anchors (rpn.py:167).  (The quotient stays behind the
        // `inter > 0` branch: evaluated unconditionally, 0 / x takes the division's slow path -- measured 25 % slower.)
        const float v = pair_iou(gb, ga, ab[a], aa[a]);
        if (v > best[a]) {
            best[a] = v;
            bidx[a] = t;
        }
        hits |= (v == rm) ? (1u << a) : 0u;  // matcher.py:110-120; skipped pairs have v = 0 and could only match rm = 0
    }
}

template <int A, bool DENSE>
__global__ void __launch_bounds__(kGridWarps * 32, A <= 3 ? 3 : 2)
match_grid_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, const float4* __restrict__ anchors,
                  int n, int imgs, int64_t r, GridLayoutDev lay, MatchRule rule, const float* __restrict__ rowmax,
                  const int32_t* __restrict__ flags, const uint32_t* __restrict__ mask, int64_t* __restrict__ matched,
                  int8_t* __restrict__ labels, float* __restrict__ matched_iou, int32_t* __restrict__ stats,
                  int32_t* __restrict__ pos_list, int list_cap) {
    const unsigned FULLMASK = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int T = blockIdx.x * kGridWarps + (threadIdx.x >> 5);
    if (T >= lay.tiles_total) return;  // warp-uniform
    int l = 0;
#pragma unroll
    for (int k = 1; k < kGridMaxLevels; ++k)
        if (k < lay.nlev && T >= lay.lv[k].first_tile) l = k;
    const GridLevelDev L = lay.lv[l];
    const int tl = T - L.first_tile;
    const int y = (tl / L.tiles_x) * kTileH + (lane >> 3), x = (tl % L.tiles_x) * kTileW + (lane & 7);
    const bool valid = y < L.h && x < L.w;
    const int64_t row0 = L.first_row + ((int64_t)y * L.w + x) * A;  // this lane's A anchors are consecutive rows
    float4 ab[A];
    float aa[A];
#pragma unroll
    for (int a = 0; a < A; ++a) {
        ab[a] = valid ? anchors[row0 + a] : make_float4(0.f, 0.f, 0.f, 0.f);
        aa[a] = box_area(ab[a]);
    }
    const int nvalid = __popc(__ballot_sync(FULLMASK, valid));
    // Output plan.  A lane computes the A anchors of ONE position, which in memory are A consecutive entries followed by the
    // next position's: stored from the computing lane, a warp store would touch every sector of the tile A times with a
    // third of it each (the L1/TEX pipe was the busiest unit of this kernel: 78 %).  Instead the tile's 32 * A results
    // pass through a per-warp shared-memory patch in memory order (entry e = lane * A + a: conflict-free both ways) and
    // are stored A times as 32 CONSECUTIVE entries: entry e = k * 32 + lane lives in tile row e / (8A), column e % (8A).
    __shared__ int s_idx[kGridWarps][32 * A];
    __shared__ int8_t s_lab[kGridWarps][32 * A];
    int* my_idx = s_idx[threadIdx.x >> 5];
    int8_t* my_lab = s_lab[threadIdx.x >> 5];
    int64_t eoff[A];   // element offset of entry k * 32 + lane from the image's row start (valid entries only)
    bool eok[A];
#pragma unroll
    for (int k = 0; k < A; ++k) {
        const int e = k * 32 + lane, er = e / (kTileW * A), ec = e - er * (kTileW * A);
        const int ey = (tl / L.tiles_x) * kTileH + er, ex = (tl % L.tiles_x) * kTileW + ec / A;
        eok[k] = ey < L.h && ex < L.w;
        eoff[k] = L.first_row + ((int64_t)ey * L.w + ex) * A + (ec - (ec / A) * A);
    }
    const int lab_none = rule.lab[0];  // label of an anchor that overlaps no gt box (IoU 0): bucket (-inf, thr[0])
    const float thr0 = rule.thr[0], thr1 = rule.thr[1];  // the reference's rules have one or two thresholds (thr[i >= nthr] = +inf)
    const int lab1 = rule.lab[1], lab2 = rule.lab[2];
    const int i0 = blockIdx.y * imgs, ni = min(imgs, n - i0);
    // the image's flags and this tile's gt mask are prefetched one image ahead
    int fl_next = flags[i0], g0_next = gt_off[i0];
    unsigned mk_next = mask[(int64_t)i0 * lay.tiles_total + T];
    for (int ii = 0; ii < ni; ++ii) {
        const int img = i0 + ii;
        const int fl = fl_next, g0 = g0_next;
        unsigned todo = mk_next;
        if (ii + 1 < ni) {
            fl_next = flags[img + 1];
            g0_next = gt_off[img + 1];
            mk_next = mask[(int64_t)(img + 1) * lay.tiles_total + T];
        }
        const bool promote_all = rule.allow_lq && (fl & kFlagPromoteAll);
        const int64_t o = (int64_t)img * r + row0;
        if (todo == 0u && !(fl & kFlagManyGt) && !promote_all) {
            // no gt box reaches this tile (the usual case on the fine levels; also an image without gt,
            // matcher.py:67-77): every anchor has IoU 0 with every box -- match 0, the label of the lowest bucket
            if (DENSE) {
                const int64_t ob = (int64_t)img * r;
#pragma unroll
                for (int k = 0; k < A; ++k)
                    if (eok[k]) {
                        matched[ob + eoff[k]] = 0;
                        labels[ob + eoff[k]] = (int8_t)lab_none;
                        if (matched_iou) matched_iou[ob + eoff[k]] = 0.0f;
                    }
            }
            // (a rule whose lowest bucket is positive makes positives dense: the list overflows by construction and the
            //  sampler takes its generic path, so untouched tiles only count)
            if (stats && lab_none != 0 && lane == 0) atomicAdd(&stats[img * 4 + (lab_none == -1 ? 1 : 0)], nvalid * A);
            continue;
        }
        // a touched tile: the image has gt boxes (an image without any has an empty mask and no flag)
        float best[A];
        int bidx[A];
        unsigned hits = 0u;
#pragma unroll
        for (int a = 0; a < A; ++a) {
            best[a] = 0.0f;  // IoUs are >= 0 and only a strictly larger one replaces the incumbent: gt 0 wins ties at 0,
            bidx[a] = 0;     // exactly like torch.max(dim=0)
        }
        if (!(fl & kFlagManyGt)) {
            while (todo) {  // ascending gt index: the first maximum wins
                const int t = __ffs(todo) - 1;
                todo &= todo - 1;
                const float4 gb = gt[g0 + t];  // warp-uniform address: one broadcast load
                const float rm = rule.allow_lq ? rowmax[g0 + t] : -1.0f;
                match_one<A>(gb, rm, t, ab, aa, best, bidx, hits);
            }
        } else {  // more than 32 boxes: cull against the tile's bounding box on the fly (rare: the box is rebuilt here)
            TileBox bb{INFINITY, INFINITY, -INFINITY, -INFINITY};
#pragma unroll
            for (int a = 0; a < A; ++a)
                if (valid) {  // fminf / fmaxf drop NaN coordinates: a NaN anchor intersects nothing
                    bb.x1 = fminf(bb.x1, ab[a].x); bb.y1 = fminf(bb.y1, ab[a].y);
                    bb.x2 = fmaxf(bb.x2, ab[a].z); bb.y2 = fmaxf(bb.y2, ab[a].w);
                }
#pragma unroll
            for (int o2 = 16; o2 > 0; o2 >>= 1) {
                bb.x1 = fminf(bb.x1, __shfl_xor_sync(FULLMASK, bb.x1, o2)); bb.y1 = fminf(bb.y1, __shfl_xor_sync(FULLMASK, bb.y1, o2));
                bb.x2 = fmaxf(bb.x2, __shfl_xor_sync(FULLMASK, bb.x2, o2)); bb.y2 = fmaxf(bb.y2, __shfl_xor_sync(FULLMASK, bb.y2, o2));
            }
            const int G = gt_off[img + 1] - g0;
            for (int t0 = 0; t0 < G; t0 += 32) {
                float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
                float rm_mine = -1.0f;
                bool over = false;
                if (t0 + lane < G) {
                    mine = gt[g0 + t0 + lane];
                    over = !tile_culls(bb, mine);
                    if (rule.allow_lq) rm_mine = rowmax[g0 + t0 + lane];
                }
                unsigned td = __ballot_sync(FULLMASK, over);
                while (td) {
                    const int src = __ffs(td) - 1;
                    td &= td - 1;
                    const float4 gb = make_float4(__shfl_sync(FULLMASK, mine.x, src), __shfl_sync(FULLMASK, mine.y, src),
                                                  __shfl_sync(FULLMASK, mine.z, src), __shfl_sync(FULLMASK, mine.w, src));
                    match_one<A>(gb, __shfl_sync(FULLMASK, rm_mine, src), t0 + src, ab, aa, best, bidx, hits);
                }
            }
        }
        if (promote_all) hits = 0xffffffffu;
        if (!rule.allow_lq) hits = 0u;
        int lab[A];
        int my_pos = 0, my_ign = 0;
#pragma unroll
        for (int a = 0; a < A; ++a) {
            int lb;
            if (rule.nthr <= 2) {
                lb = lab_none;
                if (best[a] >= thr0) lb = lab1;
                if (best[a] >= thr1) lb = lab2;
            } else {
                lb = bucket_label(rule, best[a]);
            }
            if ((hits >> a) & 1u) lb = 1;
            lab[a] = lb;
            my_pos += valid && lb != 0 && lb != -1;
            my_ign += valid && lb == -1;
        }
        const int tot_pos = stats ? __reduce_add_sync(FULLMASK, my_pos) : 0;
        const int tot_ign = stats ? __reduce_add_sync(FULLMASK, my_ign) : 0;
        if (DENSE) {
            __syncwarp();  // the previous image's reads of the patch are done
#pragma unroll
            for (int a = 0; a < A; ++a) {
                my_idx[lane * A + a] = bidx[a];
                my_lab[lane * A + a] = (int8_t)lab[a];
            }
            __syncwarp();
            const int64_t ob = (int64_t)img * r;
#pragma unroll
            for (int k = 0; k < A; ++k)
                if (eok[k]) {
                    matched[ob + eoff[k]] = my_idx[k * 32 + lane];
                    labels[ob + eoff[k]] = my_lab[k * 32 + lane];
                }
            if (matched_iou && valid) {  // (optional output, off the hot path: stored from the computing lane)
#pragma unroll
                for (int a = 0; a < A; ++a) matched_iou[o + a] = best[a];
            }
        }
        if (stats) {
            // warp-aggregated: one atomic per warp and image for each counter that is non-zero (both are rare)
            if (tot_pos) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&stats[img * 4 + 0], tot_pos);
                if (pos_list) {
                    // list slot: positives of lower lanes first, then this lane's in anchor order
                    int before = 0;
#pragma unroll
                    for (int a = 0; a < A; ++a) {
                        const bool is_pos = valid && lab[a] != 0 && lab[a] != -1;
                        before += __popc(__ballot_sync(FULLMASK, is_pos) & ((1u << lane) - 1u));
                    }
                    base = __shfl_sync(FULLMASK, base, 0) + before;
#pragma unroll
                    for (int a = 0; a < A; ++a)
                        if (valid && lab[a] != 0 && lab[a] != -1) {
                            if (base < list_cap)
                                pos_list[(int64_t)img * list_cap + base] = (int)(row0 + a) | ((int)(uint8_t)lab[a] << 24);
                            ++base;
                        }
                }
            }
            if (lane == 0 && tot_ign) atomicAdd(&stats[img * 4 + 1], tot_ign);
        }
    }
}

// ---- sampled loss: BCE-with-logits on the sampled anchors + smooth-L1 / GIoU on the sampled positives, forward and
//      backward, O(samples) traffic.  One CTA per image walks the image's sample list (<= num_samples entries written by
//      the sampler: anchor row | label << 24).  The head is read where the convolutions left it: either flat (N,R) /
//      (N,R,4) tensors or per-level NCHW planes (objectness (N,A,H,W), deltas (N,A*4,H,W)), gradients go to the same
//      layout.  Gradient buffers are NOT swept: the caller zeroes them once (cudaMemset) or keeps them persistent and
//      passes the previous step's sample list, whose entries are reset to zero first (`clear_*`).
//      The last CTA scales the sums, writes the 8-float result and re-arms the accumulators: no memset, no epilogue op.
struct HeadLevelDev {
    const float* obj;
    const float* dlt;
    float* g_obj;
    float* g_dlt;
    int h, w;
    int64_t first_row;
};
struct HeadLayoutDev {
    HeadLevelDev lv[kGridMaxLevels];
    int nlev;  // 0: flat layout, lv[0] holds the (N,R) / (N,R,4) pointers
    int a;
};

struct HeadAddr {
    int64_t obj;        // element offset of the logit
    int64_t dlt;        // element offset of delta component 0
    int64_t dlt_step;   // element stride between the 4 delta components
    int lvl;
};

__device__ __forceinline__ HeadAddr head_addr(const HeadLayoutDev& hl, int img, int64_t r, int64_t j) {
    HeadAddr ad;
    if (hl.nlev == 0) {
        ad.lvl = 0;
        ad.obj = (int64_t)img * r + j;
        ad.dlt = ad.obj * 4;
        ad.dlt_step = 1;
        return ad;
    }
    int l = 0;
#pragma unroll
    for (int k = 1; k < kGridMaxLevels; ++k)
        if (k < hl.nlev && j >= hl.lv[k].first_row) l = k;
    const HeadLevelDev& L = hl.lv[l];
    const int64_t local = j - L.first_row;
    const int a = (int)(local % hl.a);
    const int64_t pos = local / hl.a, hw = (int64_t)L.h * L.w;
    ad.lvl = l;
    ad.obj = ((int64_t)img * hl.a + a) * hw + pos;              // (N, A, H, W)
    ad.dlt = ((int64_t)img * hl.a * 4 + a * 4) * hw + pos;      // (N, A*4, H, W): channel = a*4 + component
    ad.dlt_step = hw;
    return ad;
}

constexpr int kSampledThreads = 256;  // one thread per sample (batch_size_per_image = 256): every gather is in flight at once

template <bool GIOU>
__global__ void __launch_bounds__(kSampledThreads)
rpn_loss_sampled_kernel(HeadLayoutDev hl, const int32_t* __restrict__ samples, const int32_t* __restrict__ sample_count,
                        int sample_cap, const int32_t* __restrict__ clear_samples,
                        const int32_t* __restrict__ clear_count, const int64_t* __restrict__ matched,
                        const int32_t* __restrict__ sample_gt, const float4* __restrict__ gt, const int32_t* __restrict__ gt_off,
                        const float4* __restrict__ anchors, int64_t r, CodecWeights wt, float scale_clamp, float beta,
                        float scale_cls, float scale_loc, const float* __restrict__ upstream, float* __restrict__ acc,
                        int32_t* __restrict__ ticket, float* __restrict__ sums_out, int write_grads) {
    __shared__ float s_part[4][kSampledThreads / 32];
    __shared__ float s_fin[8];
    const int img = blockIdx.x;
    float gs_cls = scale_cls, gs_loc = scale_loc;
    if (upstream) {
        gs_cls *= upstream[0];
        gs_loc *= upstream[1];
    }
    if (write_grads && clear_samples) {  // persistent gradient buffers: undo the previous step's writes of this image
        const int nc = min(clear_count[img], sample_cap);
        for (int k = threadIdx.x; k < nc; k += kSampledThreads) {
            const int packed = clear_samples[(int64_t)img * sample_cap + k];
            const HeadAddr ad = head_addr(hl, img, r, packed & 0xffffff);
            const HeadLevelDev& L = hl.lv[ad.lvl];
            L.g_obj[ad.obj] = 0.0f;
            if ((int8_t)(packed >> 24) == 1) {
                if (ad.dlt_step == 1) {
                    *reinterpret_cast<float4*>(L.g_dlt + ad.dlt) = make_float4(0.f, 0.f, 0.f, 0.f);
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c) L.g_dlt[ad.dlt + c * ad.dlt_step] = 0.0f;
                }
            }
        }
        __syncthreads();  // the same anchor may be sampled again: zero first, then write
    }
    float acc_cls = 0.f, acc_loc = 0.f;
    int npos = 0, nneg = 0;
    const int ns = min(sample_count[img], sample_cap);
    for (int k = threadIdx.x; k < ns; k += kSampledThreads) {
        const int packed = samples[(int64_t)img * sample_cap + k];
        const int64_t j = packed & 0xffffff;
        const int lab = (int)(int8_t)(packed >> 24);
        const HeadAddr ad = head_addr(hl, img, r, j);
        const HeadLevelDev& L = hl.lv[ad.lvl];
        const float x = L.obj[ad.obj];
        const float yv = (float)lab;
        // BCE with logits: (1-y)*x - log_sigmoid(x), log_sigmoid(x) = min(x,0) - log1p(exp(-|x|))  (rpn.py:233)
        const float ls = fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
        acc_cls += (1.f - yv) * x - ls;
        npos += lab == 1;
        nneg += lab == 0;
        if (write_grads) L.g_obj[ad.obj] = (1.f / (1.f + expf(-x)) - yv) * gs_cls;
        if (lab == 1) {
            const int64_t mg = sample_gt ? (int64_t)sample_gt[(int64_t)img * sample_cap + k] : matched[(int64_t)img * r + j];
            const float4 g = gt[gt_off[img] + mg];
            float4 p;
            if (ad.dlt_step == 1) {
                p = *reinterpret_cast<const float4*>(L.dlt + ad.dlt);
            } else {
                p = make_float4(L.dlt[ad.dlt], L.dlt[ad.dlt + ad.dlt_step], L.dlt[ad.dlt + 2 * ad.dlt_step],
                                L.dlt[ad.dlt + 3 * ad.dlt_step]);
            }
            float4 gd;
            if (GIOU) {
                float4 dd;
                acc_loc += giou_fwd_bwd(p, anchors[j], g, wt, scale_clamp, dd);
                gd = make_float4(dd.x * gs_loc, dd.y * gs_loc, dd.z * gs_loc, dd.w * gs_loc);
            } else {
                const float4 tgt = encode_delta(anchors[j], g, wt);
                float v, d;
                smooth_l1(p.x, tgt.x, beta, v, d); acc_loc += v; gd.x = d * gs_loc;
                smooth_l1(p.y, tgt.y, beta, v, d); acc_loc += v; gd.y = d * gs_loc;
                smooth_l1(p.z, tgt.z, beta, v, d); acc_loc += v; gd.z = d * gs_loc;
                smooth_l1(p.w, tgt.w, beta, v, d); acc_loc += v; gd.w = d * gs_loc;
            }
            if (write_grads) {
                if (ad.dlt_step == 1) {
                    *reinterpret_cast<float4*>(L.g_dlt + ad.dlt) = gd;
                } else {
                    L.g_dlt[ad.dlt] = gd.x;
                    L.g_dlt[ad.dlt + ad.dlt_step] = gd.y;
                    L.g_dlt[ad.dlt + 2 * ad.dlt_step] = gd.z;
                    L.g_dlt[ad.dlt + 3 * ad.dlt_step] = gd.w;
                }
            }
        }
    }
    acc_cls = warp_sum(acc_cls);
    acc_loc = warp_sum(acc_loc);
    const float fpos = warp_sum((float)npos), fneg = warp_sum((float)nneg);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
        s_part[0][wid] = acc_cls;
        s_part[1][wid] = acc_loc;
        s_part[2][wid] = fpos;
        s_part[3][wid] = fneg;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        float t = 0.f;
        for (int w = 0; w < kSampledThreads / 32; ++w) t += s_part[threadIdx.x][w];
        if (t != 0.f) atomicAdd(&acc[threadIdx.x], t);
    }
    // last CTA: sums_out = [cls * scale_cls, loc * scale_loc, #pos, #neg, 0...], accumulators and ticket re-armed
    if (last_cta_arrives(ticket))
        finalize_sums(acc, sums_out, s_fin, [&](int i) { return i == 0 ? scale_cls : (i == 1 ? scale_loc : 1.0f); });
}

static int fill_layout(GridLayoutDev& lay, const det_anchor_level_t* levels_host, int num_levels, int a, int64_t r) {
    if (!levels_host || num_levels < 1 || num_levels > kGridMaxLevels || a < 1 || num_levels * a > 32) {
        set_error("grid layout: 1..%d levels, levels x anchors-per-position <= 32", kGridMaxLevels);
        return DET_ERR_UNSUPPORTED;
    }
    lay.nlev = num_levels;
    lay.a = a;
    int tiles = 0;
    int64_t row = 0;
    for (int l = 0; l < num_levels; ++l) {
        const det_anchor_level_t& s = levels_host[l];
        if (s.h < 1 || s.w < 1 || s.stride < 1 || s.first_row != row) {
            set_error("grid layout: level %d must have h, w, stride >= 1 and start at row %lld", l, (long long)row);
            return DET_ERR_BAD_ARG;
        }
        GridLevelDev& d = lay.lv[l];
        d.h = s.h; d.w = s.w; d.stride = s.stride;
        d.tiles_x = (s.w + kTileW - 1) / kTileW;
        d.first_tile = tiles;
        d.first_row = row;
        tiles += d.tiles_x * ((s.h + kTileH - 1) / kTileH);
        row += (int64_t)s.h * s.w * a;
    }
    if (row != r) {
        set_error("grid layout: levels cover %lld anchors, r = %lld", (long long)row, (long long)r);
        return DET_ERR_BAD_ARG;
    }
    lay.tiles_total = tiles;
    return DET_OK;
}

}  // namespace det

using namespace det;

// assign_loss.cu (the samplers live next to subsample_image)
int launch_subsample_lazy(const float* gt_boxes, const int32_t* gt_offsets, const float* anchors, int n, int64_t r,
                          const MatchRule& rule, float tau, const float* rowmax, const int32_t* flags, const int32_t* stats,
                          const int32_t* pos_list, const int32_t* pos_gt, int list_cap, int num_samples,
                          double positive_fraction, uint64_t seed, int8_t* scratch, int32_t* samples, int32_t* sample_gt,
                          int32_t* sample_count, int sample_cap, cudaStream_t st);

extern "C" {

static int64_t align256(int64_t v) { return (v + 255) / 256 * 256; }

// workspace: row maxima (sum_g fp32) | per-image flags (n int32) | tile masks (n x tiles uint32)
int64_t det_match_grid_workspace_bytes(int n, int64_t sum_g, const det_anchor_level_t* levels_host, int num_levels) {
    int64_t tiles = 0;
    for (int l = 0; levels_host && l < num_levels; ++l)
        tiles += (int64_t)((levels_host[l].w + kTileW - 1) / kTileW) * ((levels_host[l].h + kTileH - 1) / kTileH);
    if (tiles < 1) tiles = 1;
    return align256((sum_g > 0 ? sum_g : 1) * 4) + align256((int64_t)(n > 0 ? n : 1) * 4) +
           align256((int64_t)(n > 0 ? n : 1) * tiles * 4);
}

int det_match_grid(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors, int64_t r,
                   const det_anchor_level_t* levels_host, int num_levels, int a, const float* thresholds_host,
                   const int32_t* labels_host, int num_thresholds, int allow_low_quality, int64_t* matched_idx,
                   int8_t* labels, float* matched_iou, int32_t* stats, int32_t* pos_list, int list_cap, void* workspace,
                   int64_t workspace_bytes, void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && sum_g >= 0, "negative size");
    if (n == 0 || r == 0) return DET_OK;
    DET_CHECK_ARG(gt_offsets && anchors && matched_idx && labels, "null pointer");
    DET_CHECK_ARG(sum_g == 0 || gt_boxes, "null gt_boxes");
    DET_CHECK_ARG(n <= 65535, "n > 65535");
    DET_CHECK_ARG(r < (1ll << 27) && sum_g < (1ll << 31), "r must be below 2^27");
    DET_CHECK_ARG(!pos_list || (stats && list_cap >= 1 && r < (1 << 24)), "pos_list needs stats, list_cap >= 1, r < 2^24");
    if (!aligned16(anchors) || (gt_boxes && !aligned16(gt_boxes))) {
        set_error("gt_boxes/anchors must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    MatchRule rule;
    int rc = fill_rule(rule, thresholds_host, labels_host, num_thresholds, allow_low_quality);
    if (rc != DET_OK) return rc;
    GridLayoutDev lay;
    rc = fill_layout(lay, levels_host, num_levels, a, r);
    if (rc != DET_OK) return rc;
    if (a != 1 && a != 3 && a != 9) {
        set_error("det_match_grid: anchors per position must be 1, 3 or 9 (use det_match_anchors otherwise)");
        return DET_ERR_UNSUPPORTED;
    }
    const int64_t off_flags = align256((sum_g > 0 ? sum_g : 1) * 4);
    const int64_t off_mask = off_flags + align256((int64_t)n * 4);
    const int64_t need = off_mask + align256((int64_t)n * lay.tiles_total * 4);
    if (!workspace || workspace_bytes < need) {
        set_error("workspace too small: need %lld bytes", (long long)need);
        return DET_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    char* ws = static_cast<char*>(workspace);
    float* rowmax = reinterpret_cast<float*>(ws);
    int32_t* flags = reinterpret_cast<int32_t*>(ws + off_flags);
    uint32_t* mask = reinterpret_cast<uint32_t*>(ws + off_mask);
    cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)(need - off_flags), st);  // flags + masks in one sweep
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto a4 = reinterpret_cast<const float4*>(anchors);
    const int stats_words = stats ? n * 4 : 0;
    const int64_t k1_threads = sum_g * 32 > stats_words ? sum_g * 32 : stats_words;
    if (k1_threads > 0) {
        match_rowmax_kernel<<<(unsigned)((k1_threads + 127) / 128), 128, 0, st>>>(
            g4, gt_offsets, n, sum_g, a4, lay, allow_low_quality ? 1 : 0, rowmax, flags, mask, stats, stats_words);
        DET_LAUNCH_OK("match_rowmax_kernel");
    }
    // images per CTA: amortise the anchor loads and the tile box while keeping >= 8 CTAs per SM in flight
    const int bx = (lay.tiles_total + kGridWarps - 1) / kGridWarps;
    int imgs = (int)(((int64_t)bx * n) / ((int64_t)sm_count() * 8));
    imgs = imgs < 1 ? 1 : (imgs > 8 ? 8 : imgs);
    dim3 grid((unsigned)bx, (unsigned)((n + imgs - 1) / imgs));
#define DET_LAUNCH_GRID(AA)                                                                                              \
    match_grid_kernel<AA, true><<<grid, kGridWarps * 32, 0, st>>>(g4, gt_offsets, a4, n, imgs, r, lay, rule, rowmax,      \
                                                                  flags, mask, matched_idx, labels, matched_iou, stats,  \
                                                                  pos_list, list_cap)
    if (a == 1) DET_LAUNCH_GRID(1);
    else if (a == 3) DET_LAUNCH_GRID(3);
    else DET_LAUNCH_GRID(9);
#undef DET_LAUNCH_GRID
    DET_LAUNCH_OK("match_grid_kernel");
    return DET_OK;
}

int64_t det_assign_sampled_workspace_bytes(int n, int64_t sum_g, int list_cap) {
    const int64_t nn = n > 0 ? n : 1, cap = list_cap > 0 ? list_cap : 1;
    return align256((sum_g > 0 ? sum_g : 1) * 4) + align256(nn * 4) + align256(nn * 16) + 2 * align256(nn * cap * 4);
}

int det_assign_sampled(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors,
                       int64_t r, const det_anchor_level_t* levels_host, int num_levels, int a,
                       const float* thresholds_host, const int32_t* labels_host, int num_thresholds, int allow_low_quality,
                       int num_samples, double positive_fraction, uint64_t seed, int8_t* scratch_labels, int32_t* samples,
                       int32_t* sample_gt, int32_t* sample_count, int sample_cap, void* workspace, int64_t workspace_bytes,
                       void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && sum_g >= 0 && num_samples >= 0 && sample_cap >= 1, "bad size");
    DET_CHECK_ARG(positive_fraction >= 0.0 && positive_fraction <= 1.0, "positive_fraction outside [0, 1]");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(gt_offsets && anchors && scratch_labels && samples && sample_gt && sample_count, "null pointer");
    DET_CHECK_ARG(sum_g == 0 || gt_boxes, "null gt_boxes");
    DET_CHECK_ARG(r >= 1 && r < (1 << 24) && sum_g < (1ll << 31) && n <= 65535, "1 <= r < 2^24, n <= 65535");
    if (!aligned16(anchors) || (gt_boxes && !aligned16(gt_boxes))) {
        set_error("gt_boxes/anchors must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    MatchRule rule;
    int rc = fill_rule(rule, thresholds_host, labels_host, num_thresholds, allow_low_quality);
    if (rc != DET_OK) return rc;
    if (rule.lab[0] != 0 && rule.lab[0] != -1) {
        set_error("det_assign_sampled: the lowest bucket must not be positive (labels[0] in {0, -1})");
        return DET_ERR_UNSUPPORTED;
    }
    // the lowest IoU that can make an anchor positive through the threshold rule
    float tau = INFINITY;
    for (int i = num_thresholds; i >= 1; --i)
        if (rule.lab[i] != 0 && rule.lab[i] != -1) tau = rule.thr[i - 1];
    GridLayoutDev lay;
    rc = fill_layout(lay, levels_host, num_levels, a, r);
    if (rc != DET_OK) return rc;
    const int list_cap = 1024;
    const int64_t off_flags = align256((sum_g > 0 ? sum_g : 1) * 4);
    const int64_t off_stats = off_flags + align256((int64_t)n * 4);
    const int64_t off_list = off_stats + align256((int64_t)n * 16);
    const int64_t off_gt = off_list + align256((int64_t)n * list_cap * 4);
    const int64_t need = off_gt + align256((int64_t)n * list_cap * 4);
    if (!workspace || workspace_bytes < need) {
        set_error("workspace too small: need %lld bytes", (long long)need);
        return DET_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    char* ws = static_cast<char*>(workspace);
    float* rowmax = reinterpret_cast<float*>(ws);
    int32_t* flags = reinterpret_cast<int32_t*>(ws + off_flags);
    int32_t* stats = reinterpret_cast<int32_t*>(ws + off_stats);
    int32_t* pos_list = reinterpret_cast<int32_t*>(ws + off_list);
    int32_t* pos_gt = reinterpret_cast<int32_t*>(ws + off_gt);
    cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)(off_list - off_flags), st);  // flags + stats
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto a4 = reinterpret_cast<const float4*>(anchors);
    if (sum_g > 0) {
        const unsigned blocks = (unsigned)((sum_g + kCandWarps - 1) / kCandWarps);
        if (allow_low_quality) {
            match_rowmax_kernel<<<blocks, 128, 0, st>>>(g4, gt_offsets, n, sum_g, a4, lay, 1, rowmax, flags, nullptr, nullptr, 0);
            DET_LAUNCH_OK("match_rowmax_kernel");
        }
        assign_candidates_kernel<<<blocks, kCandWarps * 32, 0, st>>>(g4, gt_offsets, n, sum_g, a4, lay, rule, tau, rowmax, flags, stats,
                                                         pos_list, pos_gt, list_cap);
        DET_LAUNCH_OK("assign_candidates_kernel");
    }
    return launch_subsample_lazy(gt_boxes, gt_offsets, anchors, n, r, rule, tau, rowmax, flags, stats, pos_list, pos_gt,
                                 list_cap, num_samples, positive_fraction, seed, scratch_labels, samples, sample_gt,
                                 sample_count, sample_cap, st);
}

int det_rpn_loss_sampled(const det_head_level_t* levels_host, int num_levels, int a, const float* logits_flat,
                         const float* deltas_flat, float* grad_logits_flat, float* grad_deltas_flat,
                         const int32_t* samples, const int32_t* sample_count, int sample_cap,
                         const int32_t* clear_samples, const int32_t* clear_count, const int64_t* matched_idx,
                         const int32_t* sample_gt, const float* gt_boxes, const int32_t* gt_offsets, const float* anchors,
                         int n, int64_t r, float wx,
                         float wy, float ww, float wh, float scale_clamp, int loss_type, float smooth_l1_beta,
                         float scale_cls, float scale_loc, const float* upstream, float* accumulators, float* sums_out,
                         void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && sample_cap >= 1, "bad size");
    DET_CHECK_ARG(loss_type == 0 || loss_type == 1, "loss_type must be 0 (smooth-L1) or 1 (GIoU)");
    DET_CHECK_ARG(sums_out && accumulators, "null output");
    if (n == 0 || r == 0) {
        cudaError_t e = cudaMemsetAsync(sums_out, 0, 8 * sizeof(float), as_stream(stream));
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
        return DET_OK;
    }
    DET_CHECK_ARG(samples && sample_count && (matched_idx || sample_gt) && gt_offsets && anchors, "null pointer");
    DET_CHECK_ARG(r < (1 << 24), "r must be below 2^24 (sample entries pack the anchor row in 24 bits)");
    DET_CHECK_ARG((clear_samples == nullptr) == (clear_count == nullptr), "clear_samples and clear_count go together");
    if (!aligned16(anchors) || (gt_boxes && !aligned16(gt_boxes))) {
        set_error("gt_boxes/anchors must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    HeadLayoutDev hl;
    int write_grads = 0;
    if (num_levels == 0) {
        DET_CHECK_ARG(logits_flat && deltas_flat, "flat layout: null logits/deltas");
        DET_CHECK_ARG((grad_logits_flat == nullptr) == (grad_deltas_flat == nullptr), "both gradients or none");
        if (!aligned16(deltas_flat) || (grad_deltas_flat && !aligned16(grad_deltas_flat))) {
            set_error("deltas / grad_deltas must be 16-byte aligned");
            return DET_ERR_ALIGN;
        }
        hl.nlev = 0;
        hl.a = 1;
        hl.lv[0] = HeadLevelDev{logits_flat, deltas_flat, grad_logits_flat, grad_deltas_flat, 1, 1, 0};
        write_grads = grad_logits_flat != nullptr;
    } else {
        DET_CHECK_ARG(levels_host && num_levels >= 1 && num_levels <= kGridMaxLevels && a >= 1, "bad head levels");
        hl.nlev = num_levels;
        hl.a = a;
        int64_t row = 0;
        int with = 0;
        for (int l = 0; l < num_levels; ++l) {
            const det_head_level_t& s = levels_host[l];
            DET_CHECK_ARG(s.objectness && s.deltas && s.h >= 1 && s.w >= 1, "head level: null pointer or empty plane");
            DET_CHECK_ARG((s.grad_objectness == nullptr) == (s.grad_deltas == nullptr), "both gradients or none");
            with += s.grad_objectness != nullptr;
            hl.lv[l] = HeadLevelDev{s.objectness, s.deltas, s.grad_objectness, s.grad_deltas, s.h, s.w, row};
            row += (int64_t)s.h * s.w * a;
        }
        DET_CHECK_ARG(row == r, "head levels do not cover r anchors");
        DET_CHECK_ARG(with == 0 || with == num_levels, "gradients for all levels or none");
        write_grads = with != 0;
    }
    const CodecWeights wt{wx, wy, ww, wh};
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto a4 = reinterpret_cast<const float4*>(anchors);
    int32_t* ticket = reinterpret_cast<int32_t*>(accumulators + 8);
    if (loss_type == 1)
        rpn_loss_sampled_kernel<true><<<n, kSampledThreads, 0, as_stream(stream)>>>(
            hl, samples, sample_count, sample_cap, clear_samples, clear_count, matched_idx, sample_gt, g4, gt_offsets, a4, r, wt,
            scale_clamp, smooth_l1_beta, scale_cls, scale_loc, upstream, accumulators, ticket, sums_out, write_grads);
    else
        rpn_loss_sampled_kernel<false><<<n, kSampledThreads, 0, as_stream(stream)>>>(
            hl, samples, sample_count, sample_cap, clear_samples, clear_count, matched_idx, sample_gt, g4, gt_offsets, a4, r, wt,
            scale_clamp, smooth_l1_beta, scale_cls, scale_loc, upstream, accumulators, ticket, sums_out, write_grads);
    DET_LAUNCH_OK("rpn_loss_sampled_kernel");
    return DET_OK;
}

}  // extern "C"
