// Fast path of the fused YOLO-grid decode + per-class NMS (det_yolo_decode_nms) for small grids:
// at most 128 predictors (s*s*b) and 32 classes, boxes clipped to the image -- BASELINE configs[0]/[1].
//
// One CTA per image, ONE WARP PER CLASS.  A class has at most 128 candidates (one per predictor), so every
// per-class step fits a warp and needs no block barrier:
//   A  stage the image's logits (16-byte loads; 8-byte loads of a bf16 / fp16 head, widened to fp32 on load), sigmoid the conf / class logits in place, decode the boxes
//   B  scores conf x class for the warp's class, threshold, class count, score histogram; one thread per predictor
//      gathers the coordinate statistics torchvision's offset trick needs
//   T  tier cut: only the first max_det kept detections (global score order) are output and a box can only be
//      suppressed by higher-scored ones, so the NMS first runs on the candidates above a histogram cut holding about
//      4/3 max_det of them; if that yields max_det kept boxes the rest cannot matter, else everything is redone
//   E  pair filter, once per image: every unordered pair of PREDICTORS is tested once, by all warps, with a conservative
//      bound that holds in every class's shifted frame (see pair_may_suppress); a pass sets a bit of the symmetric
//      predictor matrix `edge`.  Every class uses the same boxes, and nearly all pairs are far below the threshold.
//   R  per class, on `edge`: a tier candidate with no edge to another candidate of its class is kept; the others are
//      resolved greedily in (score descending, predictor ascending) order, each in-class edge decided by the exact
//      nms_suppresses on the class's (shifted) boxes -- the same decision as a sweep over all pairs of the class
//   M  the kept detections of all classes are put in output order by a counting sort on a 256-bin score histogram
//      (suffix scan -> bin-grouped placement -> rank inside the bin by direct comparison): no second sort
// Images whose offset-trick branch cannot be swept per class (non-finite or <= -1 coordinates: only possible with
// NaN/Inf logits here) take a slow exact path: repeated arg-max + suppression over all candidates.
//
// The kernel is specialised at compile time for the BASELINE shape (S=7, B=2, C=20) -- all index arithmetic folds to
// constants -- and has a generic instantiation (CS = CB = CC = 0) that reads the shape from the parameters.
//
// Specification: oracle/ref_torch.py yolo_decode / yolo_select_nms (SURVEY.md section 8 row a15: no reference
// implementation exists); the NMS semantics are the reference's batched_nms (python/src/utils.py:96-119).
#pragma once
#include "nms_core.cuh"

namespace det {

constexpr int kFastMaxP = 128;
constexpr int kFastMaxC = 32;
constexpr int kFastMinWarps = 8;
constexpr int kFastBins = 256;

struct YoloParams {
    int n, s, b, c;
    float stride_x, stride_y, img_w, img_h, scale_clamp, score_thresh, thr_f;
    int clip, mode;
    int64_t max_det;
    int flat32;  // det_flat points to int32 (serving wire format: 4 bytes less per detection over PCIe) instead of int64
};

// dynamic shared memory: staged head float[hs_floats] | boxes float4[pp] | merge: two u64 key buffers + one state byte
// per (predictor, class)
struct FastLayout {
    int hs_floats, pp, pcp;
    size_t bytes;
    __host__ __device__ constexpr FastLayout(int s2, int ch, int p, int c)
        : hs_floats((s2 * ch + 3) & ~3),
          pp((p + 3) & ~3),
          pcp((p * c + 3) & ~3),
          bytes((size_t)((s2 * ch + 3) & ~3) * 4 + (size_t)((p + 3) & ~3) * 16 +
                ((((size_t)((p * c + 3) & ~3) * 17 + 16) + 15) & ~(size_t)15)) {}
};

// histogram bin of a score: bits in [base, 0x3F800000], `shift` chosen so that the range spans <= 256 bins
__device__ __forceinline__ int score_bin(unsigned bits, unsigned base, int shift) {
    return min(kFastBins - 1, (int)((bits - base) >> shift));
}
__device__ __forceinline__ int score_shift(unsigned base) {
    return 0x3F800000u > base ? max(0, 32 - __clz(0x3F800000u - base) - 8) : 0;
}

// Pair filter: may box a suppress box b (or b suppress a) in SOME class frame?  Must be true whenever
// nms_suppresses(a + off, area, b + off, area, thr_f) is, for every shift off = fl(c * span) the image uses (off = 0
// in the per-category branch); the exact test then decides the pairs it lets through.
//   Inputs: thr_f >= 2^-60; r = max(1, largest |coordinate| of the image's candidate boxes) + the largest shift, r < 2^60
//   (the caller makes every pair an edge otherwise: a non-finite candidate coordinate makes r non-finite); dl = r * 2^-20;
//   al = lower_area(a, dl).  Only pairs of candidate boxes matter.  Let R be r before rounding and u = 2^-24.
//   1. Every shifted coordinate fl(v + off) is within u R of v + off, and |v + off| <= R.  A difference of two of them
//      (the same axis) is within 2uR of the unshifted real difference, and rounding it adds at most u * 2R(1+u): the
//      class frame's w' = fl(min(z') - max(x')) (min/max commute with the monotone shift) and a box's own side are
//      within 4.0001 uR of the real unshifted value.
//   2. dl >= 15.99 uR.  fl(min(z) - max(x)) is within 2uR of the real value, so wu = fl(fl(min(z) - max(x)) + dl) >= w'
//      (the margin left, > 7 uR, covers the rounding of the sum), and max(0, wu) >= max(0, w').  Likewise
//      max(0, fl(fl(x2 - x1) - dl)) <= the class frame's side of a box whenever that side is >= 0.
//   3. The exact test suppresses only if inter' > 0 (threshold >= 0), i.e. w', h' > 0: both boxes then have positive
//      sides in the class frame and inter' <= area_a', area_b', so denom' >= inter' > 0 (no overflow: r < 2^60).
//      Rounding is monotone and every operand below is >= 0, so iu = fl(wu * hu) >= inter', al <= area_a',
//      bl <= area_b', and den = fl(fl(al + bl) - iu) <= denom'.
//   4. Suppression needs fl(inter' / denom') > thr_f, so the real quotient exceeds thr_f and iu > thr_f * den.  With
//      den >= 2^-60 the product thr_lo * den is normal, and thr_lo = fl(thr_f * (1 - 2^-20)) gives fl(thr_lo * den) <
//      thr_f * den (an overflow to inf would need thr_f * den > 2^127 > iu): the test below then passes.  den < 2^-60
//      passes as well.
// The bound is symmetric in a and b, so one test covers both orders.  The margin only adds pairs: dl is about 0.01 px at
// the largest shifted coordinate of a 448 x 448, 20-class image.
__device__ __forceinline__ float lower_area(const float4 a, float dl) {
    return fmaxf(0.0f, (a.z - a.x) - dl) * fmaxf(0.0f, (a.w - a.y) - dl);
}
__device__ __forceinline__ bool pair_may_suppress(const float4 a, float al, const float4 b, float dl, float thr_lo) {
    const float wu = fmaxf(0.0f, (fminf(a.z, b.z) - fmaxf(a.x, b.x)) + dl);
    const float hu = fmaxf(0.0f, (fminf(a.w, b.w) - fmaxf(a.y, b.y)) + dl);
    const float iu = wu * hu;
    if (iu == 0.0f) return false;
    const float den = (al + lower_area(b, dl)) - iu;
    return !(den >= 0x1p-60f && iu <= thr_lo * den);
}

template <int MAXT, int MINB, int CS, int CB, int CC, typename HT = float>
__global__ void __launch_bounds__(MAXT, MINB)
yolo_fast_kernel(const HT* __restrict__ head, const float2* __restrict__ priors, YoloParams prm,
                 float4* __restrict__ dense_boxes, float* __restrict__ dense_conf, float* __restrict__ dense_scores,
                 int64_t* __restrict__ det_flat, float4* __restrict__ det_boxes, float* __restrict__ det_scores,
                 int32_t* __restrict__ det_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int S = CS ? CS : prm.s, B = CB ? CB : prm.b, C = CC ? CC : prm.c;
    const int S2 = S * S, ch = B * 5 + C, P = S2 * B, PC = P * C;
    const FastLayout lay(S2, ch, P, C);
    const int Pp = lay.pp;
    float* hs = reinterpret_cast<float*>(smem_raw);
    float4* pbox = reinterpret_cast<float4*>(hs + lay.hs_floats);
    uint64_t* buf_a = reinterpret_cast<uint64_t*>(pbox + Pp);  // merge key buffers (and the slow path's state bytes)
    uint64_t* buf_b = buf_a + lay.pcp;
    __shared__ int s_m[kFastMaxC];
    __shared__ float s_mx[4], s_mn[4];
    __shared__ int s_fl[4];
    __shared__ __align__(16) uint4 s_edge[kFastMaxP];  // symmetric pair-filter matrix: bit q of row p = pair (p, q)
    __shared__ int s_total;
    __shared__ struct {
        int cnt, gcat;
        unsigned cut[2];
    } s_img;
    __shared__ unsigned long long s_best;
    __shared__ __align__(16) int s_hist[kFastBins];   // candidates by score (tier cut)
    __shared__ __align__(16) int s_hist2[kFastBins];  // kept detections by score (output order)
    __shared__ int s_base[kFastBins];
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, T = blockDim.x;
    const int img = blockIdx.x;
    const int K = (int)min(prm.max_det, (int64_t)PC);

    pdl_trigger();  // the next launch of this stream may take SM slots as they free up (it parks in its own pdl_wait)
    for (int i = tid; i < kFastBins; i += T) {
        s_hist[i] = 0;
        s_hist2[i] = 0;
    }
    for (int i = tid; i < P; i += T) s_edge[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) s_total = 0;
    pdl_wait();     // everything earlier in the stream is complete and visible from here on
    DET_MARK(0);
    // ---- A: stage this image's logits with 16-byte coalesced loads over the aligned interior of its span; every value is
    // transformed on its way into shared memory -- sigmoid for tx, ty, conf and the class logits, exp(min(t, clamp)) for
    // tw, th -- so nothing is staged raw and the box assembly below is a handful of multiply-adds
    const int64_t g0 = (int64_t)img * S2 * ch, g1 = g0 + (int64_t)S2 * ch;
    const typename Head<HT>::vec* head4 = reinterpret_cast<const typename Head<HT>::vec*>(head);  // 4 elements per load
    auto activate = [&](int e, float x) -> float {  // e = element index inside the image (cell-major, channel-minor)
        const int cell = e / ch, k = e - cell * ch;
        if (k < B * 5) {
            const int bi = k / 5, comp = k - bi * 5;
            if (comp == 2 || comp == 3) return expf((x > prm.scale_clamp) ? prm.scale_clamp : x);  // clamp(max=): NaN stays
            const float y = sigmoidf_rn(x);
            if (comp == 4 && dense_conf) dense_conf[(int64_t)img * P + cell * B + bi] = y;
            return y;
        }
        return sigmoidf_rn(x);
    };
    for (int64_t v = (g0 >> 2) + tid; v < ((g1 + 3) >> 2); v += T) {
        const int64_t base = v << 2;
        const int e0 = (int)(base - g0);
        if (base >= g0 && base + 4 <= g1) {
            const float4 q = ld4_stream<HT>(head4 + v);
            float* d = hs + e0;
            d[0] = activate(e0, q.x); d[1] = activate(e0 + 1, q.y); d[2] = activate(e0 + 2, q.z); d[3] = activate(e0 + 3, q.w);
        } else {
            for (int e = 0; e < 4; ++e)
                if (base + e >= g0 && base + e < g1) hs[e0 + e] = activate(e0 + e, ld1_stream(head + base + e));
        }
    }
    __syncthreads();
    DET_MARK(1);

    // score histogram geometry: candidates have bits(score) in (bits(thr), bits(1.0)]; scores are >= +0
    const unsigned lo_bits = prm.score_thresh > 0.0f ? __float_as_uint(prm.score_thresh) : 0u;
    const int hshift = score_shift(lo_bits);
    // ---- B: the warp's class: scores, threshold, count, histogram
    const int c = wid;
    const bool cls_warp = c < C;
    float sc[4];
    bool pass[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        sc[k] = 0.f;
        pass[k] = false;
    }
    if (cls_warp) {
        int mcount = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = lane + 32 * k;
            if (p < P) {
                const int cell = p / B, bi = p - cell * B;
                sc[k] = hs[cell * ch + bi * 5 + 4] * hs[cell * ch + B * 5 + c];
                pass[k] = sc[k] > prm.score_thresh;
                if (dense_scores) dense_scores[(int64_t)img * PC + (int64_t)p * C + c] = sc[k];
                if (pass[k]) atomicAdd(&s_hist[score_bin(__float_as_uint(sc[k]), lo_bits, hshift)], 1);
            }
            mcount += __popc(__ballot_sync(FULL, pass[k]));
        }
        if (lane == 0) s_m[c] = mcount;
    }
    __syncthreads();
    // ---- image-level work, two groups of warps side by side:
    //  * warp 0 -- class counts and T: the tier cuts from the candidate histogram
    //  * the next ceil(P/32) warps -- one thread per predictor: box assembly, and the coordinate statistics torchvision's
    //    offset trick needs over the predictors that are a candidate for at least one class (conf * max class prob passes
    //    iff some conf * prob passes: rounding is monotone; NaN probabilities never pass and are skipped by fmaxf)
    const int stat_w0 = (T >> 5) > (P + 31) / 32 ? 1 : 0;  // first statistics warp (warp 0 joins in when the CTA is small)
    if (wid >= stat_w0 && wid < stat_w0 + (P + 31) / 32) {
        const int p = tid - 32 * stat_w0;
        float mx = -INFINITY, mn = INFINITY;
        int fin = 1, nonan_l = 1;
        if (p < P) {
            const int cell = p / B, bi = p - cell * B;
            const int row = cell / S, col = cell - row * S;
            const float* t = hs + cell * ch + bi * 5;
            const float2 pr = priors[bi];
            const float cx = (t[0] + (float)col) * prm.stride_x;
            const float cy = (t[1] + (float)row) * prm.stride_y;
            const float w = t[2] * pr.x, h = t[3] * pr.y;
            float4 b = make_float4(cx - 0.5f * w, cy - 0.5f * h, cx + 0.5f * w, cy + 0.5f * h);
            if (prm.clip) {  // torch clamp(min=0,max=W): NaN stays NaN
                b.x = min_nan(max_nan(b.x, 0.f), prm.img_w); b.z = min_nan(max_nan(b.z, 0.f), prm.img_w);
                b.y = min_nan(max_nan(b.y, 0.f), prm.img_h); b.w = min_nan(max_nan(b.w, 0.f), prm.img_h);
            }
            pbox[p] = b;
            if (dense_boxes) dense_boxes[(int64_t)img * P + p] = b;
            const float* pc = hs + cell * ch + B * 5;
            float best = pc[0];
            for (int q = 1; q < C; ++q) best = fmaxf(best, pc[q]);
            if (t[4] * best > prm.score_thresh) {
                mx = max_nan(max_nan(b.x, b.y), max_nan(b.z, b.w));
                mn = min_nan(min_nan(b.x, b.y), min_nan(b.z, b.w));
                fin = (int)(isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w));
                nonan_l = (int)((b.x == b.x) && (b.y == b.y) && (b.z == b.z) && (b.w == b.w));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx = max_nan(mx, __shfl_xor_sync(FULL, mx, o));
            mn = min_nan(mn, __shfl_xor_sync(FULL, mn, o));
            fin &= __shfl_xor_sync(FULL, fin, o);
            nonan_l &= __shfl_xor_sync(FULL, nonan_l, o);
        }
        if (lane == 0) {
            s_mx[wid - stat_w0] = mx;
            s_mn[wid - stat_w0] = mn;
            s_fl[wid - stat_w0] = fin | (nonan_l << 1);
        }
    }
    if (wid == 0) {
        const int mq = lane < C ? s_m[lane] : 0;
        const int cnt_w = warp_sum(mq);
        const unsigned has = __ballot_sync(FULL, mq > 0);
        // two nested cuts from the candidate histogram: the highest bins holding >= target candidates
        unsigned cut[2] = {0u, 0u};
        const int targets[2] = {K + K / 6 + 8, 2 * K + 16};
        if (cnt_w > targets[0]) {
            int h8[8];
            const int4 ha = reinterpret_cast<const int4*>(s_hist)[lane * 2], hb = reinterpret_cast<const int4*>(s_hist)[lane * 2 + 1];
            h8[0] = ha.x; h8[1] = ha.y; h8[2] = ha.z; h8[3] = ha.w; h8[4] = hb.x; h8[5] = hb.y; h8[6] = hb.z; h8[7] = hb.w;
            const int mine = h8[0] + h8[1] + h8[2] + h8[3] + h8[4] + h8[5] + h8[6] + h8[7];
            int suf = mine;  // inclusive suffix sum over lanes (high scores live in the high bins)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_down_sync(FULL, suf, o);
                if (lane + o < 32) suf += v;
            }
#pragma unroll
            for (int tq = 0; tq < 2; ++tq) {
                const int target = targets[tq];
                if (cnt_w <= target) continue;  // warp-uniform: this tier would hold everything
                const unsigned reach = __ballot_sync(FULL, suf >= target);  // a prefix of lanes (lane 0: cnt > target)
                const int L = 31 - __clz(reach);
                int bin = 0;
                if (lane == L) {
                    int run = suf - mine;
                    bin = 8 * L;
#pragma unroll
                    for (int k = 7; k >= 0; --k) {
                        run += h8[k];
                        if (run >= target) {
                            bin = 8 * L + k;
                            break;
                        }
                    }
                }
                bin = __shfl_sync(FULL, bin, L);
                cut[tq] = bin > 0 ? lo_bits + ((unsigned)bin << hshift) : 0u;
            }
        }
        if (lane == 0) {
            s_img.cnt = cnt_w;
            s_img.gcat = has ? 31 - __clz(has) : 0;
            s_img.cut[0] = cut[0];
            s_img.cut[1] = cut[1];
        }
    }
    __syncthreads();
    float gmx = -INFINITY, gmn = INFINITY;
    int gfl = 3;
    for (int q = 0; q < (P + 31) / 32; ++q) {
        gmx = max_nan(gmx, s_mx[q]);
        gmn = min_nan(gmn, s_mn[q]);
        gfl &= s_fl[q];
    }
    const int cnt = s_img.cnt, gcat = s_img.gcat;
    // reference CPU rule: boxes.numel() <= 4000 -> coordinate-offset trick (torchvision/ops/boxes.py batched_nms)
    const bool trick = (prm.mode == DET_NMS_AUTO) ? (cnt <= 1000) : (prm.mode == DET_NMS_OFFSET_TRICK);
    const float span = trick ? gmx + 1.0f : 0.0f;  // max_coordinate + torch.tensor(1).to(boxes)
    const float thr_f = prm.thr_f;
    // categories can be swept independently iff shifted boxes of different categories cannot intersect
    const float far = gmx + (float)gcat * span;
    const bool sweep_ok = (gfl & 1) && gmn > -1.0f && thr_f >= 0.0f && isfinite(far);
    const bool by_cat = !trick || sweep_ok;
    const bool nonan = (gfl & 2) != 0;
    // tiers: NMS on the candidates above cut[0] (about 7/6 max_det of them); if that does not yield max_det survivors,
    // above cut[1] (about 2 max_det); finally on everything.  A cut of 0 means "that tier already holds everything".
    const unsigned tier_cut[3] = {s_img.cut[0], s_img.cut[1], 0u};
    DET_MARK(2);

    const uint64_t* fin_keys = buf_a;
    int nout = 0;

    if (by_cat) {
        // ---- E: pair filter over all predictor pairs, once per image (pair_may_suppress).  Row i meets the partners
        // (i + d) mod P, d = 1 .. P/2 (every unordered pair once); the T / P threads of a row split its partners, so box
        // i and its area bound are loaded once per thread.
        if (cnt > 0) {
            const float max_off = trick ? (float)gcat * span : 0.0f;  // the largest shift of a class with candidates
            const float r = max_nan(max_nan(fabsf(gmx), fabsf(gmn)), 1.0f) + max_off;
            const bool every = !(thr_f >= 0x1p-60f) || !(r < 0x1p60f);
            const float dl = r * 0x1p-20f;
            const float thr_lo = thr_f * (1.0f - 0x1p-20f);
            const int half = P >> 1, per_row = T / P, chunk = (half + per_row - 1) / per_row;
            const int i = tid % P, g = tid / P;
            if (g < per_row && half > 0) {
                const float4 a = pbox[i];
                const float al = lower_area(a, dl);
                const int d0 = g * chunk + 1, d1 = min(half, d0 + chunk - 1);
                int j = i + d0 >= P ? i + d0 - P : i + d0;
                for (int d = d0; d <= d1; ++d) {
                    // distance-P/2 pairs (P even) are met from both ends: taken from the lower half only
                    if (!((P & 1) == 0 && d == half && i >= half) && (every || pair_may_suppress(a, al, pbox[j], dl, thr_lo))) {
                        atomicOr(reinterpret_cast<unsigned*>(&s_edge[i]) + (j >> 5), 1u << (j & 31));
                        atomicOr(reinterpret_cast<unsigned*>(&s_edge[j]) + (i >> 5), 1u << (i & 31));
                    }
                    j = j + 1 == P ? 0 : j + 1;
                }
            }
        }
        __syncthreads();
        DET_MARK(5);
        const float off = trick ? (float)c * span : 0.0f;  // idxs.to(boxes) * (max_coordinate + 1)
        auto class_box = [&](int p) -> float4 {
            float4 b = pbox[p];
            if (trick) {
                b.x += off; b.y += off; b.z += off; b.w += off;
            }
            return b;
        };
        uint64_t mykey[4];
        bool mine_kept[4];
        unsigned base2 = 0u;
        int shift2 = 0;
        for (int tier = 0; tier < 3; ++tier) {
            const unsigned cut_bits = tier_cut[tier];
            if (tier < 2 && (cut_bits == 0u || cut_bits == tier_cut[tier + 1])) continue;  // same set as a later tier
            base2 = cut_bits ? cut_bits : lo_bits;     // every kept score of this pass has bits >= base2
            shift2 = score_shift(base2);
#pragma unroll
            for (int k = 0; k < 4; ++k) mine_kept[k] = false;
            if (cls_warp) {
                // ---- R: the class's tier candidates (bit p = predictor p), and those with an edge to another of them
                unsigned kept[4], open[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) kept[k] = __ballot_sync(FULL, pass[k] && __float_as_uint(sc[k]) >= cut_bits);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    bool touched = false;
                    if ((kept[k] >> lane) & 1u) {
                        const uint4 e = s_edge[lane + 32 * k];
                        touched = ((e.x & kept[0]) | (e.y & kept[1]) | (e.z & kept[2]) | (e.w & kept[3])) != 0u;
                    }
                    open[k] = __ballot_sync(FULL, touched);
                }
                // greedy over the open candidates: the best one (score descending, predictor ascending) is kept, and the
                // open candidates it shares an edge with are tested against it exactly.  Scores are >= +0: bit patterns
                // order like the values.
                while (open[0] | open[1] | open[2] | open[3]) {
                    unsigned best = 0u;
                    int bp = -1;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const unsigned sb = __float_as_uint(sc[k]);
                        if (((open[k] >> lane) & 1u) && (bp < 0 || sb > best)) {
                            best = sb;
                            bp = lane + 32 * k;
                        }
                    }
                    const unsigned top = __reduce_max_sync(FULL, bp >= 0 ? best : 0u);
                    const int w = (int)__reduce_min_sync(FULL, (bp >= 0 && best == top) ? (unsigned)bp : 0xffffffffu);
#pragma unroll
                    for (int k = 0; k < 4; ++k)  // (a constant index keeps the masks in registers)
                        if (k == (w >> 5)) open[k] &= ~(1u << (w & 31));
                    const uint4 ew = s_edge[w];
                    const float4 bw = class_box(w);
                    const float aw = box_area(bw);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const unsigned ek = (k == 0 ? ew.x : k == 1 ? ew.y : k == 2 ? ew.z : ew.w) & open[k];
                        bool dead = false;
                        if ((ek >> lane) & 1u) {
                            const float4 bb = class_box(lane + 32 * k);
                            dead = nonan ? nms_suppresses<true>(bw, aw, bb, box_area(bb), thr_f)
                                         : nms_suppresses<false>(bw, aw, bb, box_area(bb), thr_f);
                        }
                        const unsigned dm = __ballot_sync(FULL, dead);
                        open[k] &= ~dm;
                        kept[k] &= ~dm;
                    }
                }
                int kc = __popc(kept[0]) + __popc(kept[1]) + __popc(kept[2]) + __popc(kept[3]);
                while (kc > K) {  // only the first K survivors of a class can reach the output: drop the last one
                    unsigned worst = 0u;
                    int wp = -1;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const unsigned sb = __float_as_uint(sc[k]);
                        if (((kept[k] >> lane) & 1u) && (wp < 0 || sb <= worst)) {
                            worst = sb;
                            wp = lane + 32 * k;
                        }
                    }
                    const unsigned low = __reduce_min_sync(FULL, wp >= 0 ? worst : 0xffffffffu);
                    const int w = (int)__reduce_max_sync(FULL, (wp >= 0 && worst == low) ? (unsigned)wp : 0u);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k == (w >> 5)) kept[k] &= ~(1u << (w & 31));
                    --kc;
                }
                // ---- G: the lane's kept keys (descending-score bits | predictor * C + class) and their histogram
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if ((kept[k] >> lane) & 1u) {
                        const unsigned sb = __float_as_uint(sc[k]);
                        mine_kept[k] = true;
                        mykey[k] = ((uint64_t)(~sb) << 32) | (uint64_t)((unsigned)(lane + 32 * k) * (unsigned)C + (unsigned)c);
                        atomicAdd(&s_hist2[score_bin(sb, base2, shift2)], 1);
                    }
                }
                if (lane == 0 && kc) atomicAdd(&s_total, kc);
                DET_MARK(8);
            }
            __syncthreads();  // every class has emitted its kept keys
            if (tier == 2 || s_total >= K) break;  // enough: the first K kept detections all lie above this cut
            __syncthreads();                       // heavy suppression: redo on every candidate
            for (int i = tid; i < kFastBins; i += T) s_hist2[i] = 0;
            if (tid == 0) s_total = 0;
            __syncthreads();
        }
        DET_MARK(3);
        // ---- M: counting sort of the kept keys by score bin.  s_base[b] = kept keys in higher bins (they come first)
        const int total = s_total;
        if (wid == 0) {
            int h8[8];
            const int4 ha = reinterpret_cast<const int4*>(s_hist2)[lane * 2], hb = reinterpret_cast<const int4*>(s_hist2)[lane * 2 + 1];
            h8[0] = ha.x; h8[1] = ha.y; h8[2] = ha.z; h8[3] = ha.w; h8[4] = hb.x; h8[5] = hb.y; h8[6] = hb.z; h8[7] = hb.w;
            const int mine = h8[0] + h8[1] + h8[2] + h8[3] + h8[4] + h8[5] + h8[6] + h8[7];
            int suf = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_down_sync(FULL, suf, o);
                if (lane + o < 32) suf += v;
            }
            int run = suf - mine;  // kept keys in the bins of higher lanes
#pragma unroll
            for (int k = 7; k >= 0; --k) {
                s_base[lane * 8 + k] = run;
                run += h8[k];
            }
        }
        __syncthreads();
        // bin-grouped placement (arbitrary order inside a bin): slots are handed out by counting the bin back down
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            if (mine_kept[w]) {
                const int bin = score_bin(~(unsigned)(mykey[w] >> 32), base2, shift2);
                const int slot = s_base[bin] + atomicSub(&s_hist2[bin], 1) - 1;
                buf_a[slot] = mykey[w];
            }
        }
        __syncthreads();
        // rank inside the bin by direct comparison (keys are distinct); only the first K positions are output.  One
        // thread per SLOT: the lanes of a warp hold neighbouring bins, so their scans have similar lengths
        for (int t = tid; t < total; t += T) {
            const uint64_t key = buf_a[t];
            const int bin = score_bin(~(unsigned)(key >> 32), base2, shift2);
            const int b0 = s_base[bin], b1 = bin > 0 ? s_base[bin - 1] : total;
            int pos = b0;
            for (int j = b0; j < b1; ++j) pos += (buf_a[j] < key) ? 1 : 0;
            if (pos < K) buf_b[pos] = key;
        }
        __syncthreads();
        fin_keys = buf_b;
        nout = min(total, K);
    } else {
        // ---- slow exact path (offset trick with non-finite / <= -1 coordinates): global greedy by repeated arg-max
        unsigned char* st = reinterpret_cast<unsigned char*>(buf_b + lay.pcp);
        for (int f = tid; f < PC; f += T) {
            const int p = f / C, q = f - p * C, cell = p / B, bi = p - cell * B;
            const float s = hs[cell * ch + bi * 5 + 4] * hs[cell * ch + B * 5 + q];
            st[f] = (s > prm.score_thresh) ? 1 : 0;
        }
        __syncthreads();
        int k = 0;
        while (k < K) {
            if (tid == 0) s_best = ~0ull;
            __syncthreads();
            unsigned long long best = ~0ull;
            for (int f = tid; f < PC; f += T) {
                if (st[f] != 1) continue;
                const int p = f / C, q = f - p * C, cell = p / B, bi = p - cell * B;
                const float s = hs[cell * ch + bi * 5 + 4] * hs[cell * ch + B * 5 + q];
                const unsigned long long key = ((unsigned long long)(~__float_as_uint(s)) << 32) | (unsigned)f;
                best = key < best ? key : best;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long v = __shfl_xor_sync(FULL, best, o);
                best = v < best ? v : best;
            }
            if (lane == 0 && best != ~0ull) atomicMin(&s_best, best);
            __syncthreads();
            const unsigned long long bk = s_best;
            if (bk == ~0ull) break;
            const int fs = (int)(unsigned)bk;
            const int ps = fs / C, qs = fs - ps * C;
            float4 kb = pbox[ps];
            const float koff = (float)qs * span;
            kb.x += koff; kb.y += koff; kb.z += koff; kb.w += koff;
            const float ka = box_area(kb);
            for (int f = tid; f < PC; f += T) {
                if (st[f] != 1 || f == fs) continue;
                const int p = f / C, q = f - p * C;
                float4 b = pbox[p];
                const float o = (float)q * span;
                b.x += o; b.y += o; b.z += o; b.w += o;
                if (nms_suppresses<false>(kb, ka, b, box_area(b), thr_f)) st[f] = 0;
            }
            if (tid == 0) {
                buf_a[k] = bk;
                st[fs] = 2;
            }
            ++k;
            __syncthreads();
        }
        __syncthreads();
        fin_keys = buf_a;
        nout = k;
    }
    DET_MARK(4);
    // ---- detections, by descending score
    for (int j = tid; j < nout; j += T) {
        const uint64_t key = fin_keys[j];
        const unsigned flat = (unsigned)key;
        const int64_t o = (int64_t)img * prm.max_det + j;
        if (prm.flat32) reinterpret_cast<int32_t*>(det_flat)[o] = (int32_t)flat;
        else det_flat[o] = (int64_t)flat;
        if (det_boxes) det_boxes[o] = pbox[flat / (unsigned)C];
        if (det_scores) det_scores[o] = __uint_as_float(~(unsigned)(key >> 32));
    }
    if (tid == 0) det_count[img] = nout;
    DET_MARK(15);
}

}  // namespace det
