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
//   C  order-preserving ballot compaction of the class's candidates
//   D  rank-by-counting sort (score descending, predictor ascending) -> boxes (+ coordinate offset when the
//      image takes torchvision's offset-trick branch), areas and scores in sorted order
//   E  every unordered pair of the class tested exactly once, load-balanced over the 32 lanes; a hit sets one bit
//      of the earlier box's suppression row (shared-memory atomicOr) and flags the row as non-empty
//   F  greedy resolution on the bit rows alone, visiting only non-empty rows
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

struct FastLayout {
    int hs_floats, pp, cls_stride, pcp;
    size_t bytes;
    __host__ __device__ constexpr FastLayout(int s2, int ch, int p, int c)
        : hs_floats((s2 * ch + 3) & ~3),
          pp((p + 3) & ~3),
          // per class: sbox float4[pp] | rows uint4[pp] | sarea float[pp] | skey u32[pp] | spred u8[pad16(pp)]
          cls_stride(((p + 3) & ~3) * 40 + ((((p + 3) & ~3) + 15) & ~15)),
          pcp((p * c + 3) & ~3),
          bytes(0) {
        size_t cls_bytes = (size_t)cls_stride * c;
        const size_t merge_bytes = (size_t)pcp * 17 + 16;  // two u64 key buffers + one state byte per (p, c)
        if (cls_bytes < merge_bytes) cls_bytes = merge_bytes;
        bytes = (size_t)hs_floats * 4 + (size_t)pp * 16 + ((cls_bytes + 15) & ~(size_t)15);
    }
};

// histogram bin of a score: bits in [base, 0x3F800000], `shift` chosen so that the range spans <= 256 bins
__device__ __forceinline__ int score_bin(unsigned bits, unsigned base, int shift) {
    return min(kFastBins - 1, (int)((bits - base) >> shift));
}
__device__ __forceinline__ int score_shift(unsigned base) {
    return 0x3F800000u > base ? max(0, 32 - __clz(0x3F800000u - base) - 8) : 0;
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
    unsigned char* cls_region = reinterpret_cast<unsigned char*>(pbox + Pp);
    __shared__ int s_m[kFastMaxC];
    __shared__ float s_mx[4], s_mn[4];
    __shared__ int s_fl[4];
    __shared__ unsigned s_nz[kFastMaxC][4];
    __shared__ __align__(16) int4 s_work[kFastMaxC];  // per class: candidates, 32-item chunks of pair tests, 2^32/half
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
    const unsigned lt_mask = (1u << lane) - 1u;
    const int img = blockIdx.x;
    const int K = (int)min(prm.max_det, (int64_t)PC);

    pdl_trigger();  // the next launch of this stream may take SM slots as they free up (it parks in its own pdl_wait)
    for (int i = tid; i < kFastBins; i += T) {
        s_hist[i] = 0;
        s_hist2[i] = 0;
    }
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

    uint64_t* buf_a = reinterpret_cast<uint64_t*>(cls_region);
    uint64_t* buf_b = buf_a + lay.pcp;
    const uint64_t* fin_keys = buf_a;
    int nout = 0;

    if (by_cat) {
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
            unsigned char* my = cls_region + (size_t)(cls_warp ? c : 0) * lay.cls_stride;
            unsigned* skey = reinterpret_cast<unsigned*>(my + Pp * 36);
            unsigned char* spred = my + Pp * 40;
            int m = 0;
            if (cls_warp) {
                float4* sbox = reinterpret_cast<float4*>(my);
                uint4* rows4 = reinterpret_cast<uint4*>(my + Pp * 16);
                unsigned* rows = reinterpret_cast<unsigned*>(rows4);
                float* sarea = reinterpret_cast<float*>(my + Pp * 32);
                unsigned* ckey = rows;  // unsorted candidates live in the row storage until the rows are needed
                unsigned char* cp = reinterpret_cast<unsigned char*>(rows + Pp);
                // ---- C: order-preserving compaction (predictor ascending)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool in = pass[k] && __float_as_uint(sc[k]) >= cut_bits;
                    const unsigned bal = __ballot_sync(FULL, in);
                    if (in) {
                        const int pos = m + __popc(bal & lt_mask);
                        ckey[pos] = __float_as_uint(sc[k]);  // scores are >= +0: bit patterns order like the values
                        cp[pos] = (unsigned char)(lane + 32 * k);
                    }
                    m += __popc(bal);
                }
                __syncwarp();
                DET_MARK(5);
                // ---- D: rank by counting -> sorted order (score descending, predictor ascending)
                const float off = trick ? (float)c * span : 0.0f;  // idxs.to(boxes) * (max_coordinate + 1)
                for (int i0 = 0; i0 < m; i0 += 32) {
                    const int i = i0 + lane;
                    const bool has = i < m;
                    const unsigned si = has ? ckey[i] : 0u;
                    int rank = 0;
#pragma unroll 4
                    for (int j = 0; j < m; ++j) {
                        const unsigned sj = ckey[j];
                        rank += ((sj > si) || (sj == si && j < i)) ? 1 : 0;
                    }
                    if (has) {
                        const int p = (int)cp[i];
                        float4 b = pbox[p];
                        if (trick) {
                            b.x += off; b.y += off; b.z += off; b.w += off;
                        }
                        sbox[rank] = b;
                        sarea[rank] = box_area(b);
                        skey[rank] = si;
                        spred[rank] = (unsigned char)p;
                    }
                }
                __syncwarp();
                for (int r = lane; r < m; r += 32) rows4[r] = make_uint4(0u, 0u, 0u, 0u);
                if (lane < 4) s_nz[c][lane] = 0u;
                if (lane == 0) {
                    // the class's pair items (m * floor(m/2), see E) in chunks of 32 for the CTA-wide sweep below
                    const int half = m >> 1;
                    s_work[c] = make_int4(m, m >= 2 ? (m * half + 31) >> 5 : 0,
                                          half > 1 ? (int)((0xFFFFFFFFu / (unsigned)half) + 1u) : 0, 0);
                }
                DET_MARK(6);
            } else if (wid < kFastMaxC && lane == 0) {
                s_work[wid] = make_int4(0, 0, 0, 0);
            }
            __syncthreads();
            // ---- E: every unordered pair of every class exactly once.  A class of m candidates has m * floor(m/2) items
            // (item q -> row r = q / half, distance d = q % half + 1, partner (r + d) mod m), cut into chunks of 32; the
            // chunks of ALL classes are dealt round-robin to the warps of the CTA, so a class with many candidates no
            // longer holds up the image (the classes' sizes differ by 2-3x and the work is quadratic in them).
            {
                const int nw = T >> 5;
                const int4 wk = lane < C ? s_work[lane] : make_int4(0, 0, 0, 0);
                int incl = wk.y;  // inclusive scan of the chunk counts over the classes (lane = class)
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(FULL, incl, o);
                    if (lane >= o) incl += v;
                }
                const int chunks = __shfl_sync(FULL, incl, 31);
                for (int g = wid; g < chunks; g += nw) {
                    const int cls = __popc(__ballot_sync(FULL, incl <= g));  // classes that end at or before chunk g
                    const int first = __shfl_sync(FULL, incl - wk.y, cls);
                    const int mm = __shfl_sync(FULL, wk.x, cls);
                    const unsigned inv = (unsigned)__shfl_sync(FULL, wk.z, cls);
                    const int half = mm >> 1, items = mm * half;
                    const int q = ((g - first) << 5) + lane;
                    if (q >= items) continue;
                    unsigned char* cm = cls_region + (size_t)cls * lay.cls_stride;
                    const float4* cbox = reinterpret_cast<const float4*>(cm);
                    unsigned* crows = reinterpret_cast<unsigned*>(cm + Pp * 16);
                    const float* carea = reinterpret_cast<const float*>(cm + Pp * 32);
                    const int r = half > 1 ? (int)__umulhi((unsigned)q, inv) : q;
                    const int d = q - r * half + 1;
                    if (((mm & 1) == 0) && d == half && r >= half) continue;  // distance-m/2 pairs: from the lower half only
                    int j = r + d;
                    j = (j >= mm) ? j - mm : j;
                    const int lo = min(r, j), hi = max(r, j);
                    const float4 ba = cbox[lo], bb = cbox[hi];
                    const float aa = carea[lo], ab = carea[hi];
                    const bool hit = nonan ? nms_suppresses<true>(ba, aa, bb, ab, thr_f)
                                           : nms_suppresses<false>(ba, aa, bb, ab, thr_f);
                    if (hit) {
                        atomicOr(crows + lo * 4 + (hi >> 5), 1u << (hi & 31));
                        atomicOr(&s_nz[cls][lo >> 5], 1u << (lo & 31));
                    }
                }
            }
            __syncthreads();
            DET_MARK(7);
            if (cls_warp) {
                const uint4* rows4 = reinterpret_cast<const uint4*>(my + Pp * 16);
                // ---- F: greedy resolution on the bit rows (uniform across the warp), only non-empty rows matter
                unsigned alive[4];
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const int bits = min(32, max(0, m - 32 * w));
                    alive[w] = bits == 32 ? 0xffffffffu : ((1u << bits) - 1u);
                }
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    unsigned nzw = s_nz[c][w];
                    while (nzw) {
                        const int b = __ffs(nzw) - 1;
                        nzw &= nzw - 1;
                        if ((alive[w] >> b) & 1u) {
                            const uint4 rw = rows4[w * 32 + b];
                            alive[0] &= ~rw.x; alive[1] &= ~rw.y; alive[2] &= ~rw.z; alive[3] &= ~rw.w;
                        }
                    }
                }
                int kc = __popc(alive[0]) + __popc(alive[1]) + __popc(alive[2]) + __popc(alive[3]);
                while (kc > K) {  // only the first K survivors of a class can reach the output
#pragma unroll
                    for (int w = 3; w >= 0; --w)
                        if (alive[w]) {
                            alive[w] &= ~(0x80000000u >> __clz(alive[w]));
                            break;
                        }
                    --kc;
                }
                // ---- G: the lane's kept keys (descending-score bits | predictor * C + class) and their histogram
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    if ((alive[w] >> lane) & 1u) {
                        const int i = lane + 32 * w;
                        const unsigned sb = skey[i];
                        mine_kept[w] = true;
                        mykey[w] = ((uint64_t)(~sb) << 32) | (uint64_t)((unsigned)spred[i] * (unsigned)C + (unsigned)c);
                        atomicAdd(&s_hist2[score_bin(sb, base2, shift2)], 1);
                    }
                }
                if (lane == 0 && kc) atomicAdd(&s_total, kc);
                DET_MARK(8);
            }
            __syncthreads();  // every class is done with its scratch: the merge buffers may now overwrite it
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
