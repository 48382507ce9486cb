// Shared pieces of the training side (assign_loss.cu: generic anchors + dense loss; assign_grid.cu: grid anchors, sampled
// loss): the Matcher rule, the counter-based sampling hashes, the label-row view and the loss arithmetic.
#pragma once
#include "common.cuh"

namespace det {

constexpr int kMaxThresholds = 8;
struct MatchRule {
    float thr[kMaxThresholds];
    int8_t lab[kMaxThresholds + 1];
    int nthr;
    int allow_lq;
};

__device__ __forceinline__ int8_t bucket_label(const MatchRule& r, float v) {
    // thresholds ascending: bucket [thr[k-1], thr[k]); static indices only, so the rule stays in the constant bank
    if (r.nthr <= 2) {  // the reference's configurations: [0.3, 0.7] (RPN) and [0.5] (ROI heads); thr[i >= nthr] = +inf
        int8_t lab = r.lab[0];
        if (v >= r.thr[0]) lab = r.lab[1];
        if (v >= r.thr[1]) lab = r.lab[2];
        return lab;
    }
    int8_t lab = r.lab[0];
#pragma unroll
    for (int i = 0; i < kMaxThresholds; ++i)
        if (i < r.nthr && v >= r.thr[i]) lab = r.lab[i + 1];
    return lab;
}

// IoUs are >= 0, so their bit patterns order like unsigned integers
__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t mix32(uint32_t h) {
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    return h;
}
__device__ __forceinline__ uint32_t sample_key(uint32_t img_seed, uint32_t j) { return mix32(j * 0x9E3779B1u + img_seed); }
// per-image seed of the 64-bit call seed: the keys of image `img` are sample_key(image_seed(seed, img), j)
__device__ __forceinline__ uint32_t image_seed(uint64_t seed, int img) {
    return mix32((uint32_t)seed ^ mix32((uint32_t)(seed >> 32) + 0x632BE5ABu * (uint32_t)(img + 1)));
}

// b-bit bijection (odd multiplies and right xor-shifts are invertible mod 2^b): k -> a pseudo-random permutation of
// [0, 2^b).  Walking k = 0, 1, 2, ... and keeping the first `want` indices that fall inside the row and carry the class
// label IS a uniformly random `want`-subset of the class -- in O(want / density) steps instead of one hash per anchor.
// Used for a DENSE class (the background of an RPN image: ~98 % of the anchors, 128-256 wanted).
__device__ __forceinline__ uint32_t perm_bits(uint32_t k, uint32_t s0, int b) {
    const uint32_t mask = (b >= 32) ? 0xffffffffu : ((1u << b) - 1u);
    const int h = (b + 1) >> 1;
    uint32_t x = (k * 0x9E3779B1u + s0) & mask;
    x ^= x >> h; x = (x * 0x7FEB352Du) & mask;
    x ^= x >> h; x = (x * 0x846CA68Bu) & mask;
    x ^= x >> h;
    return x;
}

// labels of one image in 16-byte granules of the GLOBAL address space (rows of odd length start unaligned): granule c
// covers row offsets [16c - a, 16c - a + 16), a = misalignment of the row start; bytes outside the row read as -1
struct RowView {
    int8_t* row;
    int64_t r;
    int a, ngran;
    __device__ RowView(int8_t* p, int64_t r_) : row(p), r(r_) {
        a = (int)(reinterpret_cast<uintptr_t>(p) & 15);
        ngran = (int)((a + r + 15) >> 4);
    }
    __device__ __forceinline__ int64_t first(int c) const { return (int64_t)c * 16 - a; }
    __device__ __forceinline__ bool full(int c) const { return first(c) >= 0 && first(c) + 16 <= r; }
    // the granule as 4 little-endian words of 4 labels
    __device__ __forceinline__ uint4 load(int c) const {
        const int64_t lo = first(c);
        if (full(c)) return *reinterpret_cast<const uint4*>(row + lo);
        uint32_t w[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        for (int k = 0; k < 16; ++k)
            if (lo + k >= 0 && lo + k < r)
                w[k >> 2] = (w[k >> 2] & ~(0xffu << (8 * (k & 3)))) | ((uint32_t)(uint8_t)row[lo + k] << (8 * (k & 3)));
        return make_uint4(w[0], w[1], w[2], w[3]);
    }
    __device__ __forceinline__ void store(int c, const uint4 q) const {
        const int64_t lo = first(c);
        if (full(c)) {
            *reinterpret_cast<uint4*>(row + lo) = q;
        } else {
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
            for (int k = 0; k < 16; ++k)
                if (lo + k >= 0 && lo + k < r) row[lo + k] = (int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xffu);
        }
    }
};

// cls: 0 = positive (anything that is neither -1 nor background), 1 = background (label == 0), -1 = ignored
__device__ __forceinline__ int label_class(int8_t l) { return l == 0 ? 1 : (l == -1 ? -1 : 0); }

// per-byte masks (0xff where true) of a word of 4 labels
__device__ __forceinline__ uint32_t bytes_eq(uint32_t w, uint32_t pattern) { return __vcmpeq4(w, pattern); }

// smooth-L1 value and derivative wrt the prediction (fvcore semantics: beta < 1e-5 -> pure L1)
__device__ __forceinline__ void smooth_l1(float pred, float tgt, float beta, float& val, float& grad) {
    const float d = pred - tgt, n = fabsf(d);
    const float sgn = (d > 0.f) ? 1.f : ((d < 0.f) ? -1.f : 0.f);
    if (beta < 1e-5f) {
        val = n;
        grad = sgn;
    } else if (n < beta) {
        val = 0.5f * n * n / beta;
        grad = d / beta;
    } else {
        val = n - 0.5f * beta;
        grad = sgn;
    }
}

// GIoU loss of the box decoded from deltas `p` on anchor `a` against gt `g`, and its gradient wrt the four deltas.
// Value: fvcore.nn.giou_loss restated (oracle/ref_torch.py giou_sum; third-party, unpinned by the reference):
//   iou = I / (U + eps), loss = 1 - iou + (H - U) / (H + eps), I = 0 unless the boxes strictly overlap, eps = 1e-7.
// Gradient: what autograd produces for that expression composed with Box2BoxTransform.apply_deltas
// (box_regression.py:87-115): ties of max / min split the gradient in half, clamp(max=) passes it up to equality.
__device__ __forceinline__ float giou_fwd_bwd(const float4 p, const float4 a, const float4 g, const CodecWeights wt,
                                              float scale_clamp, float4& grad) {
    const float eps = 1e-7f;
    const float w = a.z - a.x, h = a.w - a.y;
    const float cx = a.x + 0.5f * w, cy = a.y + 0.5f * h;
    const float dx = p.x / wt.wx, dy = p.y / wt.wy;
    const float dw_raw = p.z / wt.ww, dh_raw = p.w / wt.wh;
    const float dw = fminf(dw_raw, scale_clamp), dh = fminf(dh_raw, scale_clamp);
    const float pcx = dx * w + cx, pcy = dy * h + cy;
    const float pw = expf(dw) * w, ph = expf(dh) * h;
    const float x1 = pcx - 0.5f * pw, y1 = pcy - 0.5f * ph, x2 = pcx + 0.5f * pw, y2 = pcy + 0.5f * ph;
    const float ix1 = fmaxf(x1, g.x), iy1 = fmaxf(y1, g.y), ix2 = fminf(x2, g.z), iy2 = fminf(y2, g.w);
    const bool overlap = (iy2 > iy1) && (ix2 > ix1);
    const float I = overlap ? (ix2 - ix1) * (iy2 - iy1) : 0.0f;
    const float A = (x2 - x1) * (y2 - y1);
    const float U = A + (g.z - g.x) * (g.w - g.y) - I;
    const float hx1 = fminf(x1, g.x), hy1 = fminf(y1, g.y), hx2 = fmaxf(x2, g.z), hy2 = fmaxf(y2, g.w);
    const float H = (hx2 - hx1) * (hy2 - hy1);
    const float iou = I / (U + eps);
    const float loss = 1.0f - (iou - (H - U) / (H + eps));
    // partial derivatives of the loss wrt I, A (through U) and H
    const float ue = U + eps, he = H + eps;
    const float dI = -(ue + I) / (ue * ue) + 1.0f / he;
    const float dA = I / (ue * ue) - 1.0f / he;
    const float dH = ue / (he * he);
    auto sel = [](float v, float o, bool take_greater) {  // d max(v,o)/dv or d min(v,o)/dv
        return v == o ? 0.5f : ((take_greater ? v > o : v < o) ? 1.0f : 0.0f);
    };
    float gx1 = -dA * (y2 - y1) - dH * (hy2 - hy1) * sel(x1, g.x, false);
    float gx2 = dA * (y2 - y1) + dH * (hy2 - hy1) * sel(x2, g.z, true);
    float gy1 = -dA * (x2 - x1) - dH * (hx2 - hx1) * sel(y1, g.y, false);
    float gy2 = dA * (x2 - x1) + dH * (hx2 - hx1) * sel(y2, g.w, true);
    if (overlap) {
        gx1 -= dI * (iy2 - iy1) * sel(x1, g.x, true);
        gx2 += dI * (iy2 - iy1) * sel(x2, g.z, false);
        gy1 -= dI * (ix2 - ix1) * sel(y1, g.y, true);
        gy2 += dI * (ix2 - ix1) * sel(y2, g.w, false);
    }
    const float gcx = gx1 + gx2, gcy = gy1 + gy2;
    const float gpw = 0.5f * (gx2 - gx1), gph = 0.5f * (gy2 - gy1);
    grad.x = gcx * w / wt.wx;
    grad.y = gcy * h / wt.wy;
    grad.z = (dw_raw <= scale_clamp) ? gpw * pw / wt.ww : 0.0f;
    grad.w = (dh_raw <= scale_clamp) ? gph * ph / wt.wh : 0.0f;
    return loss;
}

// ---- one anchor against all gt boxes of its image (the sample-list-only assignment of assign_grid.cu and its sampler)
struct Verdict {
    float best;
    int argmax;   // first gt attaining the column maximum (torch.max(dim=0))
    int first_q;  // first gt that makes the anchor a candidate (IoU >= tau or IoU == its row maximum); -1: none
    bool hit;     // low-quality promotion (matcher.py:110-120)
};

__device__ __forceinline__ Verdict anchor_verdict(const float4 ab, const float4* __restrict__ gt, const float* __restrict__ rowmax,
                                                  int g0, int G, float tau, bool allow_lq) {
    Verdict v{0.0f, 0, -1, false};
    const float aa = box_area(ab);
    for (int t = 0; t < G; ++t) {
        const float4 gb = gt[g0 + t];
        const float q = pair_iou(gb, box_area(gb), ab, aa);
        if (q > v.best) {
            v.best = q;
            v.argmax = t;
        }
        const bool lq = allow_lq && q == rowmax[g0 + t];
        v.hit |= lq;
        if (v.first_q < 0 && (q >= tau || lq)) v.first_q = t;
    }
    return v;
}

__device__ __forceinline__ int verdict_label(const MatchRule& rule, const Verdict& v, int G) {
    if (G == 0) return rule.lab[0];
    return v.hit ? 1 : (int)bucket_label(rule, v.best);
}

#endif  // __CUDACC__

static inline int fill_rule(MatchRule& rule, const float* thresholds_host, const int32_t* labels_host, int num_thresholds,
                     int allow_low_quality) {
    if (num_thresholds < 0 || num_thresholds > kMaxThresholds || !labels_host || (num_thresholds && !thresholds_host)) {
        set_error("bad matcher rule (at most %d thresholds)", kMaxThresholds);
        return DET_ERR_BAD_ARG;
    }
    rule.nthr = num_thresholds;
    rule.allow_lq = allow_low_quality ? 1 : 0;
    for (int i = 0; i < kMaxThresholds; ++i) rule.thr[i] = i < num_thresholds ? thresholds_host[i] : INFINITY;
    for (int i = 0; i <= kMaxThresholds; ++i) rule.lab[i] = i <= num_thresholds ? (int8_t)labels_host[i] : (int8_t)0;
    for (int i = 0; i + 1 < num_thresholds; ++i)
        if (!(thresholds_host[i] <= thresholds_host[i + 1])) {
            set_error("thresholds must be ascending");
            return DET_ERR_BAD_ARG;
        }
    return DET_OK;
}

}  // namespace det
