// Training side (subsystem 4): IoU target assignment, on-device fg/bg subsampling, and the fused loss
// forward + backward kernels.
//
// Reference behaviour reproduced (paths relative to the reference root):
//   python/src/models/rpn.py:161-168        per image: pairwise_iou(gt, anchors) -> Matcher
//   python/src/models/components/matcher.py:53-120   column max/argmax, threshold buckets, low-quality promotion
//   python/src/utils.py:34-76 + rpn.py:108-130       subsample_labels / _subsample_labels (counts; RNG differs)
//   python/src/models/rpn.py:187-244 + components/box_regression.py:128-168   losses (BCE-with-logits + L1/smooth-L1)
// The (G,R) IoU matrix, the (N,R,4) matched-gt tensor and the (N,R,4) target-delta tensor of the reference are
// never materialised: IoUs are recomputed from the box tables, targets are encoded on the fly for positives only.
#include "common.cuh"
#include "peer.cuh"
#include "assign.cuh"

namespace det {

constexpr int kMatchThreads = 256;
constexpr int kMatchPerThread = 4;
constexpr int kGtChunk = 512;

// Bounding box of a group of anchors (union of finite coordinates): a gt box that does not overlap it has zero
// intersection -- hence IoU exactly 0 -- with every anchor of the group, so it is skipped as a whole ("culled").
// Anchors are laid out (h, w, a): 128 consecutive anchors are a piece of one feature-map row, and most gt boxes miss it.
struct BlockBox {
    float x1, y1, x2, y2;
};

// true iff the gt box certainly has zero intersection with every anchor inside `bb` (comparisons with NaN are false:
// a NaN gt box is never culled and takes the exact path)
__device__ __forceinline__ bool culled_by(const BlockBox& bb, const float4 g) {
    return g.z <= bb.x1 || g.x >= bb.x2 || g.w <= bb.y1 || g.y >= bb.y2;
}

constexpr int kMatchImgs = 8;  // at most this many images are walked by one CTA (anchors + block box stay in registers)

// bounding box of the 4 x 32 anchors held by a warp (finite coordinates only; NaN anchors never intersect anything)
__device__ __forceinline__ BlockBox warp_bbox(const float4* ab, const bool* valid) {
    float x1 = INFINITY, y1 = INFINITY, x2 = -INFINITY, y2 = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (valid[k]) {
            x1 = fminf(x1, ab[k].x); y1 = fminf(y1, ab[k].y);
            x2 = fmaxf(x2, ab[k].z); y2 = fmaxf(y2, ab[k].w);
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x1 = fminf(x1, __shfl_xor_sync(0xffffffffu, x1, o)); y1 = fminf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
        x2 = fmaxf(x2, __shfl_xor_sync(0xffffffffu, x2, o)); y2 = fmaxf(y2, __shfl_xor_sync(0xffffffffu, y2, o));
    }
    return BlockBox{x1, y1, x2, y2};
}

// pass 1: per anchor column max / argmax over the image's gt boxes, threshold label; per gt row max and per-CTA max.
// Every WARP is on its own (no shared memory, no block barrier): it owns 128 consecutive anchors for up to `imgs`
// images -- lane l holds anchors l, l+32, l+64, l+96 of them in registers (coalesced loads and stores) -- together
// with their bounding box.  Per image the lanes first look at one gt box each (coalesced load) and vote which boxes
// overlap the warp's bounding box at all (every other box has IoU exactly 0 with all 128 anchors); only those are
// handed round with shuffles and evaluated, 4 IoUs per lane.  Row maxima go to `rowmax` / `blockmax` (zeroed by the
// host) with one atomic per warp and surviving gt box.
template <bool FULL>
__device__ __forceinline__ void match_pass1_warp(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off,
                                                 const float4* __restrict__ anchors, int i0, int ni, int64_t r,
                                                 int64_t abase, const MatchRule& rule, int64_t* __restrict__ matched,
                                                 int8_t* __restrict__ labels, float* __restrict__ matched_iou,
                                                 float* __restrict__ rowmax, float* __restrict__ bmax) {
    const unsigned FULLMASK = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t j0 = abase + lane;  // this lane's anchors: j0 + 32 k
    float4 ab[4];
    float aa[4];
    bool valid[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        valid[k] = FULL || (j0 + 32 * k < r);
        ab[k] = valid[k] ? anchors[j0 + 32 * k] : make_float4(0.f, 0.f, 0.f, 0.f);
        aa[k] = box_area(ab[k]);
    }
    const BlockBox wb = warp_bbox(ab, valid);
    for (int ii = 0; ii < ni; ++ii) {
        const int img = i0 + ii;
        const int g0 = gt_off[img], G = gt_off[img + 1] - g0;
        float best[4] = {0.f, 0.f, 0.f, 0.f};  // IoUs are >= 0 and only a strictly larger one replaces the incumbent:
        int bidx[4] = {0, 0, 0, 0};            // gt 0 wins ties at 0, exactly like torch.max(dim=0)
        for (int t0 = 0; t0 < G; t0 += 32) {
            float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
            bool hit = false;
            if (t0 + lane < G) {
                mine = gt[g0 + t0 + lane];
                hit = !culled_by(wb, mine);
            }
            unsigned todo = __ballot_sync(FULLMASK, hit);
            while (todo) {  // ascending gt index: the first maximum wins
                const int src = __ffs(todo) - 1;
                todo &= todo - 1;
                const float4 gb = make_float4(__shfl_sync(FULLMASK, mine.x, src), __shfl_sync(FULLMASK, mine.y, src),
                                              __shfl_sync(FULLMASK, mine.z, src), __shfl_sync(FULLMASK, mine.w, src));
                const float ga = box_area(gb);
                const int t = t0 + src;
                float rm = 0.0f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // pairwise_iou(gt, anchors): boxes1 = gt, boxes2 = anchors (rpn.py:167)
                    const float v = valid[k] ? pair_iou(gb, ga, ab[k], aa[k]) : 0.0f;
                    if (v > best[k]) {
                        best[k] = v;
                        bidx[k] = t;
                    }
                    rm = fmaxf(rm, v);
                }
                if (rule.allow_lq) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) rm = fmaxf(rm, __shfl_xor_sync(FULLMASK, rm, o));
                    if (lane == 0 && rm > 0.0f) {
                        atomic_max_nonneg(&rowmax[g0 + t], rm);
                        atomic_max_nonneg(&bmax[g0 + t], rm);  // pass 2 only revisits the CTAs holding the row maximum
                    }
                }
            }
        }
        const int64_t o = (int64_t)img * r + j0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!valid[k]) continue;
            matched[o + 32 * k] = bidx[k];
            labels[o + 32 * k] = G == 0 ? rule.lab[0] : bucket_label(rule, best[k]);  // matcher.py:67-77
            if (matched_iou) matched_iou[o + 32 * k] = best[k];
        }
    }
}

__global__ void __launch_bounds__(kMatchThreads)
match_pass1_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, const float4* __restrict__ anchors,
                   int n, int imgs, int64_t r, int64_t sum_g, MatchRule rule, int64_t* __restrict__ matched,
                   int8_t* __restrict__ labels, float* __restrict__ matched_iou, float* __restrict__ rowmax,
                   float* __restrict__ blockmax) {
    const int i0 = blockIdx.y * imgs, ni = min(imgs, n - i0);
    const int64_t abase = (int64_t)blockIdx.x * (kMatchThreads * kMatchPerThread) + (int64_t)(threadIdx.x >> 5) * 128;
    float* bmax = blockmax + (int64_t)blockIdx.x * sum_g;
    if (abase + 128 <= r)  // warp-uniform: all 128 anchors exist
        match_pass1_warp<true>(gt, gt_off, anchors, i0, ni, r, abase, rule, matched, labels, matched_iou, rowmax, bmax);
    else if (abase < r)
        match_pass1_warp<false>(gt, gt_off, anchors, i0, ni, r, abase, rule, matched, labels, matched_iou, rowmax, bmax);
}

// pass 2 (low-quality promotion, matcher.py:96-120): label 1 wherever IoU(gt, anchor) == max over anchors for that gt.
// Only a CTA whose own maximum for a gt (recorded by pass 1) equals the row maximum can hold such an anchor; a gt whose
// row maximum is 0 promotes EVERY anchor (the reference's `Q == rowmax` is true everywhere, matcher.py:110-113).
__global__ void __launch_bounds__(kMatchThreads)
match_pass2_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, const float4* __restrict__ anchors,
                   int n, int imgs, int64_t r, int64_t sum_g, const float* __restrict__ rowmax,
                   const float* __restrict__ blockmax, int8_t* __restrict__ labels) {
    __shared__ unsigned short s_list[kGtChunk];
    __shared__ int s_nlist, s_all;
    __shared__ int s_off[kMatchImgs + 1];
    const int i0 = blockIdx.y * imgs, ni = min(imgs, n - i0);
    const int64_t base = (int64_t)blockIdx.x * (kMatchThreads * kMatchPerThread);
    if (threadIdx.x <= ni) s_off[threadIdx.x] = gt_off[i0 + threadIdx.x];
    __syncthreads();
    for (int ii = 0; ii < ni; ++ii) {
        const int img = i0 + ii;
        const int g0 = s_off[ii], G = s_off[ii + 1] - g0;
        for (int c0 = 0; c0 < G; c0 += kGtChunk) {
            const int cn = min(kGtChunk, G - c0);
            __syncthreads();
            if (threadIdx.x == 0) {
                s_nlist = 0;
                s_all = 0;
            }
            __syncthreads();
            for (int t = threadIdx.x; t < cn; t += kMatchThreads) {
                const float rm = rowmax[g0 + c0 + t];
                if (rm == 0.0f) s_all = 1;
                else if (blockmax[(int64_t)blockIdx.x * sum_g + g0 + c0 + t] == rm)
                    s_list[atomicAdd(&s_nlist, 1)] = (unsigned short)t;
            }
            __syncthreads();
            const int ns = s_nlist;
            const bool all = s_all != 0;
            if (ns == 0 && !all) continue;  // block-uniform: the usual case
#pragma unroll
            for (int k = 0; k < kMatchPerThread; ++k) {
                const int64_t j = base + k * kMatchThreads + threadIdx.x;
                if (j >= r) continue;
                bool hit = all;
                if (!hit) {
                    const float4 ab = anchors[j];
                    const float aa = box_area(ab);
                    for (int q = 0; q < ns; ++q) {
                        const int g = g0 + c0 + (int)s_list[q];
                        const float4 gb = gt[g];
                        hit |= (pair_iou(gb, box_area(gb), ab, aa) == rowmax[g]);
                    }
                }
                if (hit) labels[(int64_t)img * r + j] = 1;
            }
        }
    }
}

// ---- small anchor sets (r <= 128, e.g. the 98 priors of a 7x7x2 grid head): ONE WARP PER IMAGE, both passes fused.
// Lane l owns anchors l, l+32, l+64, l+96; the image's gt boxes are broadcast loads; the row maximum of a gt is a warp
// reduction, so the low-quality promotion (IoU == row max) is decided in the same iteration -- no workspace, no
// second launch, no block barrier.
constexpr int kSmallMatchWarps = 8;

__global__ void __launch_bounds__(kSmallMatchWarps * 32)
match_small_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, const float4* __restrict__ anchors,
                   int n, int r, MatchRule rule, int64_t* __restrict__ matched, int8_t* __restrict__ labels,
                   float* __restrict__ matched_iou) {
    const int lane = threadIdx.x & 31;
    const int img = blockIdx.x * kSmallMatchWarps + (threadIdx.x >> 5);
    if (img >= n) return;
    float4 ab[4];
    float aa[4], best[4];
    int bidx[4];
    bool valid[4], hit[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int j = lane + 32 * k;
        valid[k] = j < r;
        ab[k] = valid[k] ? anchors[j] : make_float4(0.f, 0.f, 0.f, 0.f);
        aa[k] = box_area(ab[k]);
        best[k] = 0.0f;  // gt 0 wins ties at IoU 0, like torch.max(dim=0)
        bidx[k] = 0;
        hit[k] = false;
    }
    const int g0 = gt_off[img], G = gt_off[img + 1] - g0;
    for (int t = 0; t < G; ++t) {
        const float4 gb = gt[g0 + t];
        const float ga = box_area(gb);
        float v[4], rm = 0.0f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k] = valid[k] ? pair_iou(gb, ga, ab[k], aa[k]) : 0.0f;
            if (v[k] > best[k]) {
                best[k] = v[k];
                bidx[k] = t;
            }
            rm = fmaxf(rm, v[k]);
        }
        if (rule.allow_lq) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, o));
#pragma unroll
            for (int k = 0; k < 4; ++k) hit[k] |= (v[k] == rm);  // matcher.py:110-120 (rm == 0 promotes everything)
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int j = lane + 32 * k;
        if (j >= r) continue;
        const int64_t o = (int64_t)img * r + j;
        if (G == 0) {  // matcher.py:67-77: no gt -> match 0, label labels[0]
            matched[o] = 0;
            labels[o] = rule.lab[0];
            if (matched_iou) matched_iou[o] = 0.0f;
        } else {
            matched[o] = bidx[k];
            labels[o] = hit[k] ? (int8_t)1 : bucket_label(rule, best[k]);
            if (matched_iou) matched_iou[o] = best[k];
        }
    }
}

// ---- Matcher on a materialised (g, r) quality matrix ------------------------------------------------------------
__global__ void __launch_bounds__(256)
quality_pass1_kernel(const float* __restrict__ q, int64_t g, int64_t r, MatchRule rule, int64_t* __restrict__ matched,
                     int8_t* __restrict__ labels, float* __restrict__ rowmax, int32_t* __restrict__ negative_flag) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    float best = 0.f;
    int bi = 0;
    bool bad = false;
    for (int64_t i = 0; i < g; ++i) {
        const float v = (j < r) ? q[i * r + j] : 0.0f;
        bad |= !(v >= 0.0f);
        // torch.max(dim=0): first maximum wins, NaN propagates (excluded by the >= 0 assertion)
        if (i == 0 || v > best) {
            best = v;
            bi = (int)i;
        }
        if (rule.allow_lq) {
            float m = (j < r) ? v : 0.0f;
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (lane == 0 && m > 0.0f) atomic_max_nonneg(&rowmax[i], m);
        }
    }
    if (bad && negative_flag) *negative_flag = 1;
    if (j < r) {
        matched[j] = bi;
        labels[j] = bucket_label(rule, best);
    }
}

__global__ void __launch_bounds__(256)
quality_pass2_kernel(const float* __restrict__ q, int64_t g, int64_t r, const float* __restrict__ rowmax,
                     int8_t* __restrict__ labels) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= r) return;
    bool hit = false;
    for (int64_t i = 0; i < g; ++i) hit |= (q[i * r + j] == rowmax[i]);
    if (hit) labels[j] = 1;
}

// ---- uniform random fg/bg subsample, one CTA per image -----------------------------------------------------------
// Every anchor gets the 32-bit key mix32(j * odd + image_seed) -- a bijection of j, so keys of one image never tie --
// and the class keeps its `want` smallest keys: a uniformly random subset, reproducible from (seed, image, anchor).
// The want-th smallest key is found without sorting the ~50k negatives: a first pass keeps only the keys under a
// threshold that lets about want + 4 sqrt(want) + 16 of them through (a few hundred), the exact order statistic is
// taken among those by rank counting, and a last pass rewrites the labels.  If the threshold pass comes back with too
// few or too many candidates (a > 4-sigma event) the CTA falls back to an exact 4 x 8-bit radix select.
constexpr int kSampleThreads = 512;
constexpr int kCandCap = 1024;

struct SampleSmem {
    int cnt[2];
    int ncand[2];
    int walk_total, walk_warp[kSampleThreads / 32];
    unsigned sel[2];      // the want-th smallest key of the class: keys <= sel are kept
    unsigned prefix[2];   // radix-select fallback state
    int remaining[2];
    int hist[2][256];
    unsigned ckey[2][kCandCap];
    int cidx[2][kCandCap];  // anchor index of the candidate | its original label in the top byte
};

// class c of one image sampled by walking a pseudo-random permutation of the row (block-wide, all threads call it):
// the first `want` hits, in walk order, land in sm.cidx[c][0..want) with key 0
__device__ __forceinline__ void walk_class(SampleSmem& sm, const RowView& rv, int c, int want, uint32_t img_seed, int pbits) {
    const int tid = threadIdx.x;
    const int64_t r = rv.r;
    const uint32_t s0 = mix32(img_seed + 0x51ED270Bu * (uint32_t)(c + 1));
    const int lane = tid & 31, wid = tid >> 5;
    int total = 0;  // accepted so far (block-uniform)
    for (uint32_t k0 = 0; total < want && k0 < (1u << pbits); k0 += kSampleThreads) {
        const uint32_t j = perm_bits(k0 + (uint32_t)tid, s0, pbits);
        int8_t l = -1;
        bool ok = false;
        if ((int64_t)j < r) {
            l = rv.row[j];
            ok = label_class(l) == c;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) sm.walk_warp[wid] = __popc(bal);
        __syncthreads();
        int before = 0, round_total = 0;
        for (int w = 0; w < kSampleThreads / 32; ++w) {
            const int v = sm.walk_warp[w];
            before += (w < wid) ? v : 0;
            round_total += v;
        }
        const int slot = total + before + __popc(bal & ((1u << lane) - 1u));  // rank in walk order
        if (ok && slot < want) {
            sm.ckey[c][slot] = 0u;
            sm.cidx[c][slot] = (int)j | ((int)(uint8_t)l << 24);
        }
        total += round_total;
        __syncthreads();
    }
    if (tid == 0) {
        sm.ncand[c] = want;
        sm.sel[c] = 0u;  // every listed candidate (key 0) is restored after the wholesale wipe
    }
}

// one image of det_subsample_labels (block-wide; every thread of the CTA calls it)
__device__ void subsample_image(SampleSmem& sm, int8_t* __restrict__ labels, int img, int64_t r, int num_samples, int pos_cap,
                                uint64_t seed) {
    const int tid = threadIdx.x;
    const RowView rv(labels + (int64_t)img * r, r);
    const uint32_t img_seed = image_seed(seed, img);
    if (tid < 2) {
        sm.cnt[tid] = 0;
        sm.ncand[tid] = 0;
    }
    __syncthreads();
    // ---- pass A: class counts, 4 labels per SIMD-in-word compare
    int c_bg = 0, c_ign = 0, c_all = 0;
    for (int c = tid; c < rv.ngran; c += kSampleThreads) {
        const uint4 q = rv.load(c);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            c_bg += __popc(bytes_eq(w[k], 0u));
            c_ign += __popc(bytes_eq(w[k], 0xffffffffu));
        }
        c_all += 16;
    }
    int c1 = warp_sum(c_bg) >> 3;                          // popc counts 8 bits per matching byte
    int c0 = warp_sum(c_all) - c1 - (warp_sum(c_ign) >> 3);  // bytes outside the row read as -1 (ignored)
    if ((tid & 31) == 0) {
        if (c0) atomicAdd(&sm.cnt[0], c0);
        if (c1) atomicAdd(&sm.cnt[1], c1);
    }
    __syncthreads();
    const int npos = sm.cnt[0], nneg = sm.cnt[1];
    // utils.py:63-69: num_pos = min(#pos, int(S*f)); num_neg = min(#neg, S - num_pos); pos_cap = int(S*f) is evaluated
    // on the host in double like the reference's Python expression (100 * 0.29 -> 28, not fp32's 29)
    const int want_pos = min(npos, pos_cap);
    const int want_neg = min(nneg, num_samples - want_pos);
    const int want[2] = {want_pos, want_neg};
    const int have[2] = {npos, nneg};
    const bool need[2] = {want_pos < npos, want_neg < nneg};  // otherwise the whole class is kept
    if (!need[0] && !need[1]) return;
    // ---- pass B: hash every label of a thinned class once; keep (key, index, label) of those under a threshold sized
    //      for want + slack survivors
    unsigned thr[2];
    bool direct[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const float slack = 4.0f * sqrtf((float)want[c]) + 16.0f;
        const double p = ((double)want[c] + (double)slack) / (double)max(have[c], 1);
        thr[c] = p >= 1.0 ? 0xffffffffu : (unsigned)(p * 4294967296.0);
        direct[c] = need[c] && want[c] > 0 && (double)want[c] + 2.0 * slack <= (double)kCandCap && r < (1 << 24);
    }
    // The background class is sampled by walking a random permutation of the row instead of hashing every anchor (it is
    // the dense class of every workload on this path: O(want / density) steps; a sparse one just takes up to one full
    // cycle, which is what hashing the row costs).  The rule is fixed per CLASS, not per density, so that the samplers
    // that never see the whole row -- subsample_stats_kernel, subsample_lazy_kernel -- draw the very same samples:
    // positives always by their hash keys, negatives always by the walk.
    bool walk[2];
    int pbits = 1;
    while ((1ll << pbits) < r) ++pbits;
    walk[0] = false;
    walk[1] = need[1] && want[1] > 0 && want[1] <= kCandCap && r < (1 << 24);
    if (walk[1]) direct[1] = false;
    if (direct[0] || direct[1]) {
        for (int c = tid; c < rv.ngran; c += kSampleThreads) {
            const uint4 q = rv.load(c);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
            const int64_t j0 = rv.first(c);
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int8_t l = (int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xffu);
                const int cls = label_class(l);
                if (cls < 0 || !direct[cls]) continue;
                const unsigned key = sample_key(img_seed, (uint32_t)(j0 + k));
                if (key <= thr[cls]) {
                    const int slot = atomicAdd(&sm.ncand[cls], 1);
                    if (slot < kCandCap) {
                        sm.ckey[cls][slot] = key;
                        sm.cidx[cls][slot] = (int)(j0 + k) | ((int)(uint8_t)l << 24);
                    }
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 2; ++c)
        if (walk[c]) walk_class(sm, rv, c, want[c], img_seed, pbits);
    __syncthreads();
    // ---- pass C: the want-th smallest key, by rank counting among the candidates
    bool radix[2], listed[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const int nc = sm.ncand[c];
        listed[c] = walk[c] || (direct[c] && nc >= want[c] && nc <= kCandCap);
        radix[c] = need[c] && want[c] > 0 && !listed[c];
        if (listed[c] && !walk[c]) {
            for (int t = tid; t < nc; t += kSampleThreads) {
                const unsigned key = sm.ckey[c][t];
                int rank = 0;
                for (int q = 0; q < nc; ++q) rank += sm.ckey[c][q] < key;
                if (rank == want[c] - 1) sm.sel[c] = key;
            }
        }
    }
    if (radix[0] || radix[1]) {  // exact fallback: 4 x 8-bit radix select of the want-th smallest key
        if (tid < 2) {
            sm.prefix[tid] = 0;
            sm.remaining[tid] = want[tid];
        }
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            __syncthreads();
            for (int t = tid; t < 512; t += kSampleThreads) (&sm.hist[0][0])[t] = 0;
            __syncthreads();
            const unsigned pre[2] = {sm.prefix[0], sm.prefix[1]};
            const unsigned himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
            for (int c = tid; c < rv.ngran; c += kSampleThreads) {
                const uint4 q = rv.load(c);
                const uint32_t w[4] = {q.x, q.y, q.z, q.w};
                const int64_t j0 = rv.first(c);
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const int cls = label_class((int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xffu));
                    if (cls < 0 || !radix[cls]) continue;
                    const unsigned key = sample_key(img_seed, (uint32_t)(j0 + k));
                    if ((key & himask) == (pre[cls] & himask)) atomicAdd(&sm.hist[cls][(key >> shift) & 255], 1);
                }
            }
            __syncthreads();
            if (tid < 2 && radix[tid]) {
                int rem = sm.remaining[tid], b = 0;
                while (b < 255 && rem > sm.hist[tid][b]) {
                    rem -= sm.hist[tid][b];
                    ++b;
                }
                sm.remaining[tid] = rem;
                sm.prefix[tid] |= (unsigned)b << shift;
            }
        }
        __syncthreads();
        if (tid < 2 && radix[tid]) sm.sel[tid] = sm.prefix[tid];
    }
    __syncthreads();
    // ---- pass D: a thinned class becomes -1 wholesale (SIMD-in-word, no hashing), except that a class that went through
    //      the radix fallback is decided label by label; then the kept candidates of the listed classes are restored
    const unsigned sel[2] = {sm.sel[0], sm.sel[1]};
    for (int c = tid; c < rv.ngran; c += kSampleThreads) {
        const uint4 q = rv.load(c);
        uint32_t w[4] = {q.x, q.y, q.z, q.w};
        bool changed = false;
        if (!radix[0] && !radix[1]) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t bg = bytes_eq(w[k], 0u), ign = bytes_eq(w[k], 0xffffffffu);
                uint32_t kill = 0u;
                if (need[1]) kill |= bg;            // background bytes -> 0xff
                if (need[0]) kill |= ~(bg | ign);   // positive bytes -> 0xff
                changed |= (kill & ~ign) != 0u;
                w[k] |= kill;
            }
        } else {
            const int64_t j0 = rv.first(c);
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int8_t l = (int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xffu);
                const int cls = label_class(l);
                if (cls < 0 || !need[cls]) continue;
                // listed classes are wiped here and restored below; radix classes are decided by their key
                const bool keep = radix[cls] && want[cls] > 0 && sample_key(img_seed, (uint32_t)(j0 + k)) <= sel[cls];
                if (!keep) {
                    w[k >> 2] |= 0xffu << (8 * (k & 3));
                    changed = true;
                }
            }
        }
        if (changed) rv.store(c, make_uint4(w[0], w[1], w[2], w[3]));
    }
    __syncthreads();  // the wipe is complete (this CTA owns the whole row) before the survivors are written back
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        if (!listed[c]) continue;
        const int nc = sm.ncand[c];
        for (int t = tid; t < nc; t += kSampleThreads)
            if (sm.ckey[c][t] <= sel[c]) {
                const int packed = sm.cidx[c][t];
                rv.row[packed & 0xffffff] = (int8_t)(packed >> 24);
            }
    }
}

__global__ void __launch_bounds__(kSampleThreads)
subsample_kernel(int8_t* __restrict__ labels, int64_t r, int num_samples, int pos_cap, uint64_t seed) {
    __shared__ SampleSmem sm;
    subsample_image(sm, labels, blockIdx.x, r, num_samples, pos_cap, seed);
}

// The same subsample driven by what det_match_grid already knows about the image -- #positives, #ignored and the list of
// positives -- so that the label row is never read in full: positives are ranked by their hash keys straight from the
// list, negatives are found by the permutation walk (O(wanted) random reads), the row is overwritten with -1 (a pure
// streaming store) and the <= num_samples survivors are written back.  Identical result to det_subsample_labels (same
// keys, same walk); images outside the fast path's preconditions take that kernel's code.  Also emits the image's sample
// list (anchor row | label << 24) for the sampled loss.
__global__ void __launch_bounds__(kSampleThreads)
subsample_stats_kernel(int8_t* __restrict__ labels, int64_t r, int num_samples, int pos_cap, uint64_t seed,
                       const int32_t* __restrict__ stats, const int32_t* __restrict__ pos_list, int list_cap,
                       int32_t* __restrict__ samples, int32_t* __restrict__ sample_count, int sample_cap) {
    __shared__ SampleSmem sm;
    __shared__ int s_nout;
    const int img = blockIdx.x, tid = threadIdx.x;
    const int npos = stats[img * 4 + 0], nign = stats[img * 4 + 1];
    const int64_t nneg64 = r - npos - nign;
    const int nneg = (int)nneg64;
    const int want_pos = min(npos, pos_cap);
    const int want_neg = min(nneg, num_samples - want_pos);
    int8_t* row = labels + (int64_t)img * r;
    const bool fast = r < (1 << 24) && npos <= min(list_cap, kCandCap) &&  // the positives are all on the list
                      want_neg < nneg && want_neg <= kCandCap;             // thinned negatives (same rule as subsample_image)
    if (tid == 0) s_nout = 0;
    if (!fast) {
        subsample_image(sm, labels, img, r, num_samples, pos_cap, seed);
        __syncthreads();
        if (samples) {  // rare: rebuild the list from the finished row
            for (int64_t j = tid; j < r; j += kSampleThreads) {
                const int8_t l = row[j];
                if (l != -1) {
                    const int slot = atomicAdd(&s_nout, 1);
                    if (slot < sample_cap) samples[(int64_t)img * sample_cap + slot] = (int)j | ((int)(uint8_t)l << 24);
                }
            }
            __syncthreads();
            if (tid == 0) sample_count[img] = min(s_nout, sample_cap);
        }
        return;
    }
    const RowView rv(row, r);
    const uint32_t img_seed = image_seed(seed, img);
    int pbits = 1;
    while ((1ll << pbits) < r) ++pbits;
    // positives: the want_pos smallest keys of the list (keys are a bijection of the anchor index: no ties)
    for (int t = tid; t < npos; t += kSampleThreads) {
        const int packed = pos_list[(int64_t)img * list_cap + t];
        sm.cidx[0][t] = packed;
        sm.ckey[0][t] = sample_key(img_seed, (uint32_t)(packed & 0xffffff));
    }
    __syncthreads();
    if (want_pos < npos) {
        for (int t = tid; t < npos; t += kSampleThreads) {
            const unsigned key = sm.ckey[0][t];
            int rank = 0;
            for (int q = 0; q < npos; ++q) rank += sm.ckey[0][q] < key;
            if (rank >= want_pos) sm.cidx[0][t] = -1;  // dropped
        }
    }
    if (want_neg > 0) walk_class(sm, rv, 1, want_neg, img_seed, pbits);  // has block barriers inside
    __syncthreads();
    // the row becomes -1 wholesale ...
    const uint4 ones = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    for (int c = tid; c < rv.ngran; c += kSampleThreads) rv.store(c, ones);
    __syncthreads();
    // ... and the survivors come back
    for (int t = tid; t < npos; t += kSampleThreads) {
        const int packed = sm.cidx[0][t];
        if (packed == -1) continue;
        row[packed & 0xffffff] = (int8_t)(packed >> 24);
        if (samples) {
            const int slot = atomicAdd(&s_nout, 1);
            if (slot < sample_cap) samples[(int64_t)img * sample_cap + slot] = packed;
        }
    }
    __syncthreads();
    const int kept_pos = s_nout;
    for (int t = tid; t < want_neg; t += kSampleThreads) {
        const int packed = sm.cidx[1][t];
        row[packed & 0xffffff] = (int8_t)(packed >> 24);
        if (samples && kept_pos + t < sample_cap) samples[(int64_t)img * sample_cap + kept_pos + t] = packed;
    }
    if (samples && tid == 0) sample_count[img] = min(samples ? kept_pos + want_neg : 0, sample_cap);
}

// ---- fused RPN loss forward + backward ---------------------------------------------------------------------------
// The sampler of the sample-list-only assignment (assign_grid.cu): nothing dense exists for the image.  Positives come from
// assign_candidates_kernel's list (ranked by their hash keys when there are too many, exactly like the other samplers);
// negatives are found by the same permutation walk, each visited anchor labelled on the fly by anchor_verdict() -- the
// walk accepts the first `want` anchors whose label is 0 and simply ends after a full cycle if the image has fewer, which
// is min(#neg, S - #pos) without ever counting the negatives.  Output: the sample list (anchor row | label << 24), the
// matched gt of every sample and the count.  Images whose positives are dense (a gt with row maximum 0 promotes every
// anchor; list overflow) are labelled in full into `scratch` (n, r) int8 and go through subsample_image().
__global__ void __launch_bounds__(kSampleThreads)
subsample_lazy_kernel(const float4* __restrict__ gt, const int32_t* __restrict__ gt_off, const float4* __restrict__ anchors,
                      int64_t r, MatchRule rule, float tau, const float* __restrict__ rowmax,
                      const int32_t* __restrict__ flags, const int32_t* __restrict__ stats,
                      const int32_t* __restrict__ pos_list, const int32_t* __restrict__ pos_gt, int list_cap,
                      int num_samples, int pos_cap, uint64_t seed, int8_t* __restrict__ scratch,
                      int32_t* __restrict__ samples, int32_t* __restrict__ sample_gt, int32_t* __restrict__ sample_count,
                      int sample_cap) {
    __shared__ SampleSmem sm;
    __shared__ int s_nout;
    const int img = blockIdx.x, tid = threadIdx.x;
    const int g0 = gt_off[img], G = gt_off[img + 1] - g0;
    const bool lq = rule.allow_lq != 0;
    const int npos = stats[img * 4 + 0];
    const bool dense = (lq && (flags[img] & 1)) || npos > min(list_cap, kCandCap) || r >= (1 << 24) ||
                       num_samples > kCandCap;  // (more samples than the walk's buffer: subsample_image's exact paths)
    if (tid == 0) s_nout = 0;
    __syncthreads();
    if (dense) {
        int8_t* row = scratch + (int64_t)img * r;
        for (int64_t j = tid; j < r; j += kSampleThreads) {
            const Verdict v = anchor_verdict(anchors[j], gt, rowmax, g0, G, tau, lq);
            row[j] = (int8_t)((lq && (flags[img] & 1) && G > 0) ? 1 : verdict_label(rule, v, G));
        }
        __syncthreads();
        subsample_image(sm, scratch, img, r, num_samples, pos_cap, seed);
        __syncthreads();
        for (int64_t j = tid; j < r; j += kSampleThreads) {
            const int8_t l = row[j];
            if (l == -1) continue;
            const int slot = atomicAdd(&s_nout, 1);
            if (slot < sample_cap) {
                samples[(int64_t)img * sample_cap + slot] = (int)j | ((int)(uint8_t)l << 24);
                sample_gt[(int64_t)img * sample_cap + slot] =
                    (l == 0) ? 0 : anchor_verdict(anchors[j], gt, rowmax, g0, G, tau, lq).argmax;
            }
        }
        __syncthreads();
        if (tid == 0) sample_count[img] = min(s_nout, sample_cap);
        return;
    }
    const uint32_t img_seed = image_seed(seed, img);
    int pbits = 1;
    while ((1ll << pbits) < r) ++pbits;
    const int want_pos = min(npos, pos_cap);
    const int want_neg_max = num_samples - want_pos;  // min(#neg, .) falls out of the walk
    // positives: the want_pos smallest keys of the list (keys are a bijection of the anchor index: no ties)
    for (int t = tid; t < npos; t += kSampleThreads) {
        const int packed = pos_list[(int64_t)img * list_cap + t];
        sm.cidx[0][t] = packed;
        sm.ckey[0][t] = sample_key(img_seed, (uint32_t)(packed & 0xffffff));
    }
    __syncthreads();
    for (int t = tid; t < npos; t += kSampleThreads) {
        bool keep = true;
        if (want_pos < npos) {
            const unsigned key = sm.ckey[0][t];
            int rank = 0;
            for (int q = 0; q < npos; ++q) rank += sm.ckey[0][q] < key;
            keep = rank < want_pos;
        }
        if (keep) {
            const int slot = atomicAdd(&s_nout, 1);
            if (slot < sample_cap) {
                samples[(int64_t)img * sample_cap + slot] = sm.cidx[0][t];
                sample_gt[(int64_t)img * sample_cap + slot] = pos_gt[(int64_t)img * list_cap + t];
            }
        }
    }
    __syncthreads();
    const int kept_pos = s_nout;
    // negatives: walk_class() with the label evaluated on the fly (same permutation, same acceptance order)
    const int want = min(want_neg_max, kCandCap);
    int total = 0;
    if (want > 0) {
        const uint32_t s0 = mix32(img_seed + 0x51ED270Bu * 2u);
        const int lane = tid & 31, wid = tid >> 5;
        for (uint32_t k0 = 0; total < want && k0 < (1u << pbits); k0 += kSampleThreads) {
            const uint32_t j = perm_bits(k0 + (uint32_t)tid, s0, pbits);
            bool ok = false;
            if ((int64_t)j < r)
                ok = verdict_label(rule, anchor_verdict(anchors[j], gt, rowmax, g0, G, tau, lq), G) == 0;
            const unsigned bal = __ballot_sync(0xffffffffu, ok);
            if (lane == 0) sm.walk_warp[wid] = __popc(bal);
            __syncthreads();
            int before = 0, round_total = 0;
            for (int w = 0; w < kSampleThreads / 32; ++w) {
                const int v = sm.walk_warp[w];
                before += (w < wid) ? v : 0;
                round_total += v;
            }
            const int slot = total + before + __popc(bal & ((1u << lane) - 1u));  // rank in walk order
            if (ok && slot < want && kept_pos + slot < sample_cap) {
                samples[(int64_t)img * sample_cap + kept_pos + slot] = (int)j;  // label 0
                sample_gt[(int64_t)img * sample_cap + kept_pos + slot] = 0;
            }
            total += round_total;
            __syncthreads();
        }
    }
    if (tid == 0) sample_count[img] = min(kept_pos + min(total, want), sample_cap);
}

constexpr int kLossThreads = 256;

template <bool GIOU>
__global__ void __launch_bounds__(kLossThreads)
rpn_loss_kernel(const float* __restrict__ logits, const float4* __restrict__ deltas, const int8_t* __restrict__ labels,
                const int64_t* __restrict__ matched, const float4* __restrict__ gt, const int32_t* __restrict__ gt_off,
                const float4* __restrict__ anchors, int64_t total, int64_t r, CodecWeights wt, float scale_clamp,
                float beta, float gs_cls,
                float gs_loc, const float* __restrict__ upstream, float* __restrict__ acc, float* __restrict__ sums_out,
                float* __restrict__ grad_logits, float4* __restrict__ grad_deltas) {
    __shared__ float s_part[4][kLossThreads / 32];
    __shared__ float s_fin[8];
    const float scale_cls = gs_cls, scale_loc = gs_loc;  // the reported losses are not multiplied by the upstream gradient
    if (upstream) {
        gs_cls *= upstream[0];
        gs_loc *= upstream[1];
    }
    float acc_cls = 0.f, acc_loc = 0.f;
    int npos = 0, nneg = 0;
    // A warp owns 128 consecutive anchors per iteration.  Labels arrive as one 32-bit word per lane (4 anchors, one
    // coalesced 128-byte load) and are re-dealt with shuffles so that in each of the 4 rounds lane l works on anchor
    // base + 32*round + l: every gradient store of a warp is then one contiguous 128-byte (logits) or 512-byte
    // (deltas) run of full sectors.
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * kLossThreads + threadIdx.x) >> 5;
    const int64_t warps_total = ((int64_t)gridDim.x * kLossThreads) >> 5;
    auto load_word = [&](int64_t base) -> uint32_t {  // labels base + 4*lane .. +3 (label -1 = ignored past the end)
        const int64_t e4 = base + 4 * lane;
        if (e4 + 4 <= total) return __ldcs(reinterpret_cast<const unsigned int*>(labels + e4));
        uint32_t word = 0xffffffffu;
        for (int k = 0; k < 4; ++k)
            if (e4 + k < total) word = (word & ~(0xffu << (8 * k))) | ((uint32_t)(uint8_t)labels[e4 + k] << (8 * k));
        return word;
    };
    const int64_t step = warps_total * 128;
    uint32_t word_next = warp_global * 128 < total ? load_word(warp_global * 128) : 0xffffffffu;
    for (int64_t base = warp_global * 128; base < total; base += step) {
        const uint32_t word = word_next;
        if (base + step < total) word_next = load_word(base + step);  // in flight while this block's stores are issued
#pragma unroll
        for (int round = 0; round < 4; ++round) {
            const uint32_t w = __shfl_sync(0xffffffffu, word, 8 * round + (lane >> 2));
            const int lab = (int)(int8_t)((w >> (8 * (lane & 3))) & 0xffu);
            const int64_t e = base + 32 * round + lane;
            if (e >= total) continue;
            float gl = 0.f;
            if (lab >= 0) {
                const float x = logits[e];
                const float y = (float)lab;
                // BCE with logits: (1-y)*x - log_sigmoid(x), log_sigmoid(x) = min(x,0) - log1p(exp(-|x|))
                const float ls = fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
                acc_cls += (1.f - y) * x - ls;
                gl = (1.f / (1.f + expf(-x)) - y) * gs_cls;
                npos += lab == 1;
                nneg += lab == 0;
            }
            if (grad_logits) st_stream(grad_logits + e, gl);
            float4 gd = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lab == 1) {
                const int64_t img = e / r, j = e - img * r;
                const float4 g = gt[gt_off[img] + matched[e]];
                const float4 p = deltas[e];
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
            }
            if (grad_deltas) st_stream(grad_deltas + e, gd);
        }
    }
    // warp-shuffle + shared-memory reduction, one atomic per CTA and quantity
    acc_cls = warp_sum(acc_cls);
    acc_loc = warp_sum(acc_loc);
    float fpos = warp_sum((float)npos), fneg = warp_sum((float)nneg);
    const int wid = threadIdx.x >> 5;
    if (lane == 0) {
        s_part[0][wid] = acc_cls;
        s_part[1][wid] = acc_loc;
        s_part[2][wid] = fpos;
        s_part[3][wid] = fneg;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        float t = 0.f;
        for (int w = 0; w < kLossThreads / 32; ++w) t += s_part[threadIdx.x][w];
        if (t != 0.f) atomicAdd(&acc[threadIdx.x], t);
    }
    // the last CTA turns the accumulators into the weighted, normalised losses (rpn.py:238-243) and re-arms them
    if (last_cta_arrives(reinterpret_cast<int32_t*>(acc + 8)))
        finalize_sums(acc, sums_out, s_fin, [&](int i) { return i == 0 ? scale_cls : (i == 1 ? scale_loc : 1.0f); });
}

// ---- fused YOLO-grid loss forward + backward: one thread per (image, cell) -----------------------------------------
struct YoloLossParams {
    int n, s, b, c;
    float stride_x, stride_y, lambda_coord, lambda_noobj, grad_scale;
};

// per (image, cell): loss terms and gradients, reading `t` (ch logits of the cell) and writing `g` (same layout) or not
__device__ __forceinline__ void yolo_cell_loss(const float* t, float* g, int img, int cell, const int8_t* __restrict__ labels,
                                               const int64_t* __restrict__ matched, const float4* __restrict__ gt,
                                               const int64_t* __restrict__ gt_cls, const int32_t* __restrict__ gt_off,
                                               const float2* __restrict__ priors, const YoloLossParams& prm, float up_loc,
                                               float up_obj, float up_cls, float (&acc)[5]) {
    const int S2 = prm.s * prm.s, B = prm.b, C = prm.c;
    const int row = cell / prm.s, col = cell - row * prm.s;
    if (g)
        for (int k = 0; k < C; ++k) g[B * 5 + k] = 0.f;
    for (int bi = 0; bi < B; ++bi) {
        const int64_t p = (int64_t)img * S2 * B + (int64_t)cell * B + bi;
        const int8_t lab = labels[p];
        float gx = 0.f, gy = 0.f, gw = 0.f, gh = 0.f, gc = 0.f;
        const float tc = t[bi * 5 + 4];
        if (lab >= 0) {
            const float y = (float)lab;
            const float wgt = (lab == 1) ? 1.0f : prm.lambda_noobj;
            const float ls = fminf(tc, 0.f) - log1pf(expf(-fabsf(tc)));
            acc[1] += wgt * ((1.f - y) * tc - ls);
            gc = wgt * (1.f / (1.f + expf(-tc)) - y) * prm.grad_scale * up_obj;
            acc[3] += lab == 1;
            acc[4] += lab == 0;
        }
        if (lab == 1) {
            const int64_t gi = gt_off[img] + matched[p];
            const float4 gb = gt[gi];
            const float2 pr = priors[bi];
            const float bw = gb.z - gb.x, bh = gb.w - gb.y;
            const float xs = (gb.x + 0.5f * bw) / prm.stride_x - (float)col;
            const float ys = (gb.y + 0.5f * bh) / prm.stride_y - (float)row;
            const float tws = logf(bw / pr.x), ths = logf(bh / pr.y);
            const float sx = 1.f / (1.f + expf(-t[bi * 5 + 0])), sy = 1.f / (1.f + expf(-t[bi * 5 + 1]));
            const float dx = sx - xs, dy = sy - ys, dw = t[bi * 5 + 2] - tws, dh = t[bi * 5 + 3] - ths;
            acc[0] += dx * dx + dy * dy + dw * dw + dh * dh;
            const float k2 = 2.0f * prm.lambda_coord * prm.grad_scale * up_loc;
            gx = k2 * dx * sx * (1.f - sx);
            gy = k2 * dy * sy * (1.f - sy);
            gw = k2 * dw;
            gh = k2 * dh;
            const int64_t cls = gt_cls[gi];
            for (int k = 0; k < C; ++k) {
                const float x = t[B * 5 + k];
                const float y = (k == cls) ? 1.f : 0.f;
                const float ls = fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
                acc[2] += (1.f - y) * x - ls;
                if (g) g[B * 5 + k] += (1.f / (1.f + expf(-x)) - y) * prm.grad_scale * up_cls;
            }
        }
        if (g) {
            g[bi * 5 + 0] = gx; g[bi * 5 + 1] = gy; g[bi * 5 + 2] = gw; g[bi * 5 + 3] = gh; g[bi * 5 + 4] = gc;
        }
    }
}

constexpr int kYoloLossThreads = 256;
constexpr int kYoloLossTile = 5888;  // floats of head staged per CTA (and as many of gradient): 2 x 23 KB

// A CTA stages the logits of `imgs` consecutive images in shared memory with coalesced 16-byte loads, one thread per
// (image, cell) works on its cell there (a cell is 5B+C scattered floats: reading it straight from HBM wastes most of
// every sector), and the gradient tile leaves the same way.
__global__ void __launch_bounds__(kYoloLossThreads)
yolo_loss_kernel(const float* __restrict__ head, const int8_t* __restrict__ labels, const int64_t* __restrict__ matched,
                 const float4* __restrict__ gt, const int64_t* __restrict__ gt_cls, const int32_t* __restrict__ gt_off,
                 const float2* __restrict__ priors, YoloLossParams prm, int imgs, const float* __restrict__ upstream,
                 float* __restrict__ gacc, float* __restrict__ sums_out, float* __restrict__ grad_head,
                 const PeerCtxDev peer) {
    extern __shared__ __align__(16) float s_tile[];
    __shared__ float s_part[5][kYoloLossThreads / 32];
    __shared__ float s_fin[8];
    const float up_loc = upstream ? upstream[0] : 1.f, up_obj = upstream ? upstream[1] : 1.f,
                up_cls = upstream ? upstream[2] : 1.f;
    const int S2 = prm.s * prm.s, ch = prm.b * 5 + prm.c, per_img = S2 * ch;
    const int img0 = blockIdx.x * imgs, ni = min(imgs, prm.n - img0);
    const int count = ni * per_img;
    const int64_t base = (int64_t)img0 * per_img;
    float* s_in = s_tile;
    float* s_out = s_tile + ((imgs * per_img + 3) & ~3);
    const bool vec = ((base & 3) == 0) && ((count & 3) == 0);
    if (vec) {
        for (int i = threadIdx.x; i < (count >> 2); i += kYoloLossThreads)
            reinterpret_cast<float4*>(s_in)[i] = ld_stream(reinterpret_cast<const float4*>(head + base) + i);
    } else {
        for (int i = threadIdx.x; i < count; i += kYoloLossThreads) s_in[i] = head[base + i];
    }
    __syncthreads();
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int ci = threadIdx.x; ci < ni * S2; ci += kYoloLossThreads) {
        const int li = ci / S2, cell = ci - li * S2;
        yolo_cell_loss(s_in + (size_t)ci * ch, grad_head ? s_out + (size_t)ci * ch : nullptr, img0 + li, cell, labels,
                       matched, gt, gt_cls, gt_off, priors, prm, up_loc, up_obj, up_cls, acc);
    }
    if (grad_head) {
        __syncthreads();
        if (vec) {
            for (int i = threadIdx.x; i < (count >> 2); i += kYoloLossThreads)
                st_stream(reinterpret_cast<float4*>(grad_head + base) + i, reinterpret_cast<const float4*>(s_out)[i]);
        } else {
            for (int i = threadIdx.x; i < count; i += kYoloLossThreads) grad_head[base + i] = s_out[i];
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const float v = warp_sum(acc[k]);
        if (lane == 0) s_part[k][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        float t = 0.f;
        for (int w = 0; w < kYoloLossThreads / 32; ++w) t += s_part[threadIdx.x][w];
        if (t != 0.f) atomicAdd(&gacc[threadIdx.x], t);
    }
    // The last CTA scales the accumulators into the reported losses [lambda_coord * loc, obj, cls] * grad_scale (counts
    // unscaled) and re-arms them.  Compute + collective in one kernel: it then publishes that vector into every peer's
    // buffer over NVLink and collects the previous step's world sum (peer.cuh).
    if (last_cta_arrives(reinterpret_cast<int32_t*>(gacc + 8))) {
        const float gs = prm.grad_scale, lc = prm.lambda_coord;
        finalize_sums(gacc, sums_out, s_fin, [&](int i) { return i == 0 ? lc * gs : (i < 3 ? gs : 1.0f); });
        if (peer.enabled) peer_exchange_warp0(peer, s_fin);
    }
}

// heads too large for the shared-memory tile: one thread per (image, cell) straight from global memory
__global__ void __launch_bounds__(128)
yolo_loss_direct_kernel(const float* __restrict__ head, const int8_t* __restrict__ labels,
                        const int64_t* __restrict__ matched, const float4* __restrict__ gt,
                        const int64_t* __restrict__ gt_cls, const int32_t* __restrict__ gt_off,
                        const float2* __restrict__ priors, YoloLossParams prm, const float* __restrict__ upstream,
                        float* __restrict__ gacc, float* __restrict__ sums_out, float* __restrict__ grad_head) {
    __shared__ float s_part[5][4];
    __shared__ float s_fin[8];
    const float up_loc = upstream ? upstream[0] : 1.f, up_obj = upstream ? upstream[1] : 1.f,
                up_cls = upstream ? upstream[2] : 1.f;
    const int S2 = prm.s * prm.s, ch = prm.b * 5 + prm.c;
    const int64_t cells = (int64_t)prm.n * S2;
    const int64_t ci = (int64_t)blockIdx.x * 128 + threadIdx.x;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (ci < cells) {
        const int img = (int)(ci / S2), cell = (int)(ci - (int64_t)img * S2);
        yolo_cell_loss(head + ci * ch, grad_head ? grad_head + ci * ch : nullptr, img, cell, labels, matched, gt, gt_cls,
                       gt_off, priors, prm, up_loc, up_obj, up_cls, acc);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const float v = warp_sum(acc[k]);
        if (lane == 0) s_part[k][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        const float t = s_part[threadIdx.x][0] + s_part[threadIdx.x][1] + s_part[threadIdx.x][2] + s_part[threadIdx.x][3];
        if (t != 0.f) atomicAdd(&gacc[threadIdx.x], t);
    }
    if (last_cta_arrives(reinterpret_cast<int32_t*>(gacc + 8))) {
        const float gs = prm.grad_scale, lc = prm.lambda_coord;
        finalize_sums(gacc, sums_out, s_fin, [&](int i) { return i == 0 ? lc * gs : (i < 3 ? gs : 1.0f); });
    }
}

}  // namespace det

using namespace det;

// second half of det_assign_sampled (assign_grid.cu launches the gt-centric kernels and then calls this)
int launch_subsample_lazy(const float* gt_boxes, const int32_t* gt_offsets, const float* anchors, int n, int64_t r,
                          const MatchRule& rule, float tau, const float* rowmax, const int32_t* flags, const int32_t* stats,
                          const int32_t* pos_list, const int32_t* pos_gt, int list_cap, int num_samples,
                          double positive_fraction, uint64_t seed, int8_t* scratch, int32_t* samples, int32_t* sample_gt,
                          int32_t* sample_count, int sample_cap, cudaStream_t st) {
    const int pos_cap = (int)((double)num_samples * positive_fraction);
    subsample_lazy_kernel<<<n, kSampleThreads, 0, st>>>(
        reinterpret_cast<const float4*>(gt_boxes), gt_offsets, reinterpret_cast<const float4*>(anchors), r, rule, tau, rowmax,
        flags, stats, pos_list, pos_gt, list_cap, num_samples, pos_cap, seed, scratch, samples, sample_gt, sample_count,
        sample_cap);
    DET_LAUNCH_OK("subsample_lazy_kernel");
    return DET_OK;
}

// CTAs per SM of the dense loss kernel's grid-stride launch
constexpr int kLossGridFactor = 16;

extern "C" {

static int64_t match_blocks(int64_t r) { return (r + kMatchThreads * kMatchPerThread - 1) / (kMatchThreads * kMatchPerThread); }

int64_t det_match_workspace_bytes(int n, int64_t r, int64_t sum_g) {
    (void)n;
    // row maxima (sum_g) + per-CTA maxima (blocks x sum_g), fp32
    return ((sum_g > 0 ? sum_g : 1) * (1 + match_blocks(r > 0 ? r : 1)) * 4 + 255) / 256 * 256;
}

int det_match_anchors(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors,
                      int64_t r, const float* thresholds_host, const int32_t* labels_host, int num_thresholds,
                      int allow_low_quality, int64_t* matched_idx, int8_t* labels, float* matched_iou,
                      void* workspace, int64_t workspace_bytes, void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && sum_g >= 0, "negative size");
    if (n == 0 || r == 0) return DET_OK;
    DET_CHECK_ARG(gt_offsets && anchors && matched_idx && labels, "null pointer");
    DET_CHECK_ARG(sum_g == 0 || gt_boxes, "null gt_boxes");
    DET_CHECK_ARG(n <= 65535, "n > 65535");
    if (!aligned16(anchors) || (gt_boxes && !aligned16(gt_boxes))) {
        set_error("gt_boxes/anchors must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    MatchRule rule;
    int rc = fill_rule(rule, thresholds_host, labels_host, num_thresholds, allow_low_quality);
    if (rc != DET_OK) return rc;
    if (r <= 128) {  // one warp per image, both passes fused, no workspace
        match_small_kernel<<<(unsigned)((n + kSmallMatchWarps - 1) / kSmallMatchWarps), kSmallMatchWarps * 32, 0,
                             as_stream(stream)>>>(reinterpret_cast<const float4*>(gt_boxes), gt_offsets,
                                                  reinterpret_cast<const float4*>(anchors), n, (int)r, rule, matched_idx,
                                                  labels, matched_iou);
        DET_LAUNCH_OK("match_small_kernel");
        return DET_OK;
    }
    if (allow_low_quality && sum_g > 0 &&
        (!workspace || workspace_bytes < (int64_t)sizeof(float) * sum_g * (1 + match_blocks(r)))) {
        set_error("workspace too small: need %lld bytes", (long long)det_match_workspace_bytes(n, r, sum_g));
        return DET_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    float* rowmax = static_cast<float*>(workspace);
    if (allow_low_quality && sum_g > 0) {
        cudaError_t e = cudaMemsetAsync(rowmax, 0, sizeof(float) * (size_t)sum_g * (size_t)(1 + match_blocks(r)), st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    }
    // images per CTA: amortise the anchor loads / block box when there are plenty of CTAs, keep one image per CTA when
    // the grid would otherwise not fill the GPU (small anchor sets such as a 7x7 grid head)
    const int64_t bx = match_blocks(r);
    int imgs = (int)((bx * n) / ((int64_t)sm_count() * 16));
    imgs = imgs < 1 ? 1 : (imgs > kMatchImgs ? kMatchImgs : imgs);
    dim3 grid((unsigned)bx, (unsigned)((n + imgs - 1) / imgs));
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto a4 = reinterpret_cast<const float4*>(anchors);
    match_pass1_kernel<<<grid, kMatchThreads, 0, st>>>(g4, gt_offsets, a4, n, imgs, r, sum_g, rule, matched_idx, labels, matched_iou,
                                                       rowmax, rowmax + sum_g);
    DET_LAUNCH_OK("match_pass1_kernel");
    if (allow_low_quality && sum_g > 0) {
        match_pass2_kernel<<<grid, kMatchThreads, 0, st>>>(g4, gt_offsets, a4, n, imgs, r, sum_g, rowmax, rowmax + sum_g, labels);
        DET_LAUNCH_OK("match_pass2_kernel");
    }
    return DET_OK;
}

int det_match_quality(const float* quality, int64_t g, int64_t r, const float* thresholds_host,
                      const int32_t* labels_host, int num_thresholds, int allow_low_quality, int64_t* matched_idx,
                      int8_t* labels, int32_t* negative_flag, void* workspace, int64_t workspace_bytes, void* stream) {
    DET_CHECK_ARG(g >= 0 && r >= 0, "negative size");
    if (r == 0) return DET_OK;
    DET_CHECK_ARG(matched_idx && labels && (quality || g == 0), "null pointer");
    MatchRule rule;
    int rc = fill_rule(rule, thresholds_host, labels_host, num_thresholds, allow_low_quality);
    if (rc != DET_OK) return rc;
    cudaStream_t st = as_stream(stream);
    if (g == 0) {  // matcher.py:67-77
        cudaError_t e = cudaMemsetAsync(matched_idx, 0, sizeof(int64_t) * (size_t)r, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(labels, (int)(uint8_t)rule.lab[0], (size_t)r, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
        return DET_OK;
    }
    float* rowmax = static_cast<float*>(workspace);
    if (allow_low_quality) {
        if (!workspace || workspace_bytes < (int64_t)sizeof(float) * g) {
            set_error("workspace too small: need %lld bytes", (long long)(sizeof(float) * g));
            return DET_ERR_WORKSPACE;
        }
        cudaError_t e = cudaMemsetAsync(rowmax, 0, sizeof(float) * (size_t)g, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    }
    const unsigned blocks = (unsigned)((r + 255) / 256);
    quality_pass1_kernel<<<blocks, 256, 0, st>>>(quality, g, r, rule, matched_idx, labels, rowmax, negative_flag);
    DET_LAUNCH_OK("quality_pass1_kernel");
    if (allow_low_quality) {
        quality_pass2_kernel<<<blocks, 256, 0, st>>>(quality, g, r, rowmax, labels);
        DET_LAUNCH_OK("quality_pass2_kernel");
    }
    return DET_OK;
}

int det_subsample_labels(int8_t* labels, int n, int64_t r, int num_samples, double positive_fraction, uint64_t seed,
                         void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && num_samples >= 0, "negative size");
    DET_CHECK_ARG(positive_fraction >= 0.0 && positive_fraction <= 1.0, "positive_fraction outside [0, 1]");
    const int pos_cap = (int)((double)num_samples * positive_fraction);  // Python: int(num_samples * positive_fraction)
    DET_CHECK_ARG(r < (1ll << 31), "r too large");
    if (n == 0 || r == 0) return DET_OK;
    DET_CHECK_ARG(labels, "null pointer");
    subsample_kernel<<<n, kSampleThreads, 0, as_stream(stream)>>>(labels, r, num_samples, pos_cap, seed);
    DET_LAUNCH_OK("subsample_kernel");
    return DET_OK;
}

int det_subsample_labels_grid(int8_t* labels, int n, int64_t r, int num_samples, double positive_fraction, uint64_t seed,
                              const int32_t* stats, const int32_t* pos_list, int list_cap, int32_t* samples,
                              int32_t* sample_count, int sample_cap, void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && num_samples >= 0, "negative size");
    DET_CHECK_ARG(r < (1ll << 31), "r too large");
    DET_CHECK_ARG(positive_fraction >= 0.0 && positive_fraction <= 1.0, "positive_fraction outside [0, 1]");
    if (n == 0 || r == 0) return DET_OK;
    DET_CHECK_ARG(labels && stats && pos_list && list_cap >= 1, "null pointer");
    DET_CHECK_ARG((samples == nullptr) == (sample_count == nullptr) && (!samples || sample_cap >= 1), "bad sample list");
    DET_CHECK_ARG(!samples || r < (1 << 24), "sample lists pack the anchor row in 24 bits");
    const int pos_cap = (int)((double)num_samples * positive_fraction);
    subsample_stats_kernel<<<n, kSampleThreads, 0, as_stream(stream)>>>(labels, r, num_samples, pos_cap, seed, stats, pos_list,
                                                                        list_cap, samples, sample_count, sample_cap);
    DET_LAUNCH_OK("subsample_stats_kernel");
    return DET_OK;
}

int det_rpn_loss(const float* logits, const float* deltas, const int8_t* labels, const int64_t* matched_idx,
                 const float* gt_boxes, const int32_t* gt_offsets, const float* anchors, int n, int64_t r, float wx,
                 float wy, float ww, float wh, float scale_clamp, int loss_type, float smooth_l1_beta,
                 float grad_scale_cls, float grad_scale_loc, const float* upstream, float* accumulators, float* sums_out,
                 float* grad_logits, float* grad_deltas, void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0, "negative size");
    DET_CHECK_ARG(loss_type == 0 || loss_type == 1, "loss_type must be 0 (smooth-L1) or 1 (GIoU)");
    DET_CHECK_ARG(accumulators && sums_out, "null accumulators / sums_out");
    if (n == 0 || r == 0) {
        cudaError_t e = cudaMemsetAsync(sums_out, 0, 8 * sizeof(float), as_stream(stream));
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
        return DET_OK;
    }
    DET_CHECK_ARG(logits && deltas && labels && matched_idx && gt_offsets && anchors, "null pointer");
    if (!aligned16(deltas) || !aligned16(anchors) || !aligned16(logits) || (gt_boxes && !aligned16(gt_boxes)) ||
        (grad_logits && !aligned16(grad_logits)) || (grad_deltas && !aligned16(grad_deltas)) ||
        (reinterpret_cast<uintptr_t>(labels) & 3u)) {
        set_error("tensors must be 16-byte aligned (labels 4-byte)");
        return DET_ERR_ALIGN;
    }
    const int64_t total = (int64_t)n * r;
    const int64_t nwarps = (total + 127) / 128;
    int64_t blocks = (nwarps + kLossThreads / 32 - 1) / (kLossThreads / 32);
    const int64_t cap = (int64_t)sm_count() * kLossGridFactor;
    if (blocks > cap) blocks = cap;
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto a4 = reinterpret_cast<const float4*>(anchors);
    auto d4 = reinterpret_cast<const float4*>(deltas);
    auto gd4 = reinterpret_cast<float4*>(grad_deltas);
    const CodecWeights wt{wx, wy, ww, wh};
    if (loss_type == 1)
        rpn_loss_kernel<true><<<(unsigned)blocks, kLossThreads, 0, as_stream(stream)>>>(
            logits, d4, labels, matched_idx, g4, gt_offsets, a4, total, r, wt, scale_clamp, smooth_l1_beta, grad_scale_cls,
            grad_scale_loc, upstream, accumulators, sums_out, grad_logits, gd4);
    else
        rpn_loss_kernel<false><<<(unsigned)blocks, kLossThreads, 0, as_stream(stream)>>>(
            logits, d4, labels, matched_idx, g4, gt_offsets, a4, total, r, wt, scale_clamp, smooth_l1_beta, grad_scale_cls,
            grad_scale_loc, upstream, accumulators, sums_out, grad_logits, gd4);
    DET_LAUNCH_OK("rpn_loss_kernel");
    return DET_OK;
}

static int yolo_loss_impl(const float* head, const int8_t* labels, const int64_t* matched_idx, const float* gt_boxes,
                          const int64_t* gt_classes, const int32_t* gt_offsets, int n, int s, int b, int c, int img_h,
                          int img_w, const float* priors, float lambda_coord, float lambda_noobj, float grad_scale,
                          const float* upstream, float* accumulators, float* sums_out, float* grad_head, void* stream,
                          const det_peer_ctx_t* peer) {
    DET_CHECK_ARG(n >= 0 && s >= 1 && b >= 1 && c >= 0, "bad size");
    DET_CHECK_ARG(accumulators && sums_out, "null accumulators / sums_out");
    if (n == 0) {
        cudaError_t e = cudaMemsetAsync(sums_out, 0, 8 * sizeof(float), as_stream(stream));
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
        return DET_OK;
    }
    DET_CHECK_ARG(head && labels && matched_idx && gt_offsets && priors, "null pointer");
    if (gt_boxes && !aligned16(gt_boxes)) {
        set_error("gt_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    YoloLossParams prm;
    prm.n = n; prm.s = s; prm.b = b; prm.c = c;
    prm.stride_x = (float)((double)img_w / (double)s);
    prm.stride_y = (float)((double)img_h / (double)s);
    prm.lambda_coord = lambda_coord; prm.lambda_noobj = lambda_noobj; prm.grad_scale = grad_scale;
    const int per_img = s * s * (b * 5 + c);
    auto g4 = reinterpret_cast<const float4*>(gt_boxes);
    auto p2 = reinterpret_cast<const float2*>(priors);
    PeerCtxDev pc;
    pc.enabled = 0;
    pc.stamp_counter = nullptr;
    if (peer) {
        DET_CHECK_ARG(peer->peers_dev && peer->out, "peer context: null pointer");
        DET_CHECK_ARG(peer->width >= 1 && peer->width <= 8, "peer context: width must be in [1, 8] (the sums vector)");
        DET_CHECK_ARG(peer->world >= 1 && peer->world <= kPeerMaxWorld && peer->rank >= 0 && peer->rank < peer->world,
                      "peer context: bad rank / world");
        DET_CHECK_ARG(peer->slots >= 4 && peer->lag >= 1 && (int)peer->lag <= peer->slots - 3 && peer->timeout_ns > 0,
                      "peer context: slots >= 4, 1 <= lag <= slots - 3");
        DET_CHECK_ARG(per_img <= kYoloLossTile, "peer context: only the shared-memory-tile kernel publishes");
        pc.peers = reinterpret_cast<float* const*>(peer->peers_dev); pc.out = peer->out;
        pc.error_flag = peer->error_flag; pc.timeout_ns = peer->timeout_ns;
        pc.width = peer->width; pc.rank = peer->rank; pc.world = peer->world; pc.slots = peer->slots;
        pc.stamp = peer->stamp; pc.lag = peer->lag; pc.stamp_counter = peer->stamp_counter; pc.enabled = 1;
    }
    if (per_img <= kYoloLossTile) {
        int imgs = kYoloLossTile / per_img;
        // enough CTAs to fill the GPU first, then as many images per CTA as the tile holds
        const int fill = (n + 2 * sm_count() - 1) / (2 * sm_count());
        if (imgs > fill) imgs = fill < 1 ? 1 : fill;
        const size_t smem = 2 * sizeof(float) * (size_t)((imgs * per_img + 3) & ~3);
        yolo_loss_kernel<<<(unsigned)((n + imgs - 1) / imgs), kYoloLossThreads, smem, as_stream(stream)>>>(
            head, labels, matched_idx, g4, gt_classes, gt_offsets, p2, prm, imgs, upstream, accumulators, sums_out, grad_head, pc);
    } else {
        const int64_t cells = (int64_t)n * s * s;
        yolo_loss_direct_kernel<<<(unsigned)((cells + 127) / 128), 128, 0, as_stream(stream)>>>(
            head, labels, matched_idx, g4, gt_classes, gt_offsets, p2, prm, upstream, accumulators, sums_out, grad_head);
    }
    DET_LAUNCH_OK("yolo_loss_kernel");
    return DET_OK;
}

int det_yolo_loss(const float* head, const int8_t* labels, const int64_t* matched_idx, const float* gt_boxes,
                  const int64_t* gt_classes, const int32_t* gt_offsets, int n, int s, int b, int c, int img_h,
                  int img_w, const float* priors, float lambda_coord, float lambda_noobj, float grad_scale,
                  const float* upstream, float* accumulators, float* sums_out, float* grad_head, void* stream) {
    return yolo_loss_impl(head, labels, matched_idx, gt_boxes, gt_classes, gt_offsets, n, s, b, c, img_h, img_w, priors,
                          lambda_coord, lambda_noobj, grad_scale, upstream, accumulators, sums_out, grad_head, stream,
                          nullptr);
}

int det_yolo_loss_peer(const float* head, const int8_t* labels, const int64_t* matched_idx, const float* gt_boxes,
                       const int64_t* gt_classes, const int32_t* gt_offsets, int n, int s, int b, int c, int img_h,
                       int img_w, const float* priors, float lambda_coord, float lambda_noobj, float grad_scale,
                       const float* upstream, float* accumulators, float* sums_out, float* grad_head,
                       const det_peer_ctx_t* peer, void* stream) {
    DET_CHECK_ARG(peer, "null peer context");
    DET_CHECK_ARG(n >= 1, "the publishing kernel needs a non-empty batch");
    return yolo_loss_impl(head, labels, matched_idx, gt_boxes, gt_classes, gt_offsets, n, s, b, c, img_h, img_w, priors,
                          lambda_coord, lambda_noobj, grad_scale, upstream, accumulators, sums_out, grad_head, stream, peer);
}

}  // extern "C"
