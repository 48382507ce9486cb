// Second-stage (Fast R-CNN box predictor) training losses, forward and backward in one launch (det_fast_rcnn_loss_typed):
// softmax cross-entropy over the K+1 logits of every row, and smooth-L1 / GIoU box regression on the 4 deltas of the
// row's gt class for the foreground rows, plus detectron2's classification statistics from the same pass.
//
// Specification: detectron2 v0.6 FastRCNNOutputLayers.losses / box_reg_loss / _log_classification_stats (own; the
// reference never wrote the ROI predictor, SURVEY.md section 0), restated in tests/fast_rcnn_loss_oracle.py.  One
// deviation: a label outside [0, K] (detectron2 device-asserts) contributes nothing and gets zero gradient rows.
//
// fast_rcnn_loss_kernel<T, NC>: one warp per row, kLossWarps rows per CTA.
//   K + 1 <= 32 * (NC + 1) columns (NC = 1 or 3): every logit of the row is loaded at once into registers (lane l
//   holds columns l, l + 32, ...), together with the foreground row's single delta group, proposal and gt box (one
//   lane).  NC = 0, larger K: the columns are walked three times (max / argmax, exp-sum, gradient); the re-reads hit L1.
//   Reductions are xor butterflies, so every lane holds the same max, sum and argmax bit for bit.
//   The lane that owns column gt adds the row's cross-entropy logsumexp - x[gt]; the lane that owns delta group gt (group
//   0 when class-agnostic) computes the box term with smooth_l1 / encode_delta / giou_fwd_bwd -- the RPN
//   losses' arithmetic.  Gradients: (softmax - onehot) * s_cls for every column, and for every delta group zero except
//   group gt of a foreground row; all stores streaming, a warp's stores covering consecutive sectors.
//   Every CTA adds its partial sums to the accumulators with one atomic per sum, and the last CTA writes the 8 weighted
//   sums and re-arms the accumulators (peer.cuh), so the launch needs neither a memset before nor an op after it.
// Compulsory traffic: M * (4(K+1) + 8) + fg * 48 bytes read, M * 4(5K+1) written with gradients (fp32); at 8192 rows and
// K = 80 that is about 16 MB -- a few microseconds of HBM time, so the call is latency-bound.
#include <limits.h>
#include "assign.cuh"
#include "peer.cuh"

namespace det {

constexpr int kLossWarps = 8;        // rows per CTA
constexpr int kLossMaxClasses = 4096;
constexpr int kLossSums = 7;         // loss_cls, loss_box_reg, num_fg, num_accurate, fg_num_accurate, false neg., bad

struct LossArgs {
    const void* logits;  // (m, K+1) elements of T
    const void* deltas;  // (m, K*4) or (m, 4) elements of T
    const float4* proposals;
    const int64_t* gt_classes;
    const float4* gt_boxes;
    int64_t m;
    int k, agnostic, giou, deltas_vec;
    CodecWeights wt;
    float scale_clamp, beta, scale_cls, scale_loc;
    const float* upstream;
    float* acc;
    float* sums_out;
    void* grad_logits;  // (m, K+1) elements of T, or NULL
    void* grad_deltas;  // like deltas, or NULL
};

// per-lane partial sums of a CTA's rows
struct LossPart {
    float cls, loc;
    int fg, accurate, fg_accurate, false_neg, bad;
};

// torch.argmax's order: a NaN beats every number and the first NaN wins; otherwise the larger value, and of equal
// values the lower column.  A total order, so the butterfly gives every lane the same winner.
__device__ __forceinline__ void argmax_take(float& v, int& i, float ov, int oi) {
    const bool vn = v != v, on = ov != ov;
    const bool take = on ? (!vn || oi < i) : (!vn && (ov > v || (ov == v && oi < i)));
    if (take) {
        v = ov;
        i = oi;
    }
}

__device__ __forceinline__ void warp_argmax(float& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        argmax_take(v, i, ov, oi);
    }
}

template <typename T>
__device__ __forceinline__ void store_group(const LossArgs& g, int64_t q, const float4 v) {
    if (g.deltas_vec) {
        st4_stream<T>(static_cast<typename Head<T>::vec*>(g.grad_deltas) + q, v);
    } else {
        T* p = static_cast<T*>(g.grad_deltas) + q * 4;
        st_stream(p, v.x); st_stream(p + 1, v.y); st_stream(p + 2, v.z); st_stream(p + 3, v.w);
    }
}

// the box term of a foreground row (one lane): adds the loss to part.loc and returns d(loss)/d(deltas) * gs_loc
template <typename T>
__device__ __forceinline__ float4 box_term(const LossArgs& g, int64_t row, int64_t q, float gs_loc, LossPart& part) {
    const float4 d = ld_group<T>(g.deltas, g.deltas_vec, q);
    const float4 pr = g.proposals[row], gb = g.gt_boxes[row];
    float4 gd;
    if (g.giou) {
        part.loc += giou_fwd_bwd(d, pr, gb, g.wt, g.scale_clamp, gd);
    } else {
        const float4 t = encode_delta(pr, gb, g.wt);
        float v;
        smooth_l1(d.x, t.x, g.beta, v, gd.x); part.loc += v;
        smooth_l1(d.y, t.y, g.beta, v, gd.y); part.loc += v;
        smooth_l1(d.z, t.z, g.beta, v, gd.z); part.loc += v;
        smooth_l1(d.w, t.w, g.beta, v, gd.w); part.loc += v;
    }
    return make_float4(gd.x * gs_loc, gd.y * gs_loc, gd.z * gs_loc, gd.w * gs_loc);
}

// counts of one row (lane 0 adds them): pred is the row's argmax, K the background column
__device__ __forceinline__ void count_row(LossPart& part, int64_t gt, int pred, int K) {
    const bool fg = gt >= 0 && gt < K;
    part.fg += fg;
    part.accurate += (int64_t)pred == gt;
    part.fg_accurate += fg && (int64_t)pred == gt;
    part.false_neg += fg && pred == K;
    part.bad += gt < 0 || gt > K;
}

// the delta-gradient row: zero everywhere except group `own` (-1: none), which gets gd
template <typename T>
__device__ __forceinline__ void store_delta_row(const LossArgs& g, int64_t row, int own, const float4 gd) {
    const int lane = threadIdx.x & 31, groups = g.agnostic ? 1 : g.k;
    const int64_t q0 = row * groups;
    for (int c = lane; c < groups; c += 32)
        store_group<T>(g, q0 + c, c == own ? gd : make_float4(0.f, 0.f, 0.f, 0.f));
}

// Register path: K + 1 <= 32 * (NC + 1) columns, all loads of the row in flight at once.
template <typename T, int NC>
__device__ __forceinline__ void row_registers(const LossArgs& g, int64_t row, float gs_cls, float gs_loc, LossPart& part) {
    const int lane = threadIdx.x & 31, K = g.k;
    const T* lr = static_cast<const T*>(g.logits) + row * (K + 1);
    const int64_t gt = g.gt_classes[row];
    float lx[NC + 1];
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        const int c = lane + 32 * j;
        lx[j] = c <= K ? ld1_stream(lr + c) : -INFINITY;
    }
    const bool fg = gt >= 0 && gt < K, valid = gt >= 0 && gt <= K;
    const int own = fg ? (g.agnostic ? 0 : (int)gt) : -1;  // the delta group that carries the box term
    float4 gd = make_float4(0.f, 0.f, 0.f, 0.f);
    if (own >= 0 && lane == (own & 31)) gd = box_term<T>(g, row, row * (g.agnostic ? 1 : K) + own, gs_loc, part);
    float mx = -INFINITY, av = -INFINITY;
    int ai = INT_MAX;
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        mx = max_nan(mx, lx[j]);
        if (lane + 32 * j <= K) argmax_take(av, ai, lx[j], lane + 32 * j);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    warp_argmax(av, ai);
    float e[NC + 1], s = 0.0f;
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        e[j] = lane + 32 * j <= K ? expf(lx[j] - mx) : 0.0f;
        s += e[j];
    }
    s = warp_sum(s);
    if (valid) {
#pragma unroll
        for (int j = 0; j <= NC; ++j)
            if (lane + 32 * j == gt) part.cls += logf(s) - (lx[j] - mx);
    }
    if (lane == 0) count_row(part, gt, ai, K);
    if (!g.grad_logits) return;
    T* gr = static_cast<T*>(g.grad_logits) + row * (K + 1);
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        const int c = lane + 32 * j;
        if (c > K) break;
        const float p = e[j] / s;
        st_stream(gr + c, valid ? (c == gt ? p - 1.0f : p) * gs_cls : 0.0f);
    }
    store_delta_row<T>(g, row, own, gd);
}

// General path: any K up to kLossMaxClasses; the row is walked three times (the re-reads are L1 hits).
template <typename T>
__device__ __forceinline__ void row_general(const LossArgs& g, int64_t row, float gs_cls, float gs_loc, LossPart& part) {
    const int lane = threadIdx.x & 31, K = g.k;
    const T* lr = static_cast<const T*>(g.logits) + row * (K + 1);
    const int64_t gt = g.gt_classes[row];
    const bool fg = gt >= 0 && gt < K, valid = gt >= 0 && gt <= K;
    const int own = fg ? (g.agnostic ? 0 : (int)gt) : -1;
    float4 gd = make_float4(0.f, 0.f, 0.f, 0.f);
    if (own >= 0 && lane == (own & 31)) gd = box_term<T>(g, row, row * (g.agnostic ? 1 : K) + own, gs_loc, part);
    float mx = -INFINITY, av = -INFINITY, xg = 0.0f;
    int ai = INT_MAX;
#pragma unroll 4
    for (int c = lane; c <= K; c += 32) {
        const float x = ld1(lr + c);
        mx = max_nan(mx, x);
        argmax_take(av, ai, x, c);
        if (c == gt) xg = x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    warp_argmax(av, ai);
    float s = 0.0f;
#pragma unroll 4
    for (int c = lane; c <= K; c += 32) s += expf(ld1(lr + c) - mx);
    s = warp_sum(s);
    if (valid && lane == (int)(gt & 31)) part.cls += logf(s) - (xg - mx);
    if (lane == 0) count_row(part, gt, ai, K);
    if (!g.grad_logits) return;
    T* gr = static_cast<T*>(g.grad_logits) + row * (K + 1);
#pragma unroll 4
    for (int c = lane; c <= K; c += 32) {
        const float p = expf(ld1(lr + c) - mx) / s;
        st_stream(gr + c, valid ? (c == gt ? p - 1.0f : p) * gs_cls : 0.0f);
    }
    store_delta_row<T>(g, row, own, gd);
}

template <typename T, int NC>
__global__ void __launch_bounds__(kLossWarps * 32) fast_rcnn_loss_kernel(const __grid_constant__ LossArgs g) {
    __shared__ float s_part[kLossSums][kLossWarps];
    __shared__ float s_fin[8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * kLossWarps + wid;
    LossPart part{0.f, 0.f, 0, 0, 0, 0, 0};
    if (row < g.m) {  // no early return: every CTA takes part in the arrival count below
        float gs_cls = g.scale_cls, gs_loc = g.scale_loc;
        if (g.upstream) {
            gs_cls *= g.upstream[0];
            gs_loc *= g.upstream[1];
        }
        if constexpr (NC > 0) row_registers<T, NC>(g, row, gs_cls, gs_loc, part);
        else row_general<T>(g, row, gs_cls, gs_loc, part);
    }
    const float v[kLossSums] = {warp_sum(part.cls), warp_sum(part.loc), (float)warp_sum(part.fg),
                                (float)warp_sum(part.accurate), (float)warp_sum(part.fg_accurate),
                                (float)warp_sum(part.false_neg), (float)warp_sum(part.bad)};
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < kLossSums; ++i) s_part[i][wid] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < kLossSums) {
        float t = 0.0f;
        for (int w = 0; w < kLossWarps; ++w) t += s_part[threadIdx.x][w];
        if (t != 0.0f) atomicAdd(&g.acc[threadIdx.x], t);
    }
    // last CTA: sums_out = [loss_cls, loss_box_reg, counts...], accumulators and ticket re-armed
    if (last_cta_arrives(reinterpret_cast<int32_t*>(g.acc + 8)))
        finalize_sums(g.acc, g.sums_out, s_fin, [&](int i) { return i == 0 ? g.scale_cls : (i == 1 ? g.scale_loc : 1.0f); });
}

template <typename T, int NC>
static int launch_loss_nc(const LossArgs& g, cudaStream_t st) {
    const int64_t blocks = (g.m + kLossWarps - 1) / kLossWarps;
    fast_rcnn_loss_kernel<T, NC><<<(unsigned)blocks, kLossWarps * 32, 0, st>>>(g);
    DET_LAUNCH_OK("fast_rcnn_loss_kernel");
    return DET_OK;
}

template <typename T>
static int fast_rcnn_loss_t(const void* class_logits, const void* box_deltas, const float* proposals,
                            const int64_t* gt_classes, const float* gt_boxes, int64_t m, int num_classes,
                            int class_agnostic, float wx, float wy, float ww, float wh, float scale_clamp, int loss_type,
                            float smooth_l1_beta, float scale_cls, float scale_loc, const float* upstream,
                            float* accumulators, float* sums_out, void* grad_logits, void* grad_deltas, void* stream) {
    DET_CHECK_ARG(m >= 0, "bad size");
    DET_CHECK_ARG(num_classes >= 1, "num_classes must be positive");
    DET_CHECK_ARG(loss_type == 0 || loss_type == 1, "loss_type must be 0 (smooth-L1) or 1 (GIoU)");
    DET_CHECK_ARG(accumulators && sums_out, "null accumulators / sums_out");
    DET_CHECK_ARG((grad_logits == nullptr) == (grad_deltas == nullptr), "both gradients or none");
    if (num_classes > kLossMaxClasses || m >= (1ll << 24)) {
        set_error("det_fast_rcnn_loss needs num_classes <= %d and m < 2^24 (got %d, %lld)", kLossMaxClasses,
                  num_classes, (long long)m);
        return DET_ERR_UNSUPPORTED;
    }
    cudaStream_t st = as_stream(stream);
    if (m == 0) {  // detectron2's empty batch: both losses and every count are 0; no input is read
        const cudaError_t e = cudaMemsetAsync(sums_out, 0, 8 * sizeof(float), st);
        return e == cudaSuccess ? DET_OK : cuda_fail(e, "cudaMemsetAsync");
    }
    DET_CHECK_ARG(class_logits && box_deltas && proposals && gt_classes && gt_boxes, "null input");
    if (!aligned16(proposals) || !aligned16(gt_boxes)) {
        set_error("proposals and gt_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    LossArgs g;
    g.logits = class_logits; g.deltas = box_deltas;
    g.proposals = reinterpret_cast<const float4*>(proposals);
    g.gt_classes = gt_classes;
    g.gt_boxes = reinterpret_cast<const float4*>(gt_boxes);
    g.m = m; g.k = num_classes; g.agnostic = class_agnostic ? 1 : 0; g.giou = loss_type;
    g.deltas_vec = aligned_to(box_deltas, 4 * sizeof(T)) && (!grad_deltas || aligned_to(grad_deltas, 4 * sizeof(T)));
    g.wt = CodecWeights{wx, wy, ww, wh};
    g.scale_clamp = scale_clamp; g.beta = smooth_l1_beta; g.scale_cls = scale_cls; g.scale_loc = scale_loc;
    g.upstream = upstream;
    g.acc = accumulators; g.sums_out = sums_out;
    g.grad_logits = grad_logits; g.grad_deltas = grad_deltas;
    // the register path up to 128 columns (COCO's 80 classes: 81 columns, four per lane), the general one above
    if (num_classes + 1 <= 64) return launch_loss_nc<T, 1>(g, st);
    if (num_classes + 1 <= 128) return launch_loss_nc<T, 3>(g, st);
    return launch_loss_nc<T, 0>(g, st);
}

}  // namespace det

using namespace det;

// C linkage through the declaration in det_b200.h.
int det_fast_rcnn_loss_typed(const void* class_logits, const void* box_deltas, int head_dtype, const float* proposals,
                             const int64_t* gt_classes, const float* gt_boxes, int64_t m, int num_classes,
                             int class_agnostic, float wx, float wy, float ww, float wh, float scale_clamp,
                             int loss_type, float smooth_l1_beta, float scale_cls, float scale_loc,
                             const float* upstream, float* accumulators, float* sums_out, void* grad_logits,
                             void* grad_deltas, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, fast_rcnn_loss_t, class_logits, box_deltas, proposals, gt_classes, gt_boxes, m,
                      num_classes, class_agnostic, wx, wy, ww, wh, scale_clamp, loss_type, smooth_l1_beta, scale_cls,
                      scale_loc, upstream, accumulators, sums_out, grad_logits, grad_deltas, stream);
}
