// Second-stage (Fast R-CNN box predictor) inference for the whole batch: softmax, class-specific decode, clip, score
// threshold and per-class NMS in two launches (det_roi_detect), and the dense form of the first four steps for the exact
// overflow route (det_roi_decode_dense).
//
// Specification: tests/fast_rcnn_oracle.py fast_rcnn_inference_single_image -- detectron2's fast_rcnn_inference_single_image
// (own; the reference never wrote the ROI predictor, SURVEY.md section 0), with one deviation: a detection's flat id
// i*K + c numbers the proposal i among the image's ORIGINAL rows, where detectron2 numbers the rows left after its
// finiteness filter.
//
// roi_detect_kernel<SELECT, T, NC>: one warp per proposal row.  The row's K+1 logits are reduced to their maximum, then
// e = exp(x - max) goes to the warp's slice of shared memory and every lane sums e[0] + e[1] + ... + e[K] in column
// order -- the order the oracle restates, so the probabilities p = e / s are bit-comparable.  K <= 96 (NC = 1 or 3):
// every load of the row is issued at once (4-byte logit loads, 16-byte delta loads) and the decoded boxes stay in
// registers.  Larger K: the general loop (16-byte logit loads when the row pitch and base allow, scalar otherwise).  Every one of the K boxes is decoded to check that the
// row is finite (detectron2's valid_mask covers all boxes and all K+1 probabilities), which is why every delta of every
// row is read: that stream -- 4(K+1) + 16K + 16 bytes per row in fp32 -- is the kernel's compulsory traffic.
// SELECT: the passing (row, class) pairs of a valid row are appended to the image's candidate list with one atomicAdd
// per row (the warp is the row, so the warp-aggregated append of det_dense_detect reduces to a ballot scan); their box
// is decoded again (the deltas are cache hits) and clipped.  The second launch is det_dense_detect's NMS kernel
// (nms_list.cuh) with cand_id = the flat id: its keys are score | id, so ties fall to the lower flat id = the row-major
// order of torch.nonzero.
// DENSE: every (row, class) of the padded (n, p_max, K) layout is written -- probability and clipped box, NaN for the
// rows of an invalid proposal and for the rows past an image's count, so that no such row ever passes a threshold.
// With `decoded` the rows hold probabilities and boxes already (fast_rcnn_inference's inputs) and only the validity
// rule, the clip and the padding apply.
#include "nms_core.cuh"
#include "nms_list.cuh"

namespace det {

constexpr int kRoiWarps = 8;  // warps (= proposal rows) per CTA
constexpr int kRoiMaxClasses = 4096;

struct RoiArgs {
    const void* logits;  // (m, K+1) elements of T
    const void* deltas;  // (m, K*4) or (m, 4) elements of T
    const float4* proposals;
    const int32_t* row_offsets;
    const int32_t* image_sizes;  // (n, 2) = (h, w)
    int n, k, agnostic;
    int decoded;  // DENSE only: logits are probabilities, deltas are boxes, both taken as they are
    int logits_vec, deltas_vec;  // rows can be read with one vector load per 4 elements
    int64_t m;
    CodecWeights wt;
    float scale_clamp;
    // SELECT
    SelectArgs sel;
    // DENSE
    int p_max;
    float* scores_out;   // (n, p_max, K)
    float4* boxes_out;   // (n, p_max, K)
};

// Boxes.clip: x to [0, w], y to [0, h].  Written as comparisons so that the result is the oracle's torch.where form on
// every input, signed zeros included; it only ever sees finite boxes of valid rows.
__device__ __forceinline__ float4 clip_box(float4 b, float w, float h) {
    b.x = b.x < 0.0f ? 0.0f : (b.x > w ? w : b.x);
    b.y = b.y < 0.0f ? 0.0f : (b.y > h ? h : b.y);
    b.z = b.z < 0.0f ? 0.0f : (b.z > w ? w : b.z);
    b.w = b.w < 0.0f ? 0.0f : (b.w > h ? h : b.w);
    return b;
}

__device__ __forceinline__ bool finite4(const float4 b) {
    return isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w);
}

// the delta group of (row, class c): group row * K + c, or group row when class-agnostic
__device__ __forceinline__ int64_t delta_group(const RoiArgs& g, int64_t row, int c) {
    return row * (g.agnostic ? 1 : g.k) + (g.agnostic ? 0 : c);
}

// General path (any K up to kRoiMaxClasses): the logits live in the warp's shared-memory slice, the deltas are read
// once for the finiteness test and again (cache hits) for the classes that pass.
template <bool SELECT, typename T>
__device__ __forceinline__ void row_general(const RoiArgs& g, float* xs, int img, int i, int64_t row, int64_t out0) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, K = g.k;
    // the box of class c, before clipping
    const float4 prop = g.decoded ? make_float4(0.f, 0.f, 0.f, 0.f) : g.proposals[row];
    auto box_of = [&](int c) {
        const float4 d = ld_group<T>(g.deltas, g.deltas_vec, delta_group(g, row, c));
        return g.decoded ? d : decode_delta(prop, d, g.wt, g.scale_clamp);
    };
    // ---- softmax over the K+1 logits
    float mx = -INFINITY;
    if (g.logits_vec) {
        const typename Head<T>::vec* lr = static_cast<const typename Head<T>::vec*>(g.logits) + row * ((K + 1) >> 2);
        for (int q = lane; q < (K + 1) >> 2; q += 32) {
            const float4 v = ld4_stream<T>(lr + q);
            reinterpret_cast<float4*>(xs)[q] = v;
            mx = max_nan(mx, max_nan(max_nan(v.x, v.y), max_nan(v.z, v.w)));
        }
    } else {
        const T* lr = static_cast<const T*>(g.logits) + row * (K + 1);
        for (int c = lane; c <= K; c += 32) {
            const float x = ld1_stream(lr + c);
            xs[c] = x;
            mx = max_nan(mx, x);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max_nan(mx, __shfl_xor_sync(FULL, mx, o));
    // ---- every box of the row must be finite (the deltas do not depend on the logits: these loads go out before the
    // softmax's dependent steps)
    int fin = 1;
    if (g.agnostic) {
        fin = finite4(box_of(0));
    } else {
#pragma unroll 4
        for (int c = lane; c < K; c += 32) fin &= finite4(box_of(c));
    }
    __syncwarp();
    float s = 1.0f;  // probabilities given: p = x / 1 = x
    if (!g.decoded) {
        for (int c = lane; c <= K; c += 32) xs[c] = expf(xs[c] - mx);
        __syncwarp();
        s = xs[0];
#pragma unroll 8
        for (int c = 1; c <= K; ++c) s += xs[c];  // column order: the oracle's sequential sum
    }
    for (int c = lane; c <= K; c += 32) fin &= (int)isfinite(xs[c] / s);
    const bool valid = __all_sync(FULL, fin);
    const float iw = (float)g.image_sizes[2 * img + 1], ih = (float)g.image_sizes[2 * img];
    if (!SELECT) {
        for (int c = lane; c < K; c += 32) {
            float p = __int_as_float(0x7fc00000);
            float4 b = make_float4(NAN, NAN, NAN, NAN);
            if (valid) {
                p = xs[c] / s;
                b = clip_box(box_of(c), iw, ih);
            }
            g.scores_out[out0 + c] = p;
            g.boxes_out[out0 + c] = b;
        }
        return;
    }
    if (!valid) return;
    // ---- append the passing classes: one atomic per row, slots in class order
    const float thr = g.sel.score_thresh;
    int total = 0;
    for (int c0 = 0; c0 < K; c0 += 32) {
        const int c = c0 + lane;
        total += __popc(__ballot_sync(FULL, c < K && xs[c] / s > thr));
    }
    if (total == 0) return;
    int base = 0;
    if (lane == 0) base = atomicAdd(g.sel.cand_count + (int64_t)img * kCountStride, total);
    base = __shfl_sync(FULL, base, 0);
    const int cap = g.sel.cand_cap;
    for (int c0 = 0; c0 < K && base < cap; c0 += 32) {
        const int c = c0 + lane;
        const float p = c < K ? xs[c] / s : 0.0f;
        const bool pass = c < K && p > thr;
        const unsigned bal = __ballot_sync(FULL, pass);
        const int slot = base + __popc(bal & ((1u << lane) - 1u));
        if (pass && slot < cap) {
            const int64_t o = (int64_t)img * cap + slot;
            g.sel.cand_box[o] = clip_box(box_of(c), iw, ih);
            g.sel.cand_score[o] = p;
            g.sel.cand_cls[o] = c;
            g.sel.cand_id[o] = i * K + c;
        }
        base += __popc(bal);
    }
}

// Register path (K <= 32 * NC): every load of the row -- K+1 logits, K delta vectors, the proposal -- is issued before
// anything waits on one, and the decoded boxes stay in registers for the append, so a row costs one memory round trip
// (plus the append's atomic) instead of three.
template <bool SELECT, typename T, int NC>
__device__ __forceinline__ void row_registers(const RoiArgs& g, float* xs, int img, int i, int64_t row, int64_t out0) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, K = g.k;
    const float4 prop = g.decoded ? make_float4(0.f, 0.f, 0.f, 0.f) : g.proposals[row];
    const T* lr = static_cast<const T*>(g.logits) + row * (K + 1);
    float lx[NC + 1];
    float4 bx[NC];
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        const int c = lane + 32 * j;
        lx[j] = c <= K ? ld1_stream(lr + c) : -INFINITY;
    }
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const int c = lane + 32 * j;
        bx[j] = c < K ? ld_group<T>(g.deltas, g.deltas_vec, delta_group(g, row, c))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j <= NC; ++j) mx = max_nan(mx, lx[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max_nan(mx, __shfl_xor_sync(FULL, mx, o));
    int fin = 1;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        if (!g.decoded) bx[j] = decode_delta(prop, bx[j], g.wt, g.scale_clamp);
        if (lane + 32 * j < K) fin &= (int)finite4(bx[j]);
    }
    float s = 1.0f;  // probabilities given: p = x / 1 = x
    if (!g.decoded) {
#pragma unroll
        for (int j = 0; j <= NC; ++j) {
            const int c = lane + 32 * j;
            lx[j] = expf(lx[j] - mx);
            if (c <= K) xs[c] = lx[j];
        }
        __syncwarp();
        s = xs[0];
#pragma unroll 8
        for (int c = 1; c <= K; ++c) s += xs[c];  // column order: the oracle's sequential sum
    }
#pragma unroll
    for (int j = 0; j <= NC; ++j) {
        lx[j] = lx[j] / s;
        if (lane + 32 * j <= K) fin &= (int)isfinite(lx[j]);
    }
    const bool valid = __all_sync(FULL, fin);
    const float iw = (float)g.image_sizes[2 * img + 1], ih = (float)g.image_sizes[2 * img];
    if (!SELECT) {
#pragma unroll
        for (int j = 0; j < NC; ++j) {
            const int c = lane + 32 * j;
            if (c >= K) break;
            g.scores_out[out0 + c] = valid ? lx[j] : __int_as_float(0x7fc00000);
            g.boxes_out[out0 + c] = valid ? clip_box(bx[j], iw, ih) : make_float4(NAN, NAN, NAN, NAN);
        }
        return;
    }
    if (!valid) return;
    // ---- append the passing classes: one atomic per row, slots in class order
    const float thr = g.sel.score_thresh;
    unsigned bal[NC];
    int total = 0;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        bal[j] = __ballot_sync(FULL, lane + 32 * j < K && lx[j] > thr);
        total += __popc(bal[j]);
    }
    if (total == 0) return;
    int base = 0;
    if (lane == 0) base = atomicAdd(g.sel.cand_count + (int64_t)img * kCountStride, total);
    base = __shfl_sync(FULL, base, 0);
    const int cap = g.sel.cand_cap;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const int c = lane + 32 * j;
        const int slot = base + __popc(bal[j] & ((1u << lane) - 1u));
        if (((bal[j] >> lane) & 1u) && slot < cap) {
            const int64_t o = (int64_t)img * cap + slot;
            g.sel.cand_box[o] = clip_box(bx[j], iw, ih);
            g.sel.cand_score[o] = lx[j];
            g.sel.cand_cls[o] = c;
            g.sel.cand_id[o] = i * K + c;
        }
        base += __popc(bal[j]);
    }
}

template <bool SELECT, typename T, int NC>
__global__ void __launch_bounds__(kRoiWarps * 32) roi_detect_kernel(const __grid_constant__ RoiArgs g) {
    extern __shared__ float roi_smem[];
    if (SELECT) {
        pdl_trigger();  // the NMS kernel's CTAs may move in as SM slots free up
        if (blockIdx.x == 0 && threadIdx.x == 0 && g.sel.overflow_flag) *g.sel.overflow_flag = 0;
    }
    const int lane = threadIdx.x & 31, K = g.k;
    float* xs = roi_smem + (threadIdx.x >> 5) * (K + 1);
    const int64_t w = (int64_t)blockIdx.x * kRoiWarps + (threadIdx.x >> 5);
    int img, i;
    int64_t row;
    if (SELECT) {
        if (w >= g.m) return;
        row = w;
        int lo = 0, hi = g.n;  // the last image whose first row is <= row
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((int64_t)g.row_offsets[mid] <= row) lo = mid;
            else hi = mid;
        }
        img = lo;
        if (row < (int64_t)g.row_offsets[img] || row >= (int64_t)g.row_offsets[img + 1]) return;
        i = (int)(row - g.row_offsets[img]);
    } else {
        if (w >= (int64_t)g.n * g.p_max) return;
        img = (int)(w / g.p_max);
        i = (int)(w - (int64_t)img * g.p_max);
        row = (int64_t)g.row_offsets[img] + i;
    }
    const int64_t out0 = SELECT ? 0 : ((int64_t)img * g.p_max + i) * K;
    if (!SELECT && i >= g.row_offsets[img + 1] - g.row_offsets[img]) {  // padding: never passes a threshold
        for (int c = lane; c < K; c += 32) {
            g.scores_out[out0 + c] = __int_as_float(0x7fc00000);
            g.boxes_out[out0 + c] = make_float4(NAN, NAN, NAN, NAN);
        }
        return;
    }
    if constexpr (NC > 0) row_registers<SELECT, T, NC>(g, xs, img, i, row, out0);
    else row_general<SELECT, T>(g, xs, img, i, row, out0);
}

}  // namespace det

using namespace det;

// The entry points below have C linkage through their declarations in det_b200.h.

int64_t det_roi_detect_workspace_bytes(int n, int64_t cand_cap) { return det_dense_detect_workspace_bytes(n, cand_cap); }

int64_t det_roi_detect_counter_bytes(int n) { return det_dense_detect_counter_bytes(n); }

template <typename T>
static int roi_args(RoiArgs& g, const void* class_logits, const void* box_deltas, const float* proposals,
                    const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                    const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp) {
    DET_CHECK_ARG(n >= 0 && m >= 0, "bad size");
    DET_CHECK_ARG(num_classes >= 1, "num_classes must be positive");
    if (num_classes > kRoiMaxClasses || m * (int64_t)num_classes >= (1ll << 31)) {
        set_error("det_roi_detect needs num_classes <= %d and m * num_classes < 2^31 (got %d, %lld)", kRoiMaxClasses,
                  num_classes, (long long)m);
        return DET_ERR_UNSUPPORTED;
    }
    g.logits = class_logits; g.deltas = box_deltas; g.proposals = reinterpret_cast<const float4*>(proposals);
    g.row_offsets = row_offsets; g.image_sizes = image_sizes;
    g.n = n; g.k = num_classes; g.agnostic = class_agnostic ? 1 : 0; g.decoded = 0; g.m = m;
    g.logits_vec = ((num_classes + 1) % 4 == 0 && aligned_to(class_logits, 4 * sizeof(T))) ? 1 : 0;
    g.deltas_vec = aligned_to(box_deltas, 4 * sizeof(T)) ? 1 : 0;
    g.wt = CodecWeights{wx, wy, ww, wh}; g.scale_clamp = scale_clamp;
    g.sel = SelectArgs{};
    g.p_max = 0; g.scores_out = nullptr; g.boxes_out = nullptr;
    return DET_OK;
}

template <bool SELECT, typename T, int NC>
static int launch_roi_nc(const RoiArgs& g, int64_t warps, cudaStream_t st) {
    const size_t smem = sizeof(float) * kRoiWarps * (size_t)(g.k + 1);
    const int64_t blocks = (warps + kRoiWarps - 1) / kRoiWarps;
    DET_CHECK_ARG(blocks < (1ll << 31), "too many rows");
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(roi_detect_kernel<SELECT, T, NC>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(roi_detect_kernel)");
    }
    roi_detect_kernel<SELECT, T, NC><<<(unsigned)blocks, kRoiWarps * 32, smem, st>>>(g);
    DET_LAUNCH_OK("roi_detect_kernel");
    return DET_OK;
}

// the register path for K <= 96 (COCO's 80 classes: three lanes' worth of classes per lane), the general one above
template <bool SELECT, typename T>
static int launch_roi(const RoiArgs& g, int64_t warps, cudaStream_t st) {
    if (g.k <= 32) return launch_roi_nc<SELECT, T, 1>(g, warps, st);
    if (g.k <= 96) return launch_roi_nc<SELECT, T, 3>(g, warps, st);
    return launch_roi_nc<SELECT, T, 0>(g, warps, st);
}

template <typename T>
static int roi_detect_t(const void* class_logits, const void* box_deltas, const float* proposals,
                        const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                        const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp,
                        float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap, int64_t max_det,
                        int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                        int32_t* overflow_flag, void* workspace, int64_t workspace_bytes, void* stream) {
    DET_CHECK_ARG(mode >= DET_NMS_AUTO && mode <= DET_NMS_OFFSET_TRICK, "unknown mode");
    DET_CHECK_ARG(max_det >= 1, "max_det must be positive");
    if (cand_cap < 1 || cand_cap > 4096) {
        set_error("det_roi_detect needs cand_cap in [1, 4096] (got %lld)", (long long)cand_cap);
        return DET_ERR_UNSUPPORTED;
    }
    RoiArgs g;
    int rc = roi_args<T>(g, class_logits, box_deltas, proposals, row_offsets, n, m, num_classes, class_agnostic,
                         image_sizes, wx, wy, ww, wh, scale_clamp);
    if (rc != DET_OK) return rc;
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(det_idx && det_boxes && det_scores && det_classes && det_count, "null output");
    cudaStream_t st = as_stream(stream);
    if (m == 0) {  // nothing to read: every image has no detection
        cudaError_t e = cudaMemsetAsync(det_count, 0, sizeof(int32_t) * (size_t)n, st);
        if (e == cudaSuccess && overflow_flag) e = cudaMemsetAsync(overflow_flag, 0, sizeof(int32_t), st);
        return e == cudaSuccess ? DET_OK : cuda_fail(e, "cudaMemsetAsync");
    }
    DET_CHECK_ARG(class_logits && box_deltas && proposals && row_offsets && image_sizes, "null input");
    if (!aligned16(proposals) || !aligned16(det_boxes)) {
        set_error("proposals and det_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    rc = bind_select_workspace(g.sel, n, cand_cap, workspace, workspace_bytes, gate & 2, st);
    if (rc != DET_OK) return rc;
    g.sel.overflow_flag = overflow_flag;
    g.sel.score_thresh = score_thresh;
    rc = launch_roi<true, T>(g, m, st);
    if (rc != DET_OK) return rc;
    return launch_list_nms(g.sel, n, float_threshold_below(iou_threshold), mode, max_det, det_idx, det_boxes, det_scores,
                           det_classes, det_count, overflow_flag, st);
}

int det_roi_detect_typed(const void* class_logits, const void* box_deltas, int head_dtype, const float* proposals,
                         const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                         const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp,
                         float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap, int64_t max_det,
                         int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                         int32_t* overflow_flag, void* workspace, int64_t workspace_bytes, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, roi_detect_t, class_logits, box_deltas, proposals, row_offsets, n, m, num_classes,
                      class_agnostic, image_sizes, wx, wy, ww, wh, scale_clamp, score_thresh, iou_threshold, mode, gate,
                      cand_cap, max_det, det_idx, det_boxes, det_scores, det_classes, det_count, overflow_flag, workspace,
                      workspace_bytes, stream);
}

template <typename T>
static int roi_decode_dense_t(const void* class_logits, const void* box_deltas, const float* proposals,
                              const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                              const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp,
                              int decoded, int p_max, float* scores_out, float* boxes_out, void* stream) {
    RoiArgs g;
    const int rc = roi_args<T>(g, class_logits, box_deltas, proposals, row_offsets, n, m, num_classes, class_agnostic,
                               image_sizes, wx, wy, ww, wh, scale_clamp);
    if (rc != DET_OK) return rc;
    DET_CHECK_ARG(p_max >= 0, "bad size");
    if (n == 0 || p_max == 0) return DET_OK;
    DET_CHECK_ARG(row_offsets && image_sizes && scores_out && boxes_out, "null pointer");
    DET_CHECK_ARG(m == 0 || (class_logits && box_deltas && (decoded || proposals)), "null input");
    if ((!decoded && !aligned16(proposals)) || !aligned16(boxes_out)) {
        set_error("proposals and boxes_out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    g.decoded = decoded ? 1 : 0;
    g.p_max = p_max;
    g.scores_out = scores_out;
    g.boxes_out = reinterpret_cast<float4*>(boxes_out);
    return launch_roi<false, T>(g, (int64_t)n * p_max, as_stream(stream));
}

int det_roi_decode_dense_typed(const void* class_logits, const void* box_deltas, int head_dtype, const float* proposals,
                               const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                               const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp,
                               int decoded, int p_max, float* scores_out, float* boxes_out, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, roi_decode_dense_t, class_logits, box_deltas, proposals, row_offsets, n, m,
                      num_classes, class_agnostic, image_sizes, wx, wy, ww, wh, scale_clamp, decoded, p_max, scores_out,
                      boxes_out, stream);
}
