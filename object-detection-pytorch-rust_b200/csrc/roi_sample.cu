// Batched ROI-head proposal sampling: the gt append, IoU matching, class labels and fg/bg subsample of
// label_and_sample_proposals for the whole batch in two launches, with no host synchronisation.
//
// Reference behaviour reproduced (paths relative to the reference root):
//   python/src/models/roi.py:68-193          per image: append gt, pairwise_iou(gt, proposals) -> Matcher -> class
//                                            labels (bg = num_classes, ignored = -1) -> subsample -> gather
//   python/src/models/utils.py:111-155       add_ground_truth_to_proposals (the gt boxes follow the proposals)
//   python/src/utils.py:34-76                subsample_labels: min(#fg, int(S*f)) fg, min(#bg, S - #fg) bg
// The random stream differs from torch.randperm (as det_subsample_labels'): candidate j of image b has the key
// sample_key(image_seed(seed, b), j), and each class keeps its `want` smallest keys -- a uniformly random subset.
//
// Launch 1 (label): CTAs over (image, 256 candidates); every candidate against the image's gt boxes staged in shared
// memory.  A pair whose intersection is 0 has IoU exactly 0 (pair_iou) and never reaches the quotient.  Writes
// (argmax, matcher label) per candidate to the workspace and, for the low-quality rule, the row maxima (atomic max).
// Launch 2 (select): one CTA per image.  Promotion + class labels, class counts, an exact 4 x 8-bit radix select of each
// thinned class's want-th smallest key, then the emit in ascending candidate order (block scans), the padding rows and
// the counts.  It also returns every workspace word it used to zero, so the workspace is all zero between calls.
#include <algorithm>

#include "common.cuh"
#include "assign.cuh"

namespace det {

constexpr int kLabelThreads = 256;
constexpr int kSelectThreads = 1024;
constexpr int kSelectWarps = kSelectThreads / 32;

struct RoiSampleArgs {
    const float4* proposals;  // (n, p_stride)
    const int32_t* counts;    // (n)
    const float4* gt;         // (sum_g)
    const int32_t* gt_off;    // (n + 1)
    const int64_t* gt_classes;
    const uint64_t* seed;
    int64_t p_stride;
    int n, num_classes, num_samples, pos_cap, append_gt;
    MatchRule rule;
    float* rowmax;  // (sum_g), zero between calls
    int32_t* info;  // image b's candidates at b * p_stride + gt_off[b]; zero between calls
    float4* out_boxes;
    int64_t* out_classes;
    float4* out_gt_boxes;
    int32_t* out_matched;
    int32_t* out_src;
    int32_t* out_count;
    int32_t* out_num_fg;
    int32_t* underfull;
};

struct ImageView {
    int64_t p0, i0;  // first proposal row, first info word
    int g0, G, P, C;
};

__device__ __forceinline__ ImageView image_view(const RoiSampleArgs& a, int b) {
    ImageView v;
    v.g0 = a.gt_off[b];
    v.G = a.gt_off[b + 1] - v.g0;
    v.P = (int)min((int64_t)max(a.counts[b], 0), a.p_stride);  // rows past the count are never read
    v.C = v.P + (a.append_gt ? v.G : 0);
    v.p0 = (int64_t)b * a.p_stride;
    v.i0 = v.p0 + v.g0;
    return v;
}

// candidate j: proposal j, then (append_gt) gt box j - P
__device__ __forceinline__ float4 candidate(const RoiSampleArgs& a, const ImageView& v, int j) {
    return j < v.P ? a.proposals[v.p0 + j] : a.gt[v.g0 + (j - v.P)];
}

// info word: matched * 4 + code; launch 1 writes code = matcher label + 1, launch 2 rewrites it as the class code
enum : int { kFg = 0, kBg = 1, kIgnored = 2 };

__global__ void __launch_bounds__(kLabelThreads) roi_sample_label_kernel(const __grid_constant__ RoiSampleArgs a) {
    __shared__ float4 s_gt[kLabelThreads];
    __shared__ float s_ga[kLabelThreads];
    __shared__ unsigned s_rm[kLabelThreads];
    const int b = blockIdx.y, tid = threadIdx.x;
    if (b == 0 && blockIdx.x == 0 && tid == 0) *a.underfull = 0;  // launch 2 sets it
    const ImageView v = image_view(a, b);
    const bool lq = a.rule.allow_lq != 0;
    for (int j0 = blockIdx.x * kLabelThreads; j0 < v.C; j0 += gridDim.x * kLabelThreads) {  // CTA-uniform
        const int j = j0 + tid;
        const bool valid = j < v.C;
        const float4 box = valid ? candidate(a, v, j) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float area = box_area(box);
        float best = 0.0f;  // IoUs are >= 0 and only a strictly larger one replaces the incumbent: gt 0 wins ties at 0,
        int arg = 0;        // and the first maximum wins, like torch.max(dim=0)
        for (int t0 = 0; t0 < v.G; t0 += kLabelThreads) {
            const int nt = min(kLabelThreads, v.G - t0);
            __syncthreads();
            if (tid < nt) {
                const float4 g = a.gt[v.g0 + t0 + tid];
                s_gt[tid] = g;
                s_ga[tid] = box_area(g);
            }
            s_rm[tid] = 0u;
            __syncthreads();
            for (int t = 0; t < nt; ++t) {
                // pair_iou(gt, candidate) (roi.py:157: boxes1 = gt): the quotient only where the intersection is > 0
                const float inter = pair_intersection(s_gt[t], box);
                if (inter > 0.0f) {
                    const float q = inter / (s_ga[t] + area - inter);
                    if (q > best) {
                        best = q;
                        arg = t0 + t;
                    }
                    if (lq && q > 0.0f) atomicMax(&s_rm[t], __float_as_uint(q));
                }
            }
            __syncthreads();
            if (lq && tid < nt && s_rm[tid] != 0u) atomic_max_nonneg(&a.rowmax[v.g0 + t0 + tid], __uint_as_float(s_rm[tid]));
        }
        if (valid) {
            const int lab = v.G == 0 ? (int)a.rule.lab[0] : (int)bucket_label(a.rule, best);  // matcher.py:67-77
            a.info[v.i0 + j] = arg * 4 + (lab + 1);
        }
    }
}

// inclusive prefix sum over a warp
__device__ __forceinline__ int warp_incl_scan(int x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

struct SelectSmem {
    int hist[2][256];
    unsigned prefix[2];
    int remaining[2];
    int cnt[2];
    int any_zero_row;
    int warp_tot[2][kSelectWarps];
};

__global__ void __launch_bounds__(kSelectThreads) roi_sample_select_kernel(const __grid_constant__ RoiSampleArgs a) {
    __shared__ SelectSmem sm;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const ImageView v = image_view(a, b);
    const bool lq = a.rule.allow_lq != 0 && v.G > 0;
    int32_t* info = a.info + v.i0;
    const float* rowmax = a.rowmax + v.g0;
    if (tid < 2) sm.cnt[tid] = 0;
    if (tid == 0) sm.any_zero_row = 0;
    __syncthreads();
    // ---- low-quality promotion (matcher.py:96-120): a gt whose row maximum is 0 promotes every candidate (Q == rowmax
    //      holds everywhere); otherwise a candidate is promoted where its IoU with a gt equals that gt's row maximum (> 0,
    //      so only intersecting pairs can)
    if (lq)
        for (int t = tid; t < v.G; t += kSelectThreads)
            if (rowmax[t] == 0.0f) sm.any_zero_row = 1;
    __syncthreads();
    const bool promote_all = lq && sm.any_zero_row != 0;
    int nfg = 0, nbg = 0;
    for (int j = tid; j < v.C; j += kSelectThreads) {
        const int w = info[j];
        const int m = w >> 2;
        int lab = (w & 3) - 1;
        if (lq && lab != 1) {
            if (promote_all) {
                lab = 1;
            } else {
                const float4 box = candidate(a, v, j);
                const float area = box_area(box);
                for (int t = 0; t < v.G; ++t) {
                    const float4 g = a.gt[v.g0 + t];
                    const float inter = pair_intersection(g, box);
                    if (inter > 0.0f && inter / (box_area(g) + area - inter) == rowmax[t]) {
                        lab = 1;
                        break;
                    }
                }
            }
        }
        // class labels (roi.py:84-95) and subsample_labels' classes (utils.py:56-57): fg = neither -1 nor num_classes
        int code = kBg;
        if (v.G > 0) {
            if (lab == -1) {
                code = kIgnored;
            } else if (lab == 1) {
                const int64_t c = a.gt_classes[v.g0 + m];
                code = c == (int64_t)a.num_classes ? kBg : (c == -1 ? kIgnored : kFg);
            }
        }
        info[j] = m * 4 + code;
        nfg += code == kFg;
        nbg += code == kBg;
    }
    nfg = warp_sum(nfg);
    nbg = warp_sum(nbg);
    if (lane == 0) {
        if (nfg) atomicAdd(&sm.cnt[0], nfg);
        if (nbg) atomicAdd(&sm.cnt[1], nbg);
    }
    __syncthreads();  // every read of the row maxima is done: leave them zero for the next call
    if (lq)
        for (int t = tid; t < v.G; t += kSelectThreads) a.rowmax[v.g0 + t] = 0.0f;
    const int have[2] = {sm.cnt[0], sm.cnt[1]};
    // utils.py:63-69 with int(S*f) evaluated in double on the host (100 * 0.29 -> 28)
    // (per-class values as scalar pairs selected with ?: -- a runtime-indexed array would live in local memory)
    const int want0 = min(have[0], a.pos_cap);
    const int want1 = min(have[1], a.num_samples - want0);
    const bool thin0 = want0 > 0 && want0 < have[0], thin1 = want1 > 0 && want1 < have[1];
    const uint32_t iseed = image_seed(*a.seed, b);
    // ---- the want-th smallest key of each thinned class (keys are a bijection of j: no ties), 4 x 8-bit radix select
    if (thin0 || thin1) {
        if (tid < 2) {
            sm.prefix[tid] = 0u;
            sm.remaining[tid] = tid == 0 ? want0 : want1;
        }
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            const unsigned himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
            __syncthreads();
            for (int t = tid; t < 512; t += kSelectThreads) (&sm.hist[0][0])[t] = 0;
            __syncthreads();
            const unsigned pre0 = sm.prefix[0], pre1 = sm.prefix[1];
            for (int j = tid; j < v.C; j += kSelectThreads) {
                const int c = info[j] & 3;
                if (c == kIgnored || !(c == kFg ? thin0 : thin1)) continue;
                const unsigned key = sample_key(iseed, (uint32_t)j);
                if ((key & himask) == ((c == kFg ? pre0 : pre1) & himask)) atomicAdd(&sm.hist[c][(key >> shift) & 255], 1);
            }
            __syncthreads();
            if (wid < 2 && (wid == 0 ? thin0 : thin1)) {  // warp c scans class c's 256 bins, 8 per lane
                int h[8], s = 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    h[i] = sm.hist[wid][lane * 8 + i];
                    s += h[i];
                }
                const int incl = warp_incl_scan(s), excl = incl - s;
                int rem = sm.remaining[wid];
                __syncwarp();
                if (excl < rem && rem <= incl) {
                    rem -= excl;
                    int bin = 0;
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (bin == 0 && rem <= h[i]) bin = i + 1;
                        else if (bin == 0) rem -= h[i];
                    sm.prefix[wid] |= (unsigned)(lane * 8 + bin - 1) << shift;
                    sm.remaining[wid] = rem;
                }
            }
        }
        __syncthreads();
    }
    const unsigned sel0 = sm.prefix[0], sel1 = sm.prefix[1];
    // ---- emit: fg rows first, then bg, each in ascending candidate order (block scans over tiles of candidates)
    const int count = want0 + want1;
    int base0 = 0, base1 = want0;
    for (int t0 = 0; t0 < v.C; t0 += kSelectThreads) {
        const int j = t0 + tid;
        int c = kIgnored, m = 0;
        bool keep = false;
        if (j < v.C) {
            const int w = info[j];
            info[j] = 0;  // the workspace is all zero between calls
            c = w & 3;
            m = w >> 2;
            if (c == kFg && want0 > 0) keep = !thin0 || sample_key(iseed, (uint32_t)j) <= sel0;
            if (c == kBg && want1 > 0) keep = !thin1 || sample_key(iseed, (uint32_t)j) <= sel1;
        }
        const unsigned bal0 = __ballot_sync(0xffffffffu, keep && c == kFg);
        const unsigned bal1 = __ballot_sync(0xffffffffu, keep && c == kBg);
        __syncthreads();  // the previous tile's totals have been read
        if (lane == 0) {
            sm.warp_tot[0][wid] = __popc(bal0);
            sm.warp_tot[1][wid] = __popc(bal1);
        }
        __syncthreads();
        int before0 = 0, before1 = 0, total0 = 0, total1 = 0;
        for (int w = 0; w < kSelectWarps; ++w) {
            const int x0 = sm.warp_tot[0][w], x1 = sm.warp_tot[1][w];
            before0 += w < wid ? x0 : 0;
            before1 += w < wid ? x1 : 0;
            total0 += x0;
            total1 += x1;
        }
        if (keep) {
            const unsigned below = (1u << lane) - 1u;
            const int row = c == kFg ? base0 + before0 + __popc(bal0 & below) : base1 + before1 + __popc(bal1 & below);
            const int64_t o = (int64_t)b * a.num_samples + row;
            const float4 box = candidate(a, v, j);
            a.out_boxes[o] = box;
            a.out_src[o] = j;
            if (v.G > 0) {
                a.out_classes[o] = c == kFg ? a.gt_classes[v.g0 + m] : (int64_t)a.num_classes;
                a.out_gt_boxes[o] = a.gt[v.g0 + m];  // roi.py:174-181 copies gt[matched] for bg rows too
                a.out_matched[o] = m;
            } else {  // no gt: background with its own box as target (what FastRCNNOutputs.losses substitutes)
                a.out_classes[o] = a.num_classes;
                a.out_gt_boxes[o] = box;
                a.out_matched[o] = -1;
            }
        }
        base0 += total0;
        base1 += total1;
    }
    for (int row = count + tid; row < a.num_samples; row += kSelectThreads) {
        const int64_t o = (int64_t)b * a.num_samples + row;
        a.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        a.out_gt_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        a.out_classes[o] = -1;
        a.out_matched[o] = -1;
        a.out_src[o] = -1;
    }
    if (tid == 0) {
        a.out_count[b] = count;
        a.out_num_fg[b] = want0;
        if (count < a.num_samples) *a.underfull = 1;
    }
}

static int64_t rowmax_bytes(int64_t sum_g) { return (sum_g * 4 + 15) & ~(int64_t)15; }

}  // namespace det

using namespace det;

// C linkage through the declarations in det_b200.h.
int64_t det_roi_sample_workspace_bytes(int n, int64_t p_stride, int64_t sum_g) {
    if (n < 0 || p_stride < 0 || sum_g < 0) return 0;
    return rowmax_bytes(sum_g) + ((int64_t)n * p_stride + sum_g) * 4;
}

int det_roi_sample_proposals(const float* proposals, const int32_t* proposal_counts, int n, int64_t p_stride,
                             const float* gt_boxes, const int32_t* gt_offsets, const int64_t* gt_classes, int64_t sum_g,
                             int num_classes, const float* thresholds_host, const int32_t* labels_host,
                             int num_thresholds, int allow_low_quality, int batch_size_per_image,
                             double positive_fraction, int append_gt, const uint64_t* seed, float* out_boxes,
                             int64_t* out_gt_classes, float* out_gt_boxes, int32_t* out_matched, int32_t* out_src,
                             int32_t* out_count, int32_t* out_num_fg, int32_t* underfull_flag, void* workspace,
                             int64_t workspace_bytes, void* stream) {
    DET_CHECK_ARG(n >= 0 && p_stride >= 0 && sum_g >= 0, "negative size");
    DET_CHECK_ARG(num_classes >= 1, "num_classes must be positive");
    DET_CHECK_ARG(batch_size_per_image >= 1, "batch_size_per_image must be positive");
    DET_CHECK_ARG(positive_fraction >= 0.0 && positive_fraction <= 1.0, "positive_fraction must be in [0, 1]");
    MatchRule rule;
    const int rc = fill_rule(rule, thresholds_host, labels_host, num_thresholds, allow_low_quality);
    if (rc != DET_OK) return rc;
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(proposal_counts && gt_offsets && seed && underfull_flag && workspace, "null pointer");
    DET_CHECK_ARG(out_boxes && out_gt_classes && out_gt_boxes && out_matched && out_src && out_count && out_num_fg,
                  "null output");
    DET_CHECK_ARG(proposals || p_stride == 0, "null proposals");
    DET_CHECK_ARG((gt_boxes && gt_classes) || sum_g == 0, "null gt_boxes / gt_classes");
    if (n > 65535 || p_stride >= (1ll << 24) || sum_g >= (1ll << 24) || batch_size_per_image >= (1 << 24) ||
        (int64_t)n * p_stride + sum_g >= (1ll << 31)) {
        set_error("det_roi_sample_proposals needs n <= 65535, p_stride < 2^24, sum_g < 2^24, batch_size_per_image < 2^24 "
                  "and n * p_stride + sum_g < 2^31");
        return DET_ERR_UNSUPPORTED;
    }
    if ((proposals && !aligned16(proposals)) || (gt_boxes && !aligned16(gt_boxes)) || !aligned16(out_boxes) ||
        !aligned16(out_gt_boxes) || !aligned16(workspace)) {
        set_error("proposals, gt_boxes, out_boxes, out_gt_boxes and workspace must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    const int64_t need = det_roi_sample_workspace_bytes(n, p_stride, sum_g);
    if (workspace_bytes < need) {
        set_error("workspace too small: need %lld bytes", (long long)need);
        return DET_ERR_WORKSPACE;
    }
    RoiSampleArgs a;
    a.proposals = reinterpret_cast<const float4*>(proposals);
    a.counts = proposal_counts;
    a.gt = reinterpret_cast<const float4*>(gt_boxes);
    a.gt_off = gt_offsets;
    a.gt_classes = gt_classes;
    a.seed = seed;
    a.p_stride = p_stride;
    a.n = n;
    a.num_classes = num_classes;
    a.num_samples = batch_size_per_image;
    a.pos_cap = (int)((double)batch_size_per_image * positive_fraction);  // the reference's Python int(S * f)
    a.append_gt = append_gt ? 1 : 0;
    a.rule = rule;
    a.rowmax = static_cast<float*>(workspace);
    a.info = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + rowmax_bytes(sum_g));
    a.out_boxes = reinterpret_cast<float4*>(out_boxes);
    a.out_classes = out_gt_classes;
    a.out_gt_boxes = reinterpret_cast<float4*>(out_gt_boxes);
    a.out_matched = out_matched;
    a.out_src = out_src;
    a.out_count = out_count;
    a.out_num_fg = out_num_fg;
    a.underfull = underfull_flag;
    cudaStream_t st = as_stream(stream);
    // enough CTAs per image for p_stride proposals + up to 1024 appended gt boxes; larger images loop (CTA-uniform)
    const int64_t cand = p_stride + (append_gt ? std::min<int64_t>(sum_g, 1024) : 0);
    const unsigned gx = (unsigned)std::max<int64_t>(1, (cand + kLabelThreads - 1) / kLabelThreads);
    roi_sample_label_kernel<<<dim3(gx, (unsigned)n), kLabelThreads, 0, st>>>(a);
    DET_LAUNCH_OK("roi_sample_label_kernel");
    roi_sample_select_kernel<<<(unsigned)n, kSelectThreads, 0, st>>>(a);
    DET_LAUNCH_OK("roi_sample_select_kernel");
    return DET_OK;
}
