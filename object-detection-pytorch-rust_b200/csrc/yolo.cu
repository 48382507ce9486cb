// Grid / anchor detection-head decode (subsystem 1) for the two YOLO-style layouts named by the north star.
//
//  * det_yolo_decode_nms : S x S x (B*5+C) channels-last grid head.  ONE launch for the whole batch, one CTA per
//    image: coalesced 16-byte loads of the image's logits into shared memory, sigmoid/exp decode, conf x class
//    scores, score threshold with an order-preserving block-scan compaction, and the per-class NMS of
//    nms_small.cuh -- the candidates never leave shared memory.
//  (the dense anchor head decode lives in dense_decode.cu)
//
// No reference implementation exists for either (SURVEY.md section 8 row a15); the specification is
// oracle/ref_torch.py (yolo_decode, yolo_select_nms, dense_decode).
#include "nms_small.cuh"
#include "yolo_fast.cuh"

namespace det {

// candidates live in shared memory as (predictor << 16 | class) + score; boxes are looked up per predictor
struct YoloCandidates {
    const float4* pbox;
    const float* cscore;
    const uint32_t* cpc;
    __device__ __forceinline__ float4 box(int i) const { return pbox[cpc[i] >> 16]; }
    __device__ __forceinline__ float score(int i) const { return cscore[i]; }
    __device__ __forceinline__ int64_t cat(int i) const { return (int64_t)(cpc[i] & 0xffffu); }
};

constexpr int kYoloThreads = 512;
constexpr int kYoloMaxPred = 1024;
constexpr int kYoloMaxHead = 6144;

template <int CAP, typename HT = float>
__global__ void __launch_bounds__(kYoloThreads, 2)
yolo_decode_nms_kernel(const HT* __restrict__ head, const float2* __restrict__ priors, YoloParams prm,
                       float4* __restrict__ dense_boxes, float* __restrict__ dense_conf,
                       float* __restrict__ dense_scores, int64_t* __restrict__ det_flat,
                       float4* __restrict__ det_boxes, float* __restrict__ det_scores,
                       int32_t* __restrict__ det_count) {
    constexpr int T = kYoloThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Smem = SmallSmem<CAP, T>;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    unsigned char* extra = smem_raw + ((sizeof(Smem) + 15) / 16) * 16;
    const int S2 = prm.s * prm.s, B = prm.b, C = prm.c, ch = B * 5 + C, P = S2 * B, PC = P * C;
    float4* pbox = reinterpret_cast<float4*>(extra);
    float* cscore = reinterpret_cast<float*>(pbox + P);
    float* hs = cscore + CAP;
    uint32_t* cpc = reinterpret_cast<uint32_t*>(hs + ((S2 * ch + 3) & ~3));
    __shared__ int s_warp_tot[T / 32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int img = blockIdx.x;

    DET_MARK(0);
    // ---- stage this image's logits: coalesced 4-element loads over the aligned interior of its span, widened to fp32
    const int64_t g0 = (int64_t)img * S2 * ch, g1 = g0 + (int64_t)S2 * ch;
    const typename Head<HT>::vec* head4 = reinterpret_cast<const typename Head<HT>::vec*>(head);
    for (int64_t v = (g0 >> 2) + tid; v < ((g1 + 3) >> 2); v += T) {
        const int64_t base = v << 2;
        if (base >= g0 && base + 4 <= g1) {
            const float4 q = ld4_stream<HT>(head4 + v);
            float* d = hs + (base - g0);
            d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
        } else {
            for (int e = 0; e < 4; ++e)
                if (base + e >= g0 && base + e < g1) hs[base + e - g0] = ld1_stream(head + base + e);
        }
    }
    __syncthreads();
    DET_MARK(1);
    // ---- transcendentals in place, one logit per thread: sigmoid for x, y, conf and the class logits, exp for w, h
    for (int i = tid; i < S2 * ch; i += T) {
        const int k = i % ch;
        const float x = hs[i];
        float y;
        if (k < B * 5) {
            const int comp = k % 5;
            if (comp == 2 || comp == 3) {
                const float cl = (x > prm.scale_clamp) ? prm.scale_clamp : x;  // torch.clamp(max=): NaN stays NaN
                y = expf(cl);
            } else {
                y = sigmoidf_rn(x);
            }
        } else {
            y = sigmoidf_rn(x);
        }
        hs[i] = y;
    }
    __syncthreads();
    // ---- boxes per predictor
    for (int p = tid; p < P; p += T) {
        const int cell = p / B, bi = p - cell * B;
        const int row = cell / prm.s, col = cell - row * prm.s;
        const float* t = hs + cell * ch + bi * 5;
        const float2 pr = priors[bi];
        const float cx = (t[0] + (float)col) * prm.stride_x;
        const float cy = (t[1] + (float)row) * prm.stride_y;
        const float w = t[2] * pr.x, h = t[3] * pr.y;
        float4 bx = make_float4(cx - 0.5f * w, cy - 0.5f * h, cx + 0.5f * w, cy + 0.5f * h);
        if (prm.clip) {  // torch clamp(min=0,max=W): NaN stays NaN
            bx.x = min_nan(max_nan(bx.x, 0.f), prm.img_w); bx.z = min_nan(max_nan(bx.z, 0.f), prm.img_w);
            bx.y = min_nan(max_nan(bx.y, 0.f), prm.img_h); bx.w = min_nan(max_nan(bx.w, 0.f), prm.img_h);
        }
        pbox[p] = bx;
        if (dense_boxes) dense_boxes[(int64_t)img * P + p] = bx;
        if (dense_conf) dense_conf[(int64_t)img * P + p] = t[4];
    }
    DET_MARK(2);
    // ---- scores, threshold, order-preserving compaction: each thread owns a contiguous run of flat ids
    //      (predictor-major, class-minor) and walks it incrementally
    const int per = (PC + T - 1) / T;
    const int f0 = min(tid * per, PC), f1 = min(f0 + per, PC);
    const int p_start = f0 / C, c_start = f0 - p_start * C;
    int mine = 0;
    {
        int p = p_start, ci = c_start, cell = p / B, bi = p - cell * B;
        for (int f = f0; f < f1; ++f) {
            const float sc = hs[cell * ch + bi * 5 + 4] * hs[cell * ch + B * 5 + ci];
            mine += (sc > prm.score_thresh) ? 1 : 0;
            if (dense_scores) dense_scores[(int64_t)img * PC + f] = sc;
            if (++ci == C) {
                ci = 0;
                ++p;
                if (++bi == B) { bi = 0; ++cell; }
            }
        }
    }
    int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp_tot[wid] = incl;
    __syncthreads();  // also orders the pbox writes before the NMS reads
    int offset = incl - mine, cnt = 0;
    for (int w = 0; w < T / 32; ++w) {
        const int tot = s_warp_tot[w];
        if (w < wid) offset += tot;
        cnt += tot;
    }
    {
        int p = p_start, ci = c_start, cell = p / B, bi = p - cell * B;
        for (int f = f0; f < f1; ++f) {
            const float sc = hs[cell * ch + bi * 5 + 4] * hs[cell * ch + B * 5 + ci];
            if (sc > prm.score_thresh) {
                cpc[offset] = ((uint32_t)p << 16) | (uint32_t)ci;
                cscore[offset] = sc;
                ++offset;
            }
            if (++ci == C) {
                ci = 0;
                ++p;
                if (++bi == B) { bi = 0; ++cell; }
            }
        }
    }
    __syncthreads();
    DET_MARK(3);
    // ---- per-class NMS in shared memory
    const int cap_out = (int)min(prm.max_det, (int64_t)CAP);
    const YoloCandidates src{pbox, cscore, cpc};
    const int kept = small_nms_body<CAP, T>(sm, src, cnt, prm.thr_f, prm.mode, cap_out);
    const int nout = kept < 0 ? 0 : min(kept, cap_out);
    using KL = KeyLayout<kSmallIdxBits>;
    for (int j = tid; j < nout; j += T) {
        const int i = (int)KL::idx(sm.keys[j]);
        const uint32_t pc = cpc[i];
        const int64_t o = (int64_t)img * prm.max_det + j;
        const int64_t flat = (int64_t)(pc >> 16) * C + (int64_t)(pc & 0xffffu);
        if (prm.flat32) reinterpret_cast<int32_t*>(det_flat)[o] = (int32_t)flat;
        else det_flat[o] = flat;
        if (det_boxes) det_boxes[o] = pbox[pc >> 16];
        if (det_scores) det_scores[o] = cscore[i];
    }
    if (tid == 0) det_count[img] = nout;
    DET_MARK(15);
}

template <int CAP, typename T>
static int launch_yolo(const T* head, const float* priors, const YoloParams& prm, float* dense_boxes,
                       float* dense_conf, float* dense_scores, int64_t* det_flat, float* det_boxes, float* det_scores,
                       int32_t* det_count, cudaStream_t st) {
    const int S2 = prm.s * prm.s, ch = prm.b * 5 + prm.c, P = S2 * prm.b;
    size_t smem = ((sizeof(SmallSmem<CAP, kYoloThreads>) + 15) / 16) * 16;
    smem += sizeof(float4) * P + sizeof(float) * CAP + sizeof(float) * ((S2 * ch + 3) & ~3) + sizeof(uint32_t) * CAP;
    cudaError_t e = cudaFuncSetAttribute(yolo_decode_nms_kernel<CAP, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(yolo_decode_nms_kernel)");
    yolo_decode_nms_kernel<CAP, T><<<prm.n, kYoloThreads, smem, st>>>(
        head, reinterpret_cast<const float2*>(priors), prm, reinterpret_cast<float4*>(dense_boxes), dense_conf,
        dense_scores, det_flat, reinterpret_cast<float4*>(det_boxes), det_scores, det_count);
    DET_LAUNCH_OK("yolo_decode_nms_kernel");
    return DET_OK;
}

template <int MAXT, int MINB, int CS, int CB, int CC, typename T>
static int launch_yolo_fast(const T* head, const float* priors, const YoloParams& prm, float* dense_boxes,
                            float* dense_conf, float* dense_scores, int64_t* det_flat, float* det_boxes,
                            float* det_scores, int32_t* det_count, cudaStream_t st) {
    const int S2 = prm.s * prm.s, ch = prm.b * 5 + prm.c, P = S2 * prm.b;
    const FastLayout lay(S2, ch, P, prm.c);
    const int warps = prm.c > kFastMinWarps ? prm.c : kFastMinWarps;
    cudaError_t e = cudaFuncSetAttribute(yolo_fast_kernel<MAXT, MINB, CS, CB, CC, T>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(yolo_fast_kernel)");
    e = launch_pdl(yolo_fast_kernel<MAXT, MINB, CS, CB, CC, T>, dim3(prm.n), dim3(warps * 32), lay.bytes, st, head,
                   reinterpret_cast<const float2*>(priors), prm, reinterpret_cast<float4*>(dense_boxes), dense_conf,
                   dense_scores, det_flat, reinterpret_cast<float4*>(det_boxes), det_scores, det_count);
    if (e != cudaSuccess) return cuda_fail(e, "yolo_fast_kernel");
    return DET_OK;
}

}  // namespace det

using namespace det;

#ifdef DET_DEBUG_PHASES
extern "C" __attribute__((visibility("default"))) int det_debug_read_phases(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, det::g_phase_clock, sizeof(long long) * 32) == cudaSuccess ? 0 : -4;
}
#endif

// The entry points below have C linkage through their declarations in det_b200.h; the per-type implementation is a C++
// template.
template <typename T>
static int yolo_decode_nms_impl(const void* head_v, int n, int s, int b, int c, int img_h, int img_w, const float* priors,
                                float scale_clamp, int clip, float score_thresh, double iou_threshold, int mode,
                                float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                                int64_t* det_flat, float* det_boxes, float* det_scores, int32_t* det_count, void* stream,
                                int flat32) {
    DET_CHECK_ARG(n >= 0 && s >= 1 && b >= 1 && c >= 1 && max_det >= 1, "bad size");
    DET_CHECK_ARG(mode >= DET_NMS_AUTO && mode <= DET_NMS_OFFSET_TRICK, "unknown mode");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(head_v && priors && det_flat && det_count, "null pointer");
    const T* head = static_cast<const T*>(head_v);
    const int64_t P = (int64_t)s * s * b, PC = P * c, HS = (int64_t)s * s * (b * 5 + c);
    if (P > kYoloMaxPred || PC > 4096 || HS > kYoloMaxHead || c > 1024) {
        set_error("grid head too large for the fused kernel (limits: s*s*b <= 1024, s*s*b*c <= 4096, "
                  "s*s*(5b+c) <= 6144); use det_dense_decode_level + det_nms_batched");
        return DET_ERR_UNSUPPORTED;
    }
    if (!aligned_to(head, 4 * sizeof(T)) || (dense_boxes && !aligned16(dense_boxes)) || (det_boxes && !aligned16(det_boxes))) {
        set_error("head must be aligned to 4 elements, box outputs to 16 bytes");
        return DET_ERR_ALIGN;
    }
    YoloParams prm;
    prm.n = n; prm.s = s; prm.b = b; prm.c = c;
    prm.stride_x = (float)((double)img_w / (double)s);
    prm.stride_y = (float)((double)img_h / (double)s);
    prm.img_w = (float)img_w; prm.img_h = (float)img_h;
    prm.scale_clamp = scale_clamp; prm.score_thresh = score_thresh;
    prm.thr_f = float_threshold_below(iou_threshold);
    prm.clip = clip; prm.mode = mode; prm.max_det = max_det; prm.flat32 = flat32;
    cudaStream_t st = as_stream(stream);
    // small clipped grids (BASELINE configs[0]/[1]): one warp per class, no CTA-wide sort
    if (P <= kFastMaxP && c <= kFastMaxC && clip && FastLayout(s * s, b * 5 + c, (int)P, c).bytes <= 200 * 1024) {
        if (s == 7 && b == 2 && c == 20)  // BASELINE configs[0]/[1]: shape folded at compile time
            return launch_yolo_fast<640, 2, 7, 2, 20>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
        if (c <= 20)
            return launch_yolo_fast<640, 2, 0, 0, 0>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
        return launch_yolo_fast<1024, 1, 0, 0, 0>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
    }
    if (PC <= 1024)
        return launch_yolo<1024>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
    if (PC <= 2048)
        return launch_yolo<2048>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
    return launch_yolo<4096>(head, priors, prm, dense_boxes, dense_conf, dense_scores, det_flat, det_boxes, det_scores, det_count, st);
}

int det_yolo_decode_nms(const float* head, int n, int s, int b, int c, int img_h, int img_w, const float* priors,
                        float scale_clamp, int clip, float score_thresh, double iou_threshold, int mode,
                        float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                        int64_t* det_flat, float* det_boxes, float* det_scores, int32_t* det_count, void* stream) {
    return yolo_decode_nms_impl<float>(head, n, s, b, c, img_h, img_w, priors, scale_clamp, clip, score_thresh,
                                       iou_threshold, mode, dense_boxes, dense_conf, dense_scores, max_det, det_flat,
                                       det_boxes, det_scores, det_count, stream, 0);
}

int det_yolo_decode_nms_i32(const float* head, int n, int s, int b, int c, int img_h, int img_w, const float* priors,
                            float scale_clamp, int clip, float score_thresh, double iou_threshold, int mode,
                            float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                            int32_t* det_flat32, float* det_boxes, float* det_scores, int32_t* det_count, void* stream) {
    return yolo_decode_nms_impl<float>(head, n, s, b, c, img_h, img_w, priors, scale_clamp, clip, score_thresh,
                                       iou_threshold, mode, dense_boxes, dense_conf, dense_scores, max_det,
                                       reinterpret_cast<int64_t*>(det_flat32), det_boxes, det_scores, det_count, stream, 1);
}

int det_yolo_decode_nms_typed(const void* head, int head_dtype, int n, int s, int b, int c, int img_h, int img_w,
                              const float* priors, float scale_clamp, int clip, float score_thresh, double iou_threshold,
                              int mode, float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                              void* det_flat, int index_bytes, float* det_boxes, float* det_scores, int32_t* det_count,
                              void* stream) {
    DET_CHECK_ARG(index_bytes == 8 || index_bytes == 4, "index_bytes must be 8 or 4");
    DET_HEAD_DISPATCH(head_dtype, yolo_decode_nms_impl, head, n, s, b, c, img_h, img_w, priors, scale_clamp, clip,
                      score_thresh, iou_threshold, mode, dense_boxes, dense_conf, dense_scores, max_det,
                      static_cast<int64_t*>(det_flat), det_boxes, det_scores, det_count, stream, index_bytes == 4 ? 1 : 0);
}
