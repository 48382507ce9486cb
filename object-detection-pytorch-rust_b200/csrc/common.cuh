// Shared device/host helpers for libdet_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "../../include/det_b200.h"

namespace det {

// ---- host-side error plumbing -------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DET_CHECK_ARG(cond, msg)                       \
    do {                                               \
        if (!(cond)) {                                 \
            det::set_error("bad argument: %s", msg);   \
            return DET_ERR_BAD_ARG;                    \
        }                                              \
    } while (0)

#define DET_LAUNCH_OK(what)                                            \
    do {                                                               \
        cudaError_t e__ = cudaGetLastError();                          \
        if (e__ != cudaSuccess) return det::cuda_fail(e__, what);      \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline bool aligned_to(const void* p, unsigned bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1u)) == 0; }
int sm_count();

// calls FN<T>(args...) with T the element type named by DET_DTYPE_* `dtype`; an unknown code is DET_ERR_BAD_ARG before
// any CUDA call
#define DET_HEAD_DISPATCH(dtype, FN, ...)                                               \
    do {                                                                                \
        switch (dtype) {                                                                \
            case DET_DTYPE_F32: return FN<float>(__VA_ARGS__);                          \
            case DET_DTYPE_BF16: return FN<__nv_bfloat16>(__VA_ARGS__);                 \
            case DET_DTYPE_F16: return FN<__half>(__VA_ARGS__);                         \
        }                                                                               \
        det::set_error("bad argument: unknown head_dtype %d", (int)(dtype));            \
        return DET_ERR_BAD_ARG;                                                         \
    } while (0)

// largest float f with (double)f <= thr: then for every float v, ((double)v > thr) == (v > f).
// torchvision's CPU NMS compares the fp32 IoU against a *double* threshold.
static inline float float_threshold_below(double thr) {
    float f = (float)thr;
    if ((double)f > thr) f = nextafterf(f, -INFINITY);
    return f;
}

// ---- programmatic dependent launch (sm_90+) ------------------------------------------------------------------------
// A kernel launched through launch_pdl() may become resident while the previous kernel of its stream is still draining:
// its CTAs take SM slots as they free up and park in pdl_wait() -- which returns once the previous grid has completed and
// its memory is visible -- so the launch gap and the ramp of the next launch overlap the tail of this one.  In-stream
// semantics are unchanged as long as a kernel touches global memory only after pdl_wait().  pdl_trigger() (first
// statement of a kernel) lets the NEXT launch_pdl() kernel in the stream start that early; after a kernel that never
// triggers (any foreign kernel, a copy) the launch simply behaves like <<<>>>.  The edges survive stream capture.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- device helpers -----------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// std::max / std::min NaN behaviour (what torchvision's CPU NMS evaluates): (a<b)?b:a and (b<a)?b:a
__device__ __forceinline__ float max_std(float a, float b) { return (a < b) ? b : a; }
__device__ __forceinline__ float min_std(float a, float b) { return (b < a) ? b : a; }

// torch.minimum / torch.maximum / clamp NaN behaviour (propagate NaN): single FMNMX.NAN each
__device__ __forceinline__ float max_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float min_nan(float a, float b) {
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// streaming (evict-first) vector accesses for write-once / read-once data
__device__ __forceinline__ void st_stream(float4* p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
// an fp32 result stored as a 16-bit feature element, rounded to nearest even as torch's CUDA .to() rounds on sm_80+
__device__ __forceinline__ void st_stream(__nv_bfloat16* p, float v) {
    __stcs(reinterpret_cast<unsigned short*>(p), __bfloat16_as_ushort(__float2bfloat16_rn(v)));
}
__device__ __forceinline__ void st_stream(__half* p, float v) {
    __stcs(reinterpret_cast<unsigned short*>(p), __half_as_ushort(__float2half_rn(v)));
}
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }

// ---- head element types (DET_DTYPE_*): a bf16 or fp16 head is widened to fp32 as it is loaded -- exact -- and the
// kernels then run the same fp32 instructions as for an fp32 head.  Head<T>::vec holds 4 consecutive elements (16 bytes
// for fp32, 8 bytes for the 16-bit types; the element at the lower address is in the low half of each 32-bit word).
template <typename T> struct Head;
template <> struct Head<float> {
    using vec = float4;
    static __device__ __forceinline__ float4 f32(const float4 v) { return v; }
    static __device__ __forceinline__ float f32(const float x) { return x; }
    static __device__ __forceinline__ float4 pack(const float4 v) { return v; }
};
template <> struct Head<__nv_bfloat16> {
    using vec = uint2;
    static __device__ __forceinline__ float f32(const unsigned short b) { return __bfloat162float(__ushort_as_bfloat16(b)); }
    static __device__ __forceinline__ float f32(const __nv_bfloat16 x) { return __bfloat162float(x); }
    static __device__ __forceinline__ float4 f32(const uint2 v) {
        return make_float4(f32((unsigned short)(v.x & 0xffffu)), f32((unsigned short)(v.x >> 16)),
                           f32((unsigned short)(v.y & 0xffffu)), f32((unsigned short)(v.y >> 16)));
    }
    // 4 fp32 values rounded to nearest even, the lower-address element in the low half of each word
    static __device__ __forceinline__ uint2 pack(const float4 v) {
        auto b = [](float x) { return (unsigned)__bfloat16_as_ushort(__float2bfloat16_rn(x)); };
        return make_uint2(b(v.x) | (b(v.y) << 16), b(v.z) | (b(v.w) << 16));
    }
};
template <> struct Head<__half> {
    using vec = uint2;
    static __device__ __forceinline__ float f32(const unsigned short b) { return __half2float(__ushort_as_half(b)); }
    static __device__ __forceinline__ float f32(const __half x) { return __half2float(x); }
    static __device__ __forceinline__ float4 f32(const uint2 v) {
        return make_float4(f32((unsigned short)(v.x & 0xffffu)), f32((unsigned short)(v.x >> 16)),
                           f32((unsigned short)(v.y & 0xffffu)), f32((unsigned short)(v.y >> 16)));
    }
    static __device__ __forceinline__ uint2 pack(const float4 v) {
        auto h = [](float x) { return (unsigned)__half_as_ushort(__float2half_rn(x)); };
        return make_uint2(h(v.x) | (h(v.y) << 16), h(v.z) | (h(v.w) << 16));
    }
};
// 4 consecutive head elements as fp32: streaming (read-once) and plain (re-read) forms
template <typename T>
__device__ __forceinline__ float4 ld4_stream(const typename Head<T>::vec* p) { return Head<T>::f32(__ldcs(p)); }
template <typename T>
__device__ __forceinline__ float4 ld4(const typename Head<T>::vec* p) { return Head<T>::f32(*p); }
// 4 fp32 results stored as 4 consecutive head elements (streaming), each rounded once as st_stream rounds one
template <typename T>
__device__ __forceinline__ void st4_stream(typename Head<T>::vec* p, const float4 v) { __stcs(p, Head<T>::pack(v)); }
// one head element as fp32
__device__ __forceinline__ float ld1_stream(const float* p) { return __ldcs(p); }
template <typename T>
__device__ __forceinline__ float ld1_stream(const T* p) {
    return Head<T>::f32(__ldcs(reinterpret_cast<const unsigned short*>(p)));
}
template <typename T>
__device__ __forceinline__ float ld1(const T* p) { return Head<T>::f32(*p); }
// 4-element group q of a (rows, groups * 4) delta tensor as fp32: one vector load when the base is aligned to 4
// elements (vec), four scalar loads otherwise
template <typename T>
__device__ __forceinline__ float4 ld_group(const void* base, int vec, int64_t q) {
    if (vec) return ld4<T>(static_cast<const typename Head<T>::vec*>(base) + q);
    const T* p = static_cast<const T*>(base) + q * 4;
    return make_float4(ld1(p), ld1(p + 1), ld1(p + 2), ld1(p + 3));
}

// 1 / (1 + e^-x): __frcp_rn is the correctly rounded reciprocal, i.e. bit-identical to the IEEE quotient 1.0f / d
__device__ __forceinline__ float sigmoidf_rn(float x) { return __frcp_rn(1.0f + expf(-x)); }

__device__ __forceinline__ float box_area(const float4 b) { return (b.z - b.x) * (b.w - b.y); }

// ---- box codec (Box2BoxTransform) ----------------------------------------------------------------
struct CodecWeights {
    float wx, wy, ww, wh;
};

// reference apply_deltas on one (anchor, delta) pair; operation order of box_regression.py:90-114
__device__ __forceinline__ float4 decode_delta(const float4 box, const float4 d, const CodecWeights wt,
                                               float scale_clamp) {
    const float w = box.z - box.x, h = box.w - box.y;
    const float cx = box.x + 0.5f * w, cy = box.y + 0.5f * h;
    const float dx = d.x / wt.wx, dy = d.y / wt.wy;
    float dw = d.z / wt.ww, dh = d.w / wt.wh;
    dw = (dw > scale_clamp) ? scale_clamp : dw;  // torch.clamp(max=): NaN stays NaN
    dh = (dh > scale_clamp) ? scale_clamp : dh;
    const float pcx = dx * w + cx, pcy = dy * h + cy;
    const float pw = expf(dw) * w, ph = expf(dh) * h;
    return make_float4(pcx - 0.5f * pw, pcy - 0.5f * ph, pcx + 0.5f * pw, pcy + 0.5f * ph);
}

// reference get_deltas on one (src, tgt) pair; operation order of box_regression.py:53-69
__device__ __forceinline__ float4 encode_delta(const float4 s, const float4 t, const CodecWeights wt) {
    const float sw = s.z - s.x, sh = s.w - s.y;
    const float scx = s.x + 0.5f * sw, scy = s.y + 0.5f * sh;
    const float tw = t.z - t.x, th = t.w - t.y;
    const float tcx = t.x + 0.5f * tw, tcy = t.y + 0.5f * th;
    return make_float4(wt.wx * (tcx - scx) / sw, wt.wy * (tcy - scy) / sh, wt.ww * logf(tw / sw),
                       wt.wh * logf(th / sh));
}

// 32-bit key that sorts ASCENDING into torch's descending-score order:
// NaN first (all NaNs tie), then +inf ... -inf, -0 == +0 tie.
__device__ __forceinline__ uint32_t score_desc_key(float s) {
    if (s != s) return 0u;
    uint32_t u = __float_as_uint(s);
    if (u == 0x80000000u) u = 0u;
    uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ~asc;
}

// exact greedy-NMS predicate of torchvision's CPU kernel: does kept box `a` suppress candidate `b`?
//     ovr = inter / (area_a + area_b - inter);  suppressed iff (double)ovr > threshold
// thr_f = float_threshold_below(double threshold), so the comparison is (ovr > thr_f) in fp32.
// The IEEE division is only executed for the knife-edge cases.  With t = fl(thr_f*denom) normal and thr_f normal and
// positive (hence denom > 0, |t/(thr_f*denom) - 1| <= 2^-24):
//   inter > fl(t*(1+2^-20))  =>  inter/denom > thr_f*(1+2^-21) >= nextafter(thr_f)  =>  fl(inter/denom) > thr_f
//   inter < fl(t*(1-17*2^-24)) =>  inter/denom < thr_f                              =>  fl(inter/denom) <= thr_f
// (rounding is monotone).  Everything else -- zero intersection, NaN/Inf, denormal or non-positive threshold or
// denominator, and the band in between -- takes the exact path, so the result is bit-identical to the plain formula.
// the exact IEEE quotient test; kept out of line so that the compiler cannot speculate the division ahead of the
// cheap guards in nms_suppresses (it is needed only for knife-edge pairs)
static __device__ __noinline__ bool nms_exact_ratio_gt(float inter, float denom, float thr_f) { return inter / denom > thr_f; }

// NONAN: the caller guarantees that no coordinate of either box is NaN; then std::max/min and FMNMX agree (the sign
// of a zero cannot change w, h) and the six selects become single FMNMX instructions.
template <bool NONAN>
__device__ __forceinline__ bool nms_suppresses(const float4 a, float area_a, const float4 b, float area_b,
                                               float thr_f) {
    float xx1, yy1, xx2, yy2, w, h;
    if (NONAN) {
        xx1 = fmaxf(a.x, b.x); yy1 = fmaxf(a.y, b.y);
        xx2 = fminf(a.z, b.z); yy2 = fminf(a.w, b.w);
        w = fmaxf(0.0f, xx2 - xx1); h = fmaxf(0.0f, yy2 - yy1);
    } else {
        xx1 = max_std(a.x, b.x); yy1 = max_std(a.y, b.y);
        xx2 = min_std(a.z, b.z); yy2 = min_std(a.w, b.w);
        w = max_std(0.0f, xx2 - xx1); h = max_std(0.0f, yy2 - yy1);
    }
    const float inter = w * h;
    const float denom = area_a + area_b - inter;
    if (inter == 0.0f)  // 0/denom is +-0 (or NaN for denom 0/NaN): suppresses only under a negative threshold
        return (thr_f < 0.0f) && (denom == denom) && (denom != 0.0f);
    const float t = thr_f * denom;
    if (thr_f > 1e-30f && t > 1e-30f && t < 1e30f) {
        if (inter > t * 1.000001f) return true;
        if (inter < t * 0.999999f) return false;
    }
    return nms_exact_ratio_gt(inter, denom, thr_f);
}

// reference pairwise IoU of one pair (boxes.py:173-214), NaN-propagating min/max like torch
__device__ __forceinline__ float pair_intersection(const float4 a, const float4 b) {
    float w = max_nan(min_nan(a.z, b.z) - max_nan(a.x, b.x), 0.0f);
    float h = max_nan(min_nan(a.w, b.w) - max_nan(a.y, b.y), 0.0f);
    return w * h;
}
__device__ __forceinline__ float pair_iou(const float4 a, float area_a, const float4 b, float area_b) {
    float inter = pair_intersection(a, b);
    return (inter > 0.0f) ? inter / (area_a + area_b - inter) : 0.0f;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Optional phase timeline (build with -DDET_DEBUG_PHASES): block 0 / thread 0 stamps clock64() at DET_MARK(i).
#ifdef DET_DEBUG_PHASES
static __device__ long long g_phase_clock[32];  // one copy per translation unit (no -rdc)
static __device__ long long g_phase_block[64][16];  // the same stamps for the first 64 blocks (marks 0..15)
#define DET_MARK(i)                                                     \
    do {                                                                \
        if (blockIdx.x == 0 && threadIdx.x == 0) g_phase_clock[i] = clock64(); \
        if (blockIdx.x < 64 && threadIdx.x == 0) g_phase_block[blockIdx.x][(i) & 15] = clock64(); \
    } while (0)
// accumulating form for phases inside loops: DET_ACC_BEGIN() once, DET_ACC(i) adds the cycles since the previous stamp
static __device__ long long g_phase_acc[16];
#define DET_ACC_BEGIN() long long det_acc_t = clock64()
#define DET_ACC(i)                                        \
    do {                                                  \
        if (blockIdx.x == 0 && threadIdx.x == 0) {        \
            const long long det_acc_n = clock64();        \
            g_phase_acc[i] += det_acc_n - det_acc_t;      \
            det_acc_t = det_acc_n;                        \
        }                                                 \
    } while (0)
#else
#define DET_MARK(i) do { } while (0)
#define DET_ACC_BEGIN() do { } while (0)
#define DET_ACC(i) do { } while (0)
#endif

#endif  // __CUDACC__
}  // namespace det
