// FPN level assignment + ROIAlign / ROIPool over a feature pyramid in ONE launch (SURVEY.md section 8f rank 2).
//
// Replaces ROIPooler.forward (reference python/src/models/modules/roi_poolers.py:269-331): there, per level,
// nonzero(level == l) -> gather boxes -> torchvision roi_align -> index_put_ into a zero-filled output.  Here every
// output element (box, channel, bin) finds its own level: det_roi_levels evaluates Eqn.(1) of the FPN paper once per
// box (roi_poolers.py:121-131), and one kernel samples all levels -- no per-level launches, no gathers, no memset.
// The sampling arithmetic restates torchvision's roi_align (third-party, un-vendored; oracle = the installed
// torchvision CPU kernel): `aligned` shifts by half a pixel, sampling_ratio <= 0 means ceil(roi / bins) samples.
// ROIPool restates torchvision's roi_pool (max over the integer bins of the rounded box, first maximum wins).
// Features are fp32, bf16 or fp16 (DET_DTYPE_*): every element is widened to fp32 on load (exact), all arithmetic is
// the fp32 path, and the output is rounded once to the feature dtype -- bit-identical to the fp32 kernel fed f.float()
// followed by torch's .to(dtype), which is what torchvision's autocast rule for roi_align / roi_pool computes.
#include <algorithm>
#include <cfloat>

#include "common.cuh"

namespace det {

constexpr int kRoiMaxLevels = 8;

struct RoiLevelDev {
    const void* data;  // (N, C, H, W) of the feature dtype; in backward the level's fp32 gradient buffer
    int h, w;
    float scale;
};

// the arguments of every pyramid kernel, forward and backward (filled by roi_setup)
struct RoiArgs {
    RoiLevelDev lv[kRoiMaxLevels];
    int num_levels, c, out_h, out_w, sampling_ratio, aligned;
    int64_t m;
    const float4* boxes;
    const int32_t* batch_index;
    const int64_t* level;  // may be null when num_levels == 1
    void* io;              // (M, C, out_h, out_w) of the feature dtype: forward the output, backward grad_out (read)
};

__global__ void __launch_bounds__(256)
roi_levels_kernel(const float4* __restrict__ boxes, int64_t m, int min_level, int max_level, float canonical_box_size,
                  float canonical_level, int64_t* __restrict__ level_out) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= m) return;
    const float4 b = boxes[i];
    const float size = sqrtf(box_area(b));                                       // torch.sqrt(area)
    float lvl = floorf(canonical_level + log2f(size / canonical_box_size + 1e-8f));  // roi_poolers.py:123-125
    lvl = fminf(fmaxf(lvl, (float)min_level), (float)max_level);                  // torch.clamp (NaN: see below)
    if (lvl != lvl) lvl = (float)min_level;  // a NaN area would make torch's int64 cast undefined: pin it to level 0
    level_out[i] = (int64_t)lvl - min_level;
}

// torchvision bilinear_interpolate (roi_align_common / cuda kernel)
template <typename T>
__device__ __forceinline__ float bilinear(const T* __restrict__ plane, int H, int W, float y, float x) {
    if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) return 0.0f;
    if (y <= 0.0f) y = 0.0f;
    if (x <= 0.0f) x = 0.0f;
    int y_low = (int)y, x_low = (int)x, y_high, x_high;
    if (y_low >= H - 1) {
        y_high = y_low = H - 1;
        y = (float)y_low;
    } else {
        y_high = y_low + 1;
    }
    if (x_low >= W - 1) {
        x_high = x_low = W - 1;
        x = (float)x_low;
    } else {
        x_high = x_low + 1;
    }
    const float ly = y - (float)y_low, lx = x - (float)x_low, hy = 1.0f - ly, hx = 1.0f - lx;
    const float v1 = ld1(plane + y_low * W + x_low), v2 = ld1(plane + y_low * W + x_high);
    const float v3 = ld1(plane + y_high * W + x_low), v4 = ld1(plane + y_high * W + x_high);
    return hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
}

// One CTA per (box, group of kRoiChans channels).  The sample geometry of a box -- which feature rows / columns every
// sample touches and with which bilinear weights -- is separable and does not depend on the channel: the CTA first
// tabulates out_h*grid_h row taps and out_w*grid_w column taps in shared memory, then its threads walk the
// (channel, bin) outputs of the group; every sample costs two shared-memory tap loads, 4 global loads and a few
// multiply-adds.  Consecutive threads are consecutive output floats (fully coalesced stores) and neighbouring bins of
// one feature plane (reads fall into the same few rows).  Boxes whose tap tables would not fit take the direct path.
constexpr int kRoiChans = 32;
constexpr int kRoiTaps = 128;  // per axis: out_h * grid_h (resp. out_w * grid_w) must not exceed this

struct AxisTap {
    int lo, hi;
    float wlo, whi;  // both 0 when the sample lies outside [-1, size] (torchvision: contributes 0)
};

__device__ __forceinline__ AxisTap axis_tap(float v, int size) {
    AxisTap t;
    if (v < -1.0f || v > (float)size) {
        t.lo = t.hi = 0;
        t.wlo = t.whi = 0.0f;
        return t;
    }
    if (v <= 0.0f) v = 0.0f;
    int lo = (int)v, hi;
    if (lo >= size - 1) {
        hi = lo = size - 1;
        v = (float)lo;
    } else {
        hi = lo + 1;
    }
    const float l = v - (float)lo;
    t.lo = lo; t.hi = hi; t.wlo = 1.0f - l; t.whi = l;
    return t;
}

template <typename T>
__global__ void __launch_bounds__(256) roi_align_levels_kernel(const __grid_constant__ RoiArgs g) {
    __shared__ AxisTap s_ty[kRoiTaps], s_tx[kRoiTaps];
    const int64_t box = blockIdx.x;
    const int c0 = blockIdx.y * kRoiChans, nc = min(kRoiChans, g.c - c0);
    const int bins = g.out_h * g.out_w;
    const int l = g.level ? (int)g.level[box] : 0;
    const RoiLevelDev& L = g.lv[l];
    const float4 b = g.boxes[box];
    const float off = g.aligned ? 0.5f : 0.0f;
    const float x1 = b.x * L.scale - off, y1 = b.y * L.scale - off;
    float rw = b.z * L.scale - off - x1, rh = b.w * L.scale - off - y1;
    if (!g.aligned) {  // legacy: force malformed ROIs to be 1x1
        rw = fmaxf(rw, 1.0f);
        rh = fmaxf(rh, 1.0f);
    }
    const float bin_h = rh / (float)g.out_h, bin_w = rw / (float)g.out_w;
    const int gh = g.sampling_ratio > 0 ? g.sampling_ratio : (int)ceilf(rh / (float)g.out_h);
    const int gw = g.sampling_ratio > 0 ? g.sampling_ratio : (int)ceilf(rw / (float)g.out_w);
    const float count = fmaxf((float)(gh * gw), 1.0f);
    const int64_t plane_sz = (int64_t)L.h * L.w;
    const T* base = static_cast<const T*>(L.data) + ((int64_t)g.batch_index[box] * g.c + c0) * plane_sz;
    T* out = static_cast<T*>(g.io) + (box * g.c + c0) * bins;
    const bool tabulated = gh >= 0 && gw >= 0 && g.out_h * gh <= kRoiTaps && g.out_w * gw <= kRoiTaps;  // CTA-uniform
    if (tabulated) {
        for (int t = threadIdx.x; t < g.out_h * gh; t += 256) {
            const int ph = t / gh, iy = t - ph * gh;
            AxisTap a = axis_tap(y1 + (float)ph * bin_h + ((float)iy + 0.5f) * bin_h / (float)gh, L.h);
            a.lo *= L.w;
            a.hi *= L.w;
            s_ty[t] = a;
        }
        for (int t = threadIdx.x; t < g.out_w * gw; t += 256) {
            const int pw = t / gw, ix = t - pw * gw;
            s_tx[t] = axis_tap(x1 + (float)pw * bin_w + ((float)ix + 0.5f) * bin_w / (float)gw, L.w);
        }
        __syncthreads();
        for (int o = threadIdx.x; o < nc * bins; o += 256) {
            const int ch = o / bins, bin = o - ch * bins;
            const int ph = bin / g.out_w, pw = bin - ph * g.out_w;
            const T* plane = base + (int64_t)ch * plane_sz;
            float acc = 0.0f;
            for (int iy = 0; iy < gh; ++iy) {
                const AxisTap ty = s_ty[ph * gh + iy];
                const T* r0 = plane + ty.lo;
                const T* r1 = plane + ty.hi;
                for (int ix = 0; ix < gw; ++ix) {
                    const AxisTap tx = s_tx[pw * gw + ix];
                    // torchvision: w1*v1 + w2*v2 + w3*v3 + w4*v4 with w1 = hy*hx, w2 = hy*lx, w3 = ly*hx, w4 = ly*lx
                    acc += ty.wlo * tx.wlo * ld1(r0 + tx.lo) + ty.wlo * tx.whi * ld1(r0 + tx.hi) +
                           ty.whi * tx.wlo * ld1(r1 + tx.lo) + ty.whi * tx.whi * ld1(r1 + tx.hi);
                }
            }
            st_stream(out + o, acc / count);
        }
    } else {
        for (int o = threadIdx.x; o < nc * bins; o += 256) {
            const int ch = o / bins, bin = o - ch * bins;
            const int ph = bin / g.out_w, pw = bin - ph * g.out_w;
            const T* plane = base + (int64_t)ch * plane_sz;
            float acc = 0.0f;
            for (int iy = 0; iy < gh; ++iy) {
                const float y = y1 + (float)ph * bin_h + ((float)iy + 0.5f) * bin_h / (float)gh;
                for (int ix = 0; ix < gw; ++ix) {
                    const float x = x1 + (float)pw * bin_w + ((float)ix + 0.5f) * bin_w / (float)gw;
                    acc += bilinear(plane, L.h, L.w, y, x);
                }
            }
            st_stream(out + o, acc / count);
        }
    }
}

// Backward of the pyramid ROIAlign: grad_input[level] (N, C, H, W; fp32, zeroed by the caller) += the bilinear weights
// of every sample times grad_out / count -- the transpose of the forward gather, so the same tap tables drive 4 atomic
// adds per sample (what autograd does through torchvision's roi_align backward).  grad_out is read in its own dtype T.
template <typename T>
__global__ void __launch_bounds__(256) roi_align_levels_backward_kernel(const __grid_constant__ RoiArgs g) {
    __shared__ AxisTap s_ty[kRoiTaps], s_tx[kRoiTaps];
    const int64_t box = blockIdx.x;
    const int c0 = blockIdx.y * kRoiChans, nc = min(kRoiChans, g.c - c0);
    const int bins = g.out_h * g.out_w;
    const int l = g.level ? (int)g.level[box] : 0;
    const RoiLevelDev& L = g.lv[l];
    const int H = L.h, W = L.w;
    const float scale = L.scale;
    const float4 b = g.boxes[box];
    const float off = g.aligned ? 0.5f : 0.0f;
    const float x1 = b.x * scale - off, y1 = b.y * scale - off;
    float rw = b.z * scale - off - x1, rh = b.w * scale - off - y1;
    if (!g.aligned) {
        rw = fmaxf(rw, 1.0f);
        rh = fmaxf(rh, 1.0f);
    }
    const float bin_h = rh / (float)g.out_h, bin_w = rw / (float)g.out_w;
    const int gh = g.sampling_ratio > 0 ? g.sampling_ratio : (int)ceilf(rh / (float)g.out_h);
    const int gw = g.sampling_ratio > 0 ? g.sampling_ratio : (int)ceilf(rw / (float)g.out_w);
    const float count = fmaxf((float)(gh * gw), 1.0f);
    const int64_t plane_sz = (int64_t)H * W;
    float* base = static_cast<float*>(const_cast<void*>(L.data)) + ((int64_t)g.batch_index[box] * g.c + c0) * plane_sz;
    const T* go = static_cast<const T*>(g.io) + (box * g.c + c0) * bins;
    const bool tabulated = gh >= 0 && gw >= 0 && g.out_h * gh <= kRoiTaps && g.out_w * gw <= kRoiTaps;  // CTA-uniform
    if (tabulated) {
        for (int t = threadIdx.x; t < g.out_h * gh; t += 256) {
            const int ph = t / gh, iy = t - ph * gh;
            AxisTap a = axis_tap(y1 + (float)ph * bin_h + ((float)iy + 0.5f) * bin_h / (float)gh, H);
            a.lo *= W;
            a.hi *= W;
            s_ty[t] = a;
        }
        for (int t = threadIdx.x; t < g.out_w * gw; t += 256) {
            const int pw = t / gw, ix = t - pw * gw;
            s_tx[t] = axis_tap(x1 + (float)pw * bin_w + ((float)ix + 0.5f) * bin_w / (float)gw, W);
        }
        __syncthreads();
    }
    for (int o = threadIdx.x; o < nc * bins; o += 256) {
        const int ch = o / bins, bin = o - ch * bins;
        const int ph = bin / g.out_w, pw = bin - ph * g.out_w;
        float* plane = base + (int64_t)ch * plane_sz;
        const float gv = ld1(go + o) / count;
        for (int iy = 0; iy < gh; ++iy) {
            AxisTap ty;
            if (tabulated) {
                ty = s_ty[ph * gh + iy];
            } else {
                ty = axis_tap(y1 + (float)ph * bin_h + ((float)iy + 0.5f) * bin_h / (float)gh, H);
                ty.lo *= W;
                ty.hi *= W;
            }
            for (int ix = 0; ix < gw; ++ix) {
                const AxisTap tx = tabulated ? s_tx[pw * gw + ix]
                                             : axis_tap(x1 + (float)pw * bin_w + ((float)ix + 0.5f) * bin_w / (float)gw, W);
                const float w1 = ty.wlo * tx.wlo, w2 = ty.wlo * tx.whi, w3 = ty.whi * tx.wlo, w4 = ty.whi * tx.whi;
                if (w1 != 0.0f) atomicAdd(plane + ty.lo + tx.lo, w1 * gv);
                if (w2 != 0.0f) atomicAdd(plane + ty.lo + tx.hi, w2 * gv);
                if (w3 != 0.0f) atomicAdd(plane + ty.hi + tx.lo, w3 * gv);
                if (w4 != 0.0f) atomicAdd(plane + ty.hi + tx.hi, w4 * gv);
            }
        }
    }
}

// ROIPool bin p of an axis: rows (columns) [floor(p * bin), ceil((p + 1) * bin)) of the rounded box, clamped to the map
__device__ __forceinline__ int2 pool_bin(int p, float bin, int start, int size) {
    const int lo = (int)floorf((float)p * bin) + start, hi = (int)ceilf((float)(p + 1) * bin) + start;
    return make_int2(min(max(lo, 0), size), min(max(hi, 0), size));
}

// torchvision roi_pool over the pyramid: the grid and thread mapping of roi_align_levels_kernel (coalesced stores); the
// bin bounds depend on the box only and are tabulated once per CTA.  Each output is the max over its bin, scanned rows
// then columns with a strict `>` from -FLT_MAX: the first maximum wins and NaN is never taken.  An empty bin gives 0.
// argmax (may be null: inference) is the index h * W + w in the level plane, -1 when nothing was taken.
template <typename T>
__global__ void __launch_bounds__(256) roi_pool_levels_kernel(const __grid_constant__ RoiArgs g,
                                                              int32_t* __restrict__ argmax) {
    __shared__ int2 s_bh[kRoiTaps], s_bw[kRoiTaps];
    const int64_t box = blockIdx.x;
    const int c0 = blockIdx.y * kRoiChans, nc = min(kRoiChans, g.c - c0);
    const int bins = g.out_h * g.out_w;
    const int l = g.level ? (int)g.level[box] : 0;
    const RoiLevelDev& L = g.lv[l];
    const float4 b = g.boxes[box];
    // round() of the C library: halves away from zero; malformed boxes are forced to 1x1
    const int x0 = (int)roundf(b.x * L.scale), y0 = (int)roundf(b.y * L.scale);
    const int rw = max((int)roundf(b.z * L.scale) - x0 + 1, 1), rh = max((int)roundf(b.w * L.scale) - y0 + 1, 1);
    const float bin_h = (float)rh / (float)g.out_h, bin_w = (float)rw / (float)g.out_w;
    const bool tabulated = g.out_h <= kRoiTaps && g.out_w <= kRoiTaps;  // CTA-uniform
    if (tabulated) {
        for (int t = threadIdx.x; t < g.out_h; t += 256) s_bh[t] = pool_bin(t, bin_h, y0, L.h);
        for (int t = threadIdx.x; t < g.out_w; t += 256) s_bw[t] = pool_bin(t, bin_w, x0, L.w);
        __syncthreads();
    }
    const int64_t plane_sz = (int64_t)L.h * L.w;
    const T* base = static_cast<const T*>(L.data) + ((int64_t)g.batch_index[box] * g.c + c0) * plane_sz;
    const int64_t obase = (box * g.c + c0) * bins;
    T* out = static_cast<T*>(g.io) + obase;
    for (int o = threadIdx.x; o < nc * bins; o += 256) {
        const int ch = o / bins, bin = o - ch * bins;
        const int ph = bin / g.out_w, pw = bin - ph * g.out_w;
        const int2 by = tabulated ? s_bh[ph] : pool_bin(ph, bin_h, y0, L.h);
        const int2 bx = tabulated ? s_bw[pw] : pool_bin(pw, bin_w, x0, L.w);
        const T* plane = base + (int64_t)ch * plane_sz;
        float best = (by.y <= by.x || bx.y <= bx.x) ? 0.0f : -FLT_MAX;
        int arg = -1;
        for (int y = by.x; y < by.y; ++y) {
            for (int x = bx.x; x < bx.y; ++x) {
                const float v = ld1(plane + y * L.w + x);
                if (v > best) {
                    best = v;
                    arg = y * L.w + x;
                }
            }
        }
        st_stream(out + o, best);
        if (argmax) __stcs(argmax + obase + o, arg);
    }
}

// Backward of the pyramid ROIPool: grad_input[level][b, c, argmax] += grad_out for every output that took a value
// (argmax >= 0), one fp32 atomic each into the zeroed fp32 gradient buffers.  A flat grid-stride loop over M*C*bins.
template <typename T>
__global__ void __launch_bounds__(256) roi_pool_levels_backward_kernel(const __grid_constant__ RoiArgs g,
                                                                       const int32_t* __restrict__ argmax, int64_t total) {
    const int64_t bins = (int64_t)g.out_h * g.out_w;
    const T* go = static_cast<const T*>(g.io);
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
        const int a = argmax[i];
        if (a < 0) continue;
        const int64_t bc = i / bins;  // box * C + channel
        const int64_t box = bc / g.c;
        const int ch = (int)(bc - box * g.c);
        const int l = g.level ? (int)g.level[box] : 0;
        const RoiLevelDev& L = g.lv[l];
        float* plane = static_cast<float*>(const_cast<void*>(L.data)) +
                       ((int64_t)g.batch_index[box] * g.c + ch) * ((int64_t)L.h * L.w);
        atomicAdd(plane + a, ld1(go + i));
    }
}

// ---- launchers ------------------------------------------------------------------------------------------------------

static bool known_dtype(int d) { return d == DET_DTYPE_F32 || d == DET_DTYPE_BF16 || d == DET_DTYPE_F16; }

// The argument checks and the level table every pyramid launcher shares.  Returns DET_OK without filling `g` when
// m == 0 (the caller then launches nothing).  `boxes` is required unless !needs_boxes (the ROIPool backward reads the
// saved argmax instead).  `io`: the forward output or the backward grad_out.
static int roi_setup(RoiArgs& g, const det_feature_level_t* levels_host, int num_levels, int n, int c,
                     const float* boxes, bool needs_boxes, const int32_t* batch_index, const int64_t* level, int64_t m,
                     int out_h, int out_w, const void* io, int dtype) {
    DET_CHECK_ARG(num_levels >= 1 && num_levels <= kRoiMaxLevels && n >= 0 && c >= 1 && m >= 0 && out_h >= 1 && out_w >= 1,
                  "bad size");
    DET_CHECK_ARG(known_dtype(dtype), "unknown feature / gradient dtype");
    if (m == 0) return DET_OK;
    DET_CHECK_ARG(levels_host && (boxes || !needs_boxes) && batch_index && io && (level || num_levels == 1),
                  "null pointer");
    if (needs_boxes && !aligned16(boxes)) {
        set_error("boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    for (int l = 0; l < kRoiMaxLevels; ++l) {
        if (l < num_levels) {
            DET_CHECK_ARG(levels_host[l].data && levels_host[l].h >= 1 && levels_host[l].w >= 1, "bad level");
            g.lv[l].data = levels_host[l].data; g.lv[l].h = levels_host[l].h; g.lv[l].w = levels_host[l].w;
            g.lv[l].scale = levels_host[l].spatial_scale;
        } else {
            g.lv[l].data = nullptr; g.lv[l].h = 1; g.lv[l].w = 1; g.lv[l].scale = 1.f;
        }
    }
    DET_CHECK_ARG(m < (1ll << 31) && (c + kRoiChans - 1) / kRoiChans <= 65535, "too many boxes / channels");
    g.num_levels = num_levels; g.c = c; g.out_h = out_h; g.out_w = out_w; g.sampling_ratio = 0; g.aligned = 0;
    g.m = m; g.boxes = reinterpret_cast<const float4*>(boxes); g.batch_index = batch_index;
    g.level = num_levels > 1 ? level : nullptr; g.io = const_cast<void*>(io);
    return DET_OK;
}

static dim3 roi_grid(const RoiArgs& g) { return dim3((unsigned)g.m, (unsigned)((g.c + kRoiChans - 1) / kRoiChans)); }

template <typename T>
static int launch_align(const RoiArgs& g, cudaStream_t st) {
    roi_align_levels_kernel<T><<<roi_grid(g), 256, 0, st>>>(g);
    DET_LAUNCH_OK("roi_align_levels_kernel");
    return DET_OK;
}

template <typename T>
static int launch_align_backward(const RoiArgs& g, cudaStream_t st) {
    roi_align_levels_backward_kernel<T><<<roi_grid(g), 256, 0, st>>>(g);
    DET_LAUNCH_OK("roi_align_levels_backward_kernel");
    return DET_OK;
}

template <typename T>
static int launch_pool(const RoiArgs& g, int32_t* argmax, cudaStream_t st) {
    roi_pool_levels_kernel<T><<<roi_grid(g), 256, 0, st>>>(g, argmax);
    DET_LAUNCH_OK("roi_pool_levels_kernel");
    return DET_OK;
}

template <typename T>
static int launch_pool_backward(const RoiArgs& g, const int32_t* argmax, cudaStream_t st) {
    const int64_t total = g.m * g.c * g.out_h * g.out_w;
    const int64_t blocks = std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 32);
    roi_pool_levels_backward_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(g, argmax, total);
    DET_LAUNCH_OK("roi_pool_levels_backward_kernel");
    return DET_OK;
}

}  // namespace det

using namespace det;

extern "C" {

int det_roi_levels(const float* boxes, int64_t m, int min_level, int max_level, float canonical_box_size,
                   int canonical_level, int64_t* level_out, void* stream) {
    DET_CHECK_ARG(m >= 0 && min_level <= max_level && canonical_box_size > 0.f, "bad argument");
    if (m == 0) return DET_OK;
    DET_CHECK_ARG(boxes && level_out, "null pointer");
    if (!aligned16(boxes)) {
        set_error("boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    roi_levels_kernel<<<(unsigned)((m + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(boxes), m, min_level, max_level, canonical_box_size, (float)canonical_level, level_out);
    DET_LAUNCH_OK("roi_levels_kernel");
    return DET_OK;
}

int det_roi_align_levels_typed(const det_feature_level_t* levels_host, int num_levels, int n, int c, const float* boxes,
                               const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w,
                               int sampling_ratio, int aligned, void* out, int feat_dtype, void* stream) {
    RoiArgs g;
    const int rc = roi_setup(g, levels_host, num_levels, n, c, boxes, true, batch_index, level, m, out_h, out_w, out,
                             feat_dtype);
    if (rc != DET_OK || m == 0) return rc;
    g.sampling_ratio = sampling_ratio; g.aligned = aligned ? 1 : 0;
    DET_HEAD_DISPATCH(feat_dtype, launch_align, g, as_stream(stream));
}

int det_roi_align_levels(const det_feature_level_t* levels_host, int num_levels, int n, int c, const float* boxes,
                         const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w,
                         int sampling_ratio, int aligned, float* out, void* stream) {
    return det_roi_align_levels_typed(levels_host, num_levels, n, c, boxes, batch_index, level, m, out_h, out_w,
                                      sampling_ratio, aligned, out, DET_DTYPE_F32, stream);
}

int det_roi_align_levels_backward_typed(const det_feature_level_t* grad_levels_host, int num_levels, int n, int c,
                                        const float* boxes, const int32_t* batch_index, const int64_t* level, int64_t m,
                                        int out_h, int out_w, int sampling_ratio, int aligned, const void* grad_out,
                                        int grad_dtype, void* stream) {
    RoiArgs g;
    const int rc = roi_setup(g, grad_levels_host, num_levels, n, c, boxes, true, batch_index, level, m, out_h, out_w,
                             grad_out, grad_dtype);
    if (rc != DET_OK || m == 0) return rc;
    g.sampling_ratio = sampling_ratio; g.aligned = aligned ? 1 : 0;
    DET_HEAD_DISPATCH(grad_dtype, launch_align_backward, g, as_stream(stream));
}

int det_roi_align_levels_backward(const det_feature_level_t* grad_levels_host, int num_levels, int n, int c,
                                  const float* boxes, const int32_t* batch_index, const int64_t* level, int64_t m,
                                  int out_h, int out_w, int sampling_ratio, int aligned, const float* grad_out,
                                  void* stream) {
    return det_roi_align_levels_backward_typed(grad_levels_host, num_levels, n, c, boxes, batch_index, level, m, out_h,
                                               out_w, sampling_ratio, aligned, grad_out, DET_DTYPE_F32, stream);
}

int det_roi_pool_levels(const det_feature_level_t* levels_host, int num_levels, int n, int c, const float* boxes,
                        const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w, void* out,
                        int32_t* argmax, int feat_dtype, void* stream) {
    RoiArgs g;
    const int rc = roi_setup(g, levels_host, num_levels, n, c, boxes, true, batch_index, level, m, out_h, out_w, out,
                             feat_dtype);
    if (rc != DET_OK || m == 0) return rc;
    for (int l = 0; l < num_levels; ++l)  // argmax is an int32 index into a level plane
        DET_CHECK_ARG((int64_t)g.lv[l].h * g.lv[l].w <= INT32_MAX, "level plane too large for int32 argmax");
    DET_HEAD_DISPATCH(feat_dtype, launch_pool, g, argmax, as_stream(stream));
}

int det_roi_pool_levels_backward(const det_feature_level_t* grad_levels_host, int num_levels, int n, int c,
                                 const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w,
                                 const int32_t* argmax, const void* grad_out, int grad_dtype, void* stream) {
    RoiArgs g;
    const int rc = roi_setup(g, grad_levels_host, num_levels, n, c, nullptr, false, batch_index, level, m, out_h, out_w,
                             grad_out, grad_dtype);
    if (rc != DET_OK || m == 0) return rc;
    DET_CHECK_ARG(argmax, "null pointer");
    DET_HEAD_DISPATCH(grad_dtype, launch_pool_backward, g, argmax, as_stream(stream));
}

}  // extern "C"
