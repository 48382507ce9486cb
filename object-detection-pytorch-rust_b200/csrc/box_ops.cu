// Box math kernels: pairwise overlap (IoU / IoA / intersection), matched IoU, the R-CNN box codec
// (apply_deltas / get_deltas), grid-anchor synthesis and the NCHW-native RPN head decode.
//
// Reference behaviour reproduced (paths relative to the reference root):
//   python/src/structures/boxes.py:173-258            pairwise_intersection / iou / ioa / matched_boxlist_iou
//   python/src/models/components/box_regression.py:33-115   get_deltas / apply_deltas
//   python/src/models/modules/anchor_generators.py:31-56,158-179   grid anchors, order (h, w, a)
//   python/src/models/rpn.py:270-284, 330-348          layout change + _decode_proposals
// All arithmetic is IEEE fp32 in the reference's operation order (the library is built with -fmad=false).
#include "common.cuh"

namespace det {

// ------------------------------------------------------------------------------------------------
// pairwise overlap: out[i*m + j] for boxes1[i], boxes2[j].
// HBM-write bound (4 B per pair).  One CTA owns a 32-row x 1024-column tile: the 32 row boxes (+areas)
// are staged in shared memory and broadcast, each thread keeps its 4 column boxes (+areas) in registers
// and emits one 16-byte streaming store per row => every warp writes 512 contiguous bytes per row.
// ------------------------------------------------------------------------------------------------
constexpr int kPairRows = 32;
constexpr int kPairThreads = 256;
constexpr int kPairCols = kPairThreads * 4;

template <int MODE>
__device__ __forceinline__ float overlap_one(const float4 a, float area_a, const float4 b, float area_b) {
    if (MODE == DET_OVERLAP_IOU) return pair_iou(a, area_a, b, area_b);
    float inter = pair_intersection(a, b);
    if (MODE == DET_OVERLAP_IOA) return (inter > 0.0f) ? inter / area_b : 0.0f;
    return inter;
}

// Measured (profiles/README.md, r02): 20 000 x 20 000 boxes, 5 % of the pairs intersecting: 377 us = 0.65 of the copy peak,
// 368 M warp-instructions at 89 % issue utilisation -- the IEEE quotient runs in ~3 of 4 (warp, row, column) steps with a
// lane or two active.  No pair intersecting: 242 us = the write roofline.  A variant that defers the quotients (mask pass,
// pooled exact evaluation into a shared-memory patch) was built and measured: 367 us at 5 %, 496 us at 31 % (406 us here),
// 272 us at 0 % -- the bookkeeping costs what the divergence did, so the in-line form stays.
template <int MODE, bool VEC>
__global__ void __launch_bounds__(kPairThreads)
pairwise_overlap_kernel(const float4* __restrict__ b1, int64_t n, const float4* __restrict__ b2, int64_t m,
                        float* __restrict__ out) {
    __shared__ float4 s_box[kPairRows];
    __shared__ float s_area[kPairRows];
    const int64_t row0 = (int64_t)blockIdx.y * kPairRows;
    const int64_t col0 = (int64_t)blockIdx.x * kPairCols + (int64_t)threadIdx.x * 4;
    const int rows = (int)min((int64_t)kPairRows, n - row0);
    if (threadIdx.x < rows) {
        float4 b = b1[row0 + threadIdx.x];
        s_box[threadIdx.x] = b;
        s_area[threadIdx.x] = box_area(b);
    }
    float4 cb[4];
    float ca[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // out-of-range columns read a dummy box; their results are never stored
        cb[k] = (col0 + k < m) ? b2[col0 + k] : make_float4(0.f, 0.f, 0.f, 0.f);
        ca[k] = box_area(cb[k]);
    }
    __syncthreads();
    if (col0 >= m) return;
    for (int r = 0; r < rows; ++r) {
        const float4 a = s_box[r];
        const float aa = s_area[r];
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = overlap_one<MODE>(a, aa, cb[k], ca[k]);
        float* dst = out + (row0 + r) * m + col0;
        if (VEC) {
            st_stream(reinterpret_cast<float4*>(dst), make_float4(v[0], v[1], v[2], v[3]));
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (col0 + k < m) st_stream(dst + k, v[k]);
        }
    }
}

template <int MODE>
static int launch_pairwise(const float* b1, int64_t n, const float* b2, int64_t m, float* out, cudaStream_t st) {
    dim3 grid((unsigned)((m + kPairCols - 1) / kPairCols), (unsigned)((n + kPairRows - 1) / kPairRows));
    const bool vec = (m % 4 == 0) && aligned16(out);
    auto p1 = reinterpret_cast<const float4*>(b1);
    auto p2 = reinterpret_cast<const float4*>(b2);
    if (vec)
        pairwise_overlap_kernel<MODE, true><<<grid, kPairThreads, 0, st>>>(p1, n, p2, m, out);
    else
        pairwise_overlap_kernel<MODE, false><<<grid, kPairThreads, 0, st>>>(p1, n, p2, m, out);
    DET_LAUNCH_OK("pairwise_overlap_kernel");
    return DET_OK;
}

__global__ void matched_iou_kernel(const float4* __restrict__ b1, const float4* __restrict__ b2, int64_t n,
                                   float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 a = b1[i], b = b2[i];
    // boxes.py:251-257: lt=max, rb=min, (rb-lt).clamp(min=0), no empty guard
    float inter = pair_intersection(a, b);
    out[i] = inter / (box_area(a) + box_area(b) - inter);
}

// ------------------------------------------------------------------------------------------------
// box codec
// ------------------------------------------------------------------------------------------------
// CodecWeights, decode_delta, encode_delta: common.cuh (shared with roi_detect.cu and the loss kernels)

__global__ void apply_deltas_kernel(const float4* __restrict__ deltas, const float4* __restrict__ boxes,
                                    int64_t total, int k, CodecWeights wt, float scale_clamp,
                                    float4* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    out[i] = decode_delta(boxes[i / k], deltas[i], wt, scale_clamp);
}

// backward of apply_deltas (what autograd produces for box_regression.py:87-115): one thread per box row, its k
// class-specific deltas in a loop so that the gradient of the box itself (summed over k) needs no atomics.
// torch.clamp(max=) passes the gradient where the input is <= the bound.
__global__ void apply_deltas_backward_kernel(const float4* __restrict__ deltas, const float4* __restrict__ boxes,
                                             const float4* __restrict__ grad_out, int64_t m, int k, CodecWeights wt,
                                             float scale_clamp, float4* __restrict__ grad_deltas,
                                             float4* __restrict__ grad_boxes) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float4 box = boxes[i];
    const float w = box.z - box.x, h = box.w - box.y;
    float4 gb = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < k; ++c) {
        const float4 d = deltas[i * k + c], g = grad_out[i * k + c];
        const float dx = d.x / wt.wx, dy = d.y / wt.wy;
        const float dw_raw = d.z / wt.ww, dh_raw = d.w / wt.wh;
        const float ew = expf((dw_raw > scale_clamp) ? scale_clamp : dw_raw);
        const float eh = expf((dh_raw > scale_clamp) ? scale_clamp : dh_raw);
        const float gcx = g.x + g.z, gcy = g.y + g.w;                   // d/d pred_ctr
        const float gpw = 0.5f * (g.z - g.x), gph = 0.5f * (g.w - g.y);  // d/d pred_w, pred_h
        if (grad_deltas)
            grad_deltas[i * k + c] = make_float4(gcx * w / wt.wx, gcy * h / wt.wy,
                                                 (dw_raw <= scale_clamp) ? gpw * ew * w / wt.ww : 0.0f,
                                                 (dh_raw <= scale_clamp) ? gph * eh * h / wt.wh : 0.0f);
        // pred_ctr = dx * w + (x1 + 0.5 w), pred_w = e^dw * w, w = x2 - x1
        gb.x += gcx * (0.5f - dx) - gpw * ew;
        gb.z += gcx * (0.5f + dx) + gpw * ew;
        gb.y += gcy * (0.5f - dy) - gph * eh;
        gb.w += gcy * (0.5f + dy) + gph * eh;
    }
    if (grad_boxes) grad_boxes[i] = gb;
}

__global__ void get_deltas_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, int64_t m,
                                  CodecWeights wt, float4* __restrict__ out, int32_t* __restrict__ invalid) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float4 s = src[i];
    out[i] = encode_delta(s, tgt[i], wt);
    if (!((s.z - s.x) > 0.0f) && invalid) *invalid = 1;
}

// ------------------------------------------------------------------------------------------------
// anchors
// ------------------------------------------------------------------------------------------------
// torch.arange(offset*stride, size*stride, step=stride, dtype=float32): value_i = float(start + i*step),
// evaluated in double (anchor_generators.py:45-50).
__device__ __forceinline__ float grid_shift(int i, int stride, float offset) {
    return (float)((double)offset * (double)stride + (double)i * (double)stride);
}

__global__ void grid_anchors_kernel(const float4* __restrict__ cell, int a, int h, int w, int stride, float offset,
                                    float4* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)h * w * a) return;
    const int ai = (int)(i % a);
    const int64_t loc = i / a;
    const float sx = grid_shift((int)(loc % w), stride, offset), sy = grid_shift((int)(loc / w), stride, offset);
    const float4 c = cell[ai];
    out[i] = make_float4(sx + c.x, sy + c.y, sx + c.z, sy + c.w);
}

// ------------------------------------------------------------------------------------------------
// RPN head decode straight from the conv layout.
// objectness (n,a,h,w), deltas (n,a*4,h,w)  ->  logits (n, hw*a) and proposals (n, hw*a, 4), order (h,w,a).
// A thread owns V consecutive spatial positions of one image: every plane read is a coalesced (V=4: 16-byte)
// load along the contiguous hw axis, the anchor is synthesised from (y, x, a), and the A boxes of a position are
// written back-to-back so a warp's stores cover one contiguous span.  The (n,hw*a[,4]) transposed copies that
// rpn.py:273/282 materialise never exist.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxCellAnchors = 16;

template <int V, typename T = float>
__global__ void __launch_bounds__(256)
rpn_decode_level_kernel(const T* __restrict__ obj, const T* __restrict__ deltas, int n, int a, int h, int w,
                        int stride, float offset, const float4* __restrict__ cell, CodecWeights wt,
                        float scale_clamp, float* __restrict__ logits_out, float4* __restrict__ boxes_out,
                        int64_t out_img_stride, int64_t out_offset) {
    __shared__ float4 s_cell[kMaxCellAnchors];
    if (threadIdx.x < a) s_cell[threadIdx.x] = cell[threadIdx.x];
    __syncthreads();
    const int64_t hw = (int64_t)h * w;
    const int64_t groups = (hw + V - 1) / V;
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int img = blockIdx.y;
    if (g >= groups) return;
    const int64_t p0 = g * V;
    const T* obj_img = obj + (int64_t)img * a * hw;
    const T* del_img = deltas + (int64_t)img * a * 4 * hw;
    float* lo = logits_out + (int64_t)img * out_img_stride + out_offset;
    float4* bo = boxes_out + (int64_t)img * out_img_stride + out_offset;
    float sx[V], sy[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int64_t p = p0 + v;
        sx[v] = grid_shift((int)(p % w), stride, offset);
        sy[v] = grid_shift((int)(p / w), stride, offset);
    }
    for (int ai = 0; ai < a; ++ai) {
        float lg[V], d[4][V];
        if (V == 4) {
            using HV = typename Head<T>::vec;
            const float4 l4 = ld4_stream<T>(reinterpret_cast<const HV*>(obj_img + ai * hw + p0));
            lg[0] = l4.x; lg[1] = l4.y; lg[2] = l4.z; lg[3] = l4.w;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float4 q = ld4_stream<T>(reinterpret_cast<const HV*>(del_img + (ai * 4 + c) * hw + p0));
                d[c][0] = q.x; d[c][1] = q.y; d[c][2] = q.z; d[c][3] = q.w;
            }
        } else {
            lg[0] = ld1_stream(obj_img + ai * hw + p0);
#pragma unroll
            for (int c = 0; c < 4; ++c) d[c][0] = ld1_stream(del_img + (ai * 4 + c) * hw + p0);
        }
        const float4 ca = s_cell[ai];
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 anchor = make_float4(sx[v] + ca.x, sy[v] + ca.y, sx[v] + ca.z, sy[v] + ca.w);
            const float4 box = decode_delta(anchor, make_float4(d[0][v], d[1][v], d[2][v], d[3][v]), wt, scale_clamp);
            const int64_t o = (p0 + v) * a + ai;
            lo[o] = lg[v];
            bo[o] = box;
        }
    }
}


// ---- all pyramid levels in ONE launch, outputs staged through shared memory --------------------------------------------
// One warp owns a tile of 128 consecutive positions of one (level, image): every lane loads its 4 positions of the A
// objectness planes and 4A delta planes with 16-byte loads (5A independent loads in flight), decodes, and parks the
// results in the warp's shared-memory slab in output order (position-major, anchor-minor); the warp then writes the
// slab -- one contiguous span of 128*A boxes and logits -- with fully coalesced stores.  Small levels ride along with
// the big one instead of paying their own launch, ramp and tail.  (Issuing the 15 loads of all three anchors before the
// first decode -- A as a template parameter, 100 registers -- was measured: 35.1 vs 33.1 us per 64 images, 107.0 vs
// 105.5 us per 256; the bytes in flight are not what holds this kernel at 0.74 of the copy peak.  Rejected.  So was an
// odd slab pitch (4A+1 entries per lane) that removes the 10-way bank conflict ncu reports on the slab stores: 33.3 vs
// 33.1 us per 64 images, 113.0 vs 105.5 us per 256.)
constexpr int kRpnFlatMaxLevels = 8;
constexpr int kRpnFlatMaxA = 4;
constexpr int kRpnTilePos = 128;
constexpr int kRpnFlatWarps = 8;

struct RpnLevelDev {
    const void* obj;     // elements of the kernel's head type T
    const void* deltas;
    const float4* cell;
    int w, hw, tiles;  // tiles of 128 positions per image
    int stride, vec;   // vec: planes are whole 4-element vectors (hw % 4 == 0, heads aligned to 4 elements)
    int64_t out_offset;
};

struct RpnFlatArgs {
    RpnLevelDev lv[kRpnFlatMaxLevels];
    long long tile_begin[kRpnFlatMaxLevels + 1];  // first flat tile of each level
    int num_levels, n, a;
    float offset, scale_clamp;
    CodecWeights wt;
    int64_t out_img_stride;
    float* logits_out;
    float4* boxes_out;
};

template <typename T = float>
__global__ void __launch_bounds__(kRpnFlatWarps * 32) rpn_decode_flat_kernel(const __grid_constant__ RpnFlatArgs g) {
    using HV = typename Head<T>::vec;
    extern __shared__ __align__(16) unsigned char rpn_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long tile = (long long)blockIdx.x * kRpnFlatWarps + wid;
    if (tile >= g.tile_begin[g.num_levels]) return;  // warp-uniform
    int l = 0;
#pragma unroll
    for (int q = 1; q < kRpnFlatMaxLevels; ++q)
        if (q < g.num_levels && tile >= g.tile_begin[q]) l = q;
    const RpnLevelDev& L = g.lv[l];
    const int A = g.a;
    const long long local = tile - g.tile_begin[l];
    const int img = (int)(local / L.tiles), t = (int)(local - (long long)img * L.tiles);
    const int pos0 = t * kRpnTilePos, npos = min(kRpnTilePos, L.hw - pos0);
    float4* s_box = reinterpret_cast<float4*>(rpn_smem) + (size_t)wid * kRpnTilePos * A;
    float* s_log = reinterpret_cast<float*>(reinterpret_cast<float4*>(rpn_smem) + (size_t)kRpnFlatWarps * kRpnTilePos * A) +
                   (size_t)wid * kRpnTilePos * A;
    const int p0 = pos0 + lane * 4;
    if (lane * 4 < npos) {  // vec levels (hw % 4 == 0): a lane's 4 positions are all inside or all outside
        const T* obj_img = static_cast<const T*>(L.obj) + (int64_t)img * A * L.hw + p0;
        const T* del_img = static_cast<const T*>(L.deltas) + (int64_t)img * A * 4 * L.hw + p0;
        float sx[4], sy[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int p = p0 + v;
            sx[v] = grid_shift(p % L.w, L.stride, g.offset);
            sy[v] = grid_shift(p / L.w, L.stride, g.offset);
        }
        for (int ai = 0; ai < A; ++ai) {
            float4 l4, q[4];
            if (L.vec) {
                l4 = ld4_stream<T>(reinterpret_cast<const HV*>(obj_img + (int64_t)ai * L.hw));
#pragma unroll
                for (int c = 0; c < 4; ++c) q[c] = ld4_stream<T>(reinterpret_cast<const HV*>(del_img + (int64_t)(ai * 4 + c) * L.hw));
            } else {
                // a level whose planes are not 16-byte tiles (h*w not a multiple of 4, e.g. the 7x7 level of a 448^2
                // pyramid, or an unaligned view): scalar loads, positions past the plane read as 0 and are never written
                auto ld4s = [&](const T* pl) {
                    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p0 + 0 < L.hw) r.x = ld1(pl + 0);
                    if (p0 + 1 < L.hw) r.y = ld1(pl + 1);
                    if (p0 + 2 < L.hw) r.z = ld1(pl + 2);
                    if (p0 + 3 < L.hw) r.w = ld1(pl + 3);
                    return r;
                };
                l4 = ld4s(obj_img + (int64_t)ai * L.hw);
#pragma unroll
                for (int c = 0; c < 4; ++c) q[c] = ld4s(del_img + (int64_t)(ai * 4 + c) * L.hw);
            }
            const float lg[4] = {l4.x, l4.y, l4.z, l4.w};
            const float d0[4] = {q[0].x, q[0].y, q[0].z, q[0].w}, d1[4] = {q[1].x, q[1].y, q[1].z, q[1].w};
            const float d2[4] = {q[2].x, q[2].y, q[2].z, q[2].w}, d3[4] = {q[3].x, q[3].y, q[3].z, q[3].w};
            const float4 ca = L.cell[ai];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const float4 anchor = make_float4(sx[v] + ca.x, sy[v] + ca.y, sx[v] + ca.z, sy[v] + ca.w);
                const int o = (lane * 4 + v) * A + ai;
                s_box[o] = decode_delta(anchor, make_float4(d0[v], d1[v], d2[v], d3[v]), g.wt, g.scale_clamp);
                s_log[o] = lg[v];
            }
        }
    }
    __syncwarp();
    const int64_t obase = (int64_t)img * g.out_img_stride + L.out_offset + (int64_t)pos0 * A;
    const int total = npos * A;
    for (int i = lane; i < total; i += 32) {
        st_stream(g.boxes_out + obase + i, s_box[i]);
        st_stream(g.logits_out + obase + i, s_log[i]);
    }
}

}  // namespace det

using namespace det;

#ifdef DET_DEBUG_PHASES
// write-only bandwidth probe (profiles/scripts/write_probe2.py): 16-byte streaming stores of a payload derived from the index
// mode 0: zeros; 1: every value distinct and non-zero; 2: zeros with ~5 % non-zero values (the IoU matrix of a detection set)
__global__ void write_probe_kernel(float4* __restrict__ out, int64_t n4, int mode) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (mode == 1) {
            const float f = (float)(i & 0xffffff) + 1.0f;
            v = make_float4(f, f + 0.25f, f + 0.5f, f + 0.75f);
        } else if (mode == 2) {
            const uint32_t h = (uint32_t)i * 0x9E3779B1u;
            if ((h >> 24) < 51u) v.x = (float)(h & 0xffff) * (1.0f / 65536.0f) + 0.01f;   // one value in 20 % of the float4s
        }
        det::st_stream(out + i, v);
    }
}
extern "C" __attribute__((visibility("default"))) int det_debug_write_probe(float* out, int64_t n, int mode, int blocks, void* stream) {
    write_probe_kernel<<<blocks, 256, 0, det::as_stream(stream)>>>(reinterpret_cast<float4*>(out), n / 4, mode);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}
#endif

extern "C" {

int det_pairwise_overlap(const float* boxes1, int64_t n, const float* boxes2, int64_t m, int mode, float* out,
                         void* stream) {
    DET_CHECK_ARG(n >= 0 && m >= 0, "negative size");
    if (n == 0 || m == 0) return DET_OK;
    DET_CHECK_ARG(boxes1 && boxes2 && out, "null pointer");
    if (!aligned16(boxes1) || !aligned16(boxes2)) {
        set_error("boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    DET_CHECK_ARG((n + kPairRows - 1) / kPairRows <= 65535, "more than 2M rows: split the call");
    cudaStream_t st = as_stream(stream);
    switch (mode) {
        case DET_OVERLAP_IOU: return launch_pairwise<DET_OVERLAP_IOU>(boxes1, n, boxes2, m, out, st);
        case DET_OVERLAP_IOA: return launch_pairwise<DET_OVERLAP_IOA>(boxes1, n, boxes2, m, out, st);
        case DET_OVERLAP_INTERSECTION: return launch_pairwise<DET_OVERLAP_INTERSECTION>(boxes1, n, boxes2, m, out, st);
    }
    set_error("unknown overlap mode %d", mode);
    return DET_ERR_BAD_ARG;
}

int det_matched_iou(const float* boxes1, const float* boxes2, int64_t n, float* out, void* stream) {
    DET_CHECK_ARG(n >= 0, "negative size");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(boxes1 && boxes2 && out, "null pointer");
    if (!aligned16(boxes1) || !aligned16(boxes2)) {
        set_error("boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    matched_iou_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(boxes1), reinterpret_cast<const float4*>(boxes2), n, out);
    DET_LAUNCH_OK("matched_iou_kernel");
    return DET_OK;
}

int det_apply_deltas(const float* deltas, const float* boxes, int64_t m, int k, float wx, float wy, float ww,
                     float wh, float scale_clamp, float* out, void* stream) {
    DET_CHECK_ARG(m >= 0 && k >= 1, "bad size");
    if (m == 0) return DET_OK;
    DET_CHECK_ARG(deltas && boxes && out, "null pointer");
    if (!aligned16(deltas) || !aligned16(boxes) || !aligned16(out)) {
        set_error("deltas/boxes/out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    const int64_t total = m * k;
    apply_deltas_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(deltas), reinterpret_cast<const float4*>(boxes), total, k,
        CodecWeights{wx, wy, ww, wh}, scale_clamp, reinterpret_cast<float4*>(out));
    DET_LAUNCH_OK("apply_deltas_kernel");
    return DET_OK;
}

int det_apply_deltas_backward(const float* deltas, const float* boxes, const float* grad_out, int64_t m, int k, float wx,
                              float wy, float ww, float wh, float scale_clamp, float* grad_deltas, float* grad_boxes,
                              void* stream) {
    DET_CHECK_ARG(m >= 0 && k >= 1, "bad size");
    if (m == 0) return DET_OK;
    DET_CHECK_ARG(deltas && boxes && grad_out && (grad_deltas || grad_boxes), "null pointer");
    if (!aligned16(deltas) || !aligned16(boxes) || !aligned16(grad_out) || (grad_deltas && !aligned16(grad_deltas)) ||
        (grad_boxes && !aligned16(grad_boxes))) {
        set_error("deltas/boxes/gradients must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    apply_deltas_backward_kernel<<<(unsigned)((m + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(deltas), reinterpret_cast<const float4*>(boxes),
        reinterpret_cast<const float4*>(grad_out), m, k, CodecWeights{wx, wy, ww, wh}, scale_clamp,
        reinterpret_cast<float4*>(grad_deltas), reinterpret_cast<float4*>(grad_boxes));
    DET_LAUNCH_OK("apply_deltas_backward_kernel");
    return DET_OK;
}

int det_get_deltas(const float* src, const float* tgt, int64_t m, float wx, float wy, float ww, float wh, float* out,
                   int32_t* invalid_flag, void* stream) {
    DET_CHECK_ARG(m >= 0, "bad size");
    if (m == 0) return DET_OK;
    DET_CHECK_ARG(src && tgt && out, "null pointer");
    if (!aligned16(src) || !aligned16(tgt) || !aligned16(out)) {
        set_error("src/tgt/out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    get_deltas_kernel<<<(unsigned)((m + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(src), reinterpret_cast<const float4*>(tgt), m, CodecWeights{wx, wy, ww, wh},
        reinterpret_cast<float4*>(out), invalid_flag);
    DET_LAUNCH_OK("get_deltas_kernel");
    return DET_OK;
}

int det_grid_anchors(const float* cell_anchors, int a, int h, int w, int stride, float offset, float* out,
                     void* stream) {
    DET_CHECK_ARG(a >= 1 && h >= 0 && w >= 0, "bad size");
    const int64_t total = (int64_t)h * w * a;
    if (total == 0) return DET_OK;
    DET_CHECK_ARG(cell_anchors && out, "null pointer");
    if (!aligned16(cell_anchors) || !aligned16(out)) {
        set_error("cell_anchors/out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    grid_anchors_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(cell_anchors), a, h, w, stride, offset, reinterpret_cast<float4*>(out));
    DET_LAUNCH_OK("grid_anchors_kernel");
    return DET_OK;
}

}  // extern "C"

// The entry points below have C linkage through their declarations in det_b200.h; the per-type implementations
// between them are C++ templates.
template <typename T>
static int rpn_decode_level_t(const T* objectness, const T* deltas, int n, int a, int h, int w, int stride,
                              float offset, const float* cell_anchors, float wx, float wy, float ww, float wh,
                              float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                              int64_t out_offset, void* stream) {
    DET_CHECK_ARG(n >= 0 && a >= 1 && a <= kMaxCellAnchors && h >= 0 && w >= 0, "bad size (a <= 16)");
    const int64_t hw = (int64_t)h * w;
    if (n == 0 || hw == 0) return DET_OK;
    DET_CHECK_ARG(objectness && deltas && cell_anchors && logits_out && boxes_out, "null pointer");
    DET_CHECK_ARG(out_img_stride >= hw * a + out_offset && out_offset >= 0, "output slot out of range");
    DET_CHECK_ARG(n <= 65535, "n > 65535");
    if (!aligned16(cell_anchors) || !aligned16(boxes_out)) {
        set_error("cell_anchors/boxes_out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    const CodecWeights wt{wx, wy, ww, wh};
    auto cell = reinterpret_cast<const float4*>(cell_anchors);
    auto bo = reinterpret_cast<float4*>(boxes_out);
    cudaStream_t st = as_stream(stream);
    const bool vec = (hw % 4 == 0) && aligned_to(objectness, 4 * sizeof(T)) && aligned_to(deltas, 4 * sizeof(T));
    if (vec) {
        dim3 grid((unsigned)((hw / 4 + 255) / 256), (unsigned)n);
        rpn_decode_level_kernel<4, T><<<grid, 256, 0, st>>>(objectness, deltas, n, a, h, w, stride, offset, cell, wt,
                                                         scale_clamp, logits_out, bo, out_img_stride, out_offset);
    } else {
        dim3 grid((unsigned)((hw + 255) / 256), (unsigned)n);
        rpn_decode_level_kernel<1, T><<<grid, 256, 0, st>>>(objectness, deltas, n, a, h, w, stride, offset, cell, wt,
                                                         scale_clamp, logits_out, bo, out_img_stride, out_offset);
    }
    DET_LAUNCH_OK("rpn_decode_level_kernel");
    return DET_OK;
}

int det_rpn_decode_level(const float* objectness, const float* deltas, int n, int a, int h, int w, int stride,
                         float offset, const float* cell_anchors, float wx, float wy, float ww, float wh,
                         float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                         int64_t out_offset, void* stream) {
    return rpn_decode_level_t<float>(objectness, deltas, n, a, h, w, stride, offset, cell_anchors, wx, wy, ww, wh,
                                     scale_clamp, logits_out, boxes_out, out_img_stride, out_offset, stream);
}

template <typename T>
static int rpn_decode_t(const det_rpn_level_t* levels_host, int num_levels, int n, int a, float offset, float wx, float wy,
                        float ww, float wh, float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                        void* stream) {
    DET_CHECK_ARG(num_levels >= 0 && n >= 0 && a >= 1 && a <= kMaxCellAnchors, "bad size (a <= 16)");
    if (num_levels == 0 || n == 0) return DET_OK;
    DET_CHECK_ARG(levels_host && logits_out && boxes_out, "null pointer");
    const bool flat_ok = a <= kRpnFlatMaxA && aligned16(boxes_out);
    RpnFlatArgs f;
    f.num_levels = 0; f.n = n; f.a = a; f.offset = offset; f.scale_clamp = scale_clamp;
    f.wt = CodecWeights{wx, wy, ww, wh};
    f.out_img_stride = out_img_stride; f.logits_out = logits_out; f.boxes_out = reinterpret_cast<float4*>(boxes_out);
    long long tb = 0;
    for (int l = 0; l < num_levels; ++l) {
        const det_rpn_level_t& L = levels_host[l];
        DET_CHECK_ARG(L.objectness && L.deltas && L.cell_anchors && L.h >= 0 && L.w >= 0 && L.out_offset >= 0, "bad level");
        const int64_t hw = (int64_t)L.h * L.w;
        DET_CHECK_ARG(out_img_stride >= L.out_offset + hw * a, "output slot out of range");
        // (levels whose planes are not 16-byte tiles ride along with scalar loads: they are the small ones)
        const bool flat = flat_ok && f.num_levels < kRpnFlatMaxLevels && hw < (1ll << 30) && aligned16(L.cell_anchors);
        const bool vec_ok = hw % 4 == 0 && aligned_to(L.objectness, 4 * sizeof(T)) && aligned_to(L.deltas, 4 * sizeof(T));
        if (!flat) {  // this level takes its own launch: same results
            const int rc = rpn_decode_level_t<T>(reinterpret_cast<const T*>(L.objectness),
                                                 reinterpret_cast<const T*>(L.deltas), n, a, L.h, L.w, L.stride, offset, L.cell_anchors, wx,
                                                wy, ww, wh, scale_clamp, logits_out, boxes_out, out_img_stride,
                                                L.out_offset, stream);
            if (rc != DET_OK) return rc;
            continue;
        }
        RpnLevelDev& D = f.lv[f.num_levels];
        f.tile_begin[f.num_levels] = tb;
        D.obj = L.objectness; D.deltas = L.deltas; D.cell = reinterpret_cast<const float4*>(L.cell_anchors);
        D.w = L.w > 0 ? L.w : 1; D.hw = L.h * L.w; D.tiles = (D.hw + kRpnTilePos - 1) / kRpnTilePos;
        D.stride = L.stride; D.vec = vec_ok ? 1 : 0; D.out_offset = L.out_offset;
        tb += (long long)n * D.tiles;
        ++f.num_levels;
    }
    for (int l = f.num_levels; l < kRpnFlatMaxLevels; ++l) {
        RpnLevelDev& D = f.lv[l];
        D.obj = nullptr; D.deltas = nullptr; D.cell = nullptr; D.w = 1; D.hw = 0; D.tiles = 1; D.stride = 0; D.vec = 1;
        D.out_offset = 0;
    }
    for (int l = f.num_levels; l <= kRpnFlatMaxLevels; ++l) f.tile_begin[l] = tb;
    if (tb == 0) return DET_OK;
    const long long blocks = (tb + kRpnFlatWarps - 1) / kRpnFlatWarps;
    DET_CHECK_ARG(blocks < (1ll << 31), "too many positions");
    const size_t smem = (size_t)kRpnFlatWarps * kRpnTilePos * a * (sizeof(float4) + sizeof(float));
    cudaError_t e = cudaFuncSetAttribute(rpn_decode_flat_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(rpn_decode_flat_kernel)");
    rpn_decode_flat_kernel<T><<<(unsigned)blocks, kRpnFlatWarps * 32, smem, as_stream(stream)>>>(f);
    DET_LAUNCH_OK("rpn_decode_flat_kernel");
    return DET_OK;
}

int det_rpn_decode(const det_rpn_level_t* levels_host, int num_levels, int n, int a, float offset, float wx, float wy,
                   float ww, float wh, float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                   void* stream) {
    return rpn_decode_t<float>(levels_host, num_levels, n, a, offset, wx, wy, ww, wh, scale_clamp, logits_out, boxes_out,
                               out_img_stride, stream);
}

int det_rpn_decode_typed(const det_rpn_level_t* levels_host, int num_levels, int n, int a, float offset, float wx,
                         float wy, float ww, float wh, float scale_clamp, float* logits_out, float* boxes_out,
                         int64_t out_img_stride, int head_dtype, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, rpn_decode_t, levels_host, num_levels, n, a, offset, wx, wy, ww, wh, scale_clamp,
                      logits_out, boxes_out, out_img_stride, stream);
}
