// Dense anchor head decode for ALL pyramid levels in one launch (subsystem 1, BASELINE configs[3]).
//
// head of level l: (N, A*(5+C), Hl, Wl) fp32, the conv's own NCHW layout.  Output: boxes (N,R,4), best score (N,R),
// best class (N,R) int64 with R = sum_l Hl*Wl*A in (level, h, w, a) order.  340 bytes are read per anchor and 28
// written: a pure HBM stream.
//
// One thread per (level, image, anchor, 4 consecutive positions) walks all 5+C planes of its anchor with 16-byte
// loads, 8 in flight, and keeps 4 independent (running max, first arg-max) chains in registers.  Consecutive threads
// read consecutive 16 bytes of the same plane (full 128-byte lines); the flat grid covers every level, so small
// levels ride along with the big one instead of paying their own launch and tail; 64 registers -> 1024 resident
// threads per SM keep ~130 KB per SM in flight.  Measured (profiles/README.md): 4.9 TB/s algorithmic at N=32
// (297 MB, ramp-limited like torch's own reductions), 6.1 TB/s = 93 % of the measured copy peak at N=256.
// A level whose planes are not whole 4-position vectors (h*w % 4 != 0, e.g. 13x13, or a head not aligned to 4
// elements) rides in the same launch: its threads read their 4 positions with scalar loads and skip the ones past h*w.
// A bulk-async-copy (cp.async.bulk + mbarrier, producer warp / consumer warps) pipeline was built and measured
// first (commit "Dense head decode: one-launch ..."): 4.2 TB/s -- the 1 KB-per-plane slabs need 85 copy
// instructions each and only two 87 KB stages fit, so it lost to plain loads and was removed.
//
// Specification: oracle/ref_torch.py dense_decode (own; SURVEY.md section 8 row a15 -- no reference implementation).
//
// det_dense_detect (BASELINE configs[3] as a detector runs it: decode -> score threshold -> per-class NMS -> top
// max_det) uses the same streaming kernel in SELECT mode: nothing dense is written, a position whose score passes the
// threshold appends (box, score, class, row index) to its image's candidate list; `dense_detect_nms_kernel` (one CTA
// per image, nms_small.cuh) then orders the list by row index (= the order torch.nonzero gives the oracle, which
// decides ties), runs the exact greedy NMS and writes the detections.  GATED select reads the objectness plane first
// and skips the other 84 planes of a thread's 4 positions when sigmoid(obj) <= thresh for all of them -- exact, since
// score = sigmoid(obj) * sigmoid(best) <= sigmoid(obj) in fp32 (a factor <= 1 cannot round a product upwards).
#include <type_traits>

#include "nms_core.cuh"
#include "nms_small.cuh"
#include "nms_list.cuh"

namespace det {

constexpr int kMaxLevels = 8;
constexpr int kModeDense = 0, kModeSelect = 1, kModeSelectGated = 2;

struct DenseLevelDev {
    const void* head;  // elements of the kernel's head type T
    const float2* anchors_wh;
    int w, hw;
    float stride;
    int vec;  // planes are whole 4-element vectors (hw % 4 == 0, head aligned to 4 elements): one vector load per plane
    int64_t out_offset;
};

constexpr int kFlatThreads = 128;  // 8 CTAs per SM: at one or two waves (N=32) the finer grain trims the tail, 62.0 -> 61.2 us

struct FlatArgs {
    DenseLevelDev lv[kMaxLevels];
    long long thread_begin[kMaxLevels + 1];  // first flat thread of each level
    int num_levels, n, a, c;
    float scale_clamp;
    int64_t out_img_stride;
    float4* boxes_out;
    float* score_out;
    int64_t* class_out;
    // SELECT modes: per-image candidate lists of capacity cand_cap (row index inside the image, box, score, class)
    float score_thresh;
    int cand_cap;
    int32_t* cand_count;
    float4* cand_box;
    float* cand_score;
    int32_t* cand_cls;
    int32_t* cand_id;
    int32_t* overflow_flag;  // cleared here (first thread of the grid); the NMS kernel behind this one sets it
};

// Four consecutive positions of one plane as fp32; STREAM: evict-first (read once).  Through a vector pointer: one
// load.  Through an element pointer (a level that is not vec): scalar loads of the first m positions, and the positions
// past the plane's end read as 0.
template <typename T, bool STREAM>
__device__ __forceinline__ float4 ld_quad(const typename Head<T>::vec* p, int) {
    return STREAM ? ld4_stream<T>(p) : ld4<T>(p);
}
template <typename T, bool STREAM>
__device__ __forceinline__ float4 ld_quad(const T* p, int m) {
    float r[4];
#pragma unroll
    for (int v = 0; v < 4; ++v) r[v] = v < m ? (STREAM ? ld1_stream(p + v) : ld1(p + v)) : 0.0f;
    return make_float4(r[0], r[1], r[2], r[3]);
}

// Flat thread gt of level l (tid = threadIdx.x): 4 consecutive positions of one anchor.  VEC == L.vec.  A non-vec level
// has ceil(hw / 4) position groups; the positions of its last group that lie past hw are never written.
template <int MODE, typename T, bool VEC>
__device__ __forceinline__ void decode_quad(const FlatArgs& g, int l, long long gt, bool active, unsigned tid) {
    const DenseLevelDev& L = g.lv[l];
    // one step along a plane: 4 positions (16 bytes for fp32, 8 for bf16 / fp16) or, on a non-vec level, one
    using P = typename std::conditional<VEC, typename Head<T>::vec, T>::type;
    const int groups = VEC ? L.hw >> 2 : (L.hw + 3) >> 2, A = g.a, C = g.c, nch = 5 + C;
    const long long local = gt - g.thread_begin[l];
    const int grp = (int)(local % groups);
    const int ia = (int)(local / groups);  // image * A + anchor
    const int img = ia / A, ai = ia - img * A;
    const int plane = VEC ? groups : L.hw;  // stride between planes, in steps P
    const int m = L.hw - grp * 4;           // positions of the group inside the plane: < 4 only at a non-vec plane's end
    const P* pl = reinterpret_cast<const P*>(static_cast<const T*>(L.head) + (int64_t)ia * nch * L.hw) + (VEC ? grp : grp * 4);
    const P* pk = pl + (int64_t)5 * plane;
    if (MODE == kModeSelectGated && active) {
        const float4 q = ld_quad<T, true>(pl + (int64_t)4 * plane, m);
        const float thr = g.score_thresh;
        // `!(x > thr)` also holds for NaN: a NaN objectness gives a NaN score, which is no candidate either
        if (!(sigmoidf_rn(q.x) > thr) && !(sigmoidf_rn(q.y) > thr) && !(sigmoidf_rn(q.z) > thr) &&
            !(sigmoidf_rn(q.w) > thr))
            active = false;
    }
    float4 box[4];
    float score[4];
    int bidx[4] = {0, 0, 0, 0};
    if (active) {
        float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        // class planes in flight: 8 vector loads, or 4 x 4 scalar loads, which keeps the decode kernel at 64 registers
        constexpr int U = VEC ? 8 : 4;
        int k = 0;
        for (; k + U <= C; k += U) {
            float4 q[U];
#pragma unroll
            for (int i = 0; i < U; ++i) q[i] = ld_quad<T, true>(pk + (int64_t)(k + i) * plane, m);
#pragma unroll
            for (int i = 0; i < U; ++i) {
                bidx[0] = (q[i].x > best[0]) ? k + i : bidx[0]; best[0] = max_nan(best[0], q[i].x);
                bidx[1] = (q[i].y > best[1]) ? k + i : bidx[1]; best[1] = max_nan(best[1], q[i].y);
                bidx[2] = (q[i].z > best[2]) ? k + i : bidx[2]; best[2] = max_nan(best[2], q[i].z);
                bidx[3] = (q[i].w > best[3]) ? k + i : bidx[3]; best[3] = max_nan(best[3], q[i].w);
            }
        }
        for (; k < C; ++k) {
            const float4 q = ld_quad<T, true>(pk + (int64_t)k * plane, m);
            bidx[0] = (q.x > best[0]) ? k : bidx[0]; best[0] = max_nan(best[0], q.x);
            bidx[1] = (q.y > best[1]) ? k : bidx[1]; best[1] = max_nan(best[1], q.y);
            bidx[2] = (q.z > best[2]) ? k : bidx[2]; best[2] = max_nan(best[2], q.z);
            bidx[3] = (q.w > best[3]) ? k : bidx[3]; best[3] = max_nan(best[3], q.w);
        }
        // the running max is NaN-propagating and `q > max` is false once it is NaN: a NaN column is finished by an
        // exact rescan (torch.max: the first NaN wins)
        if (best[0] != best[0] || best[1] != best[1] || best[2] != best[2] || best[3] != best[3]) {
            bool found[4] = {false, false, false, false};
            for (int j = 0; j < C; ++j) {
                const float4 q4 = ld_quad<T, false>(pk + (int64_t)j * plane, m);
                const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                for (int v = 0; v < 4; ++v)
                    if (q[v] != q[v] && !found[v]) {
                        found[v] = true;
                        bidx[v] = j;
                    }
            }
        }
        float t[5][4];  // box logits last: they would only occupy registers during the class loop
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float4 q = ld_quad<T, true>(pl + (int64_t)j * plane, m);
            t[j][0] = q.x; t[j][1] = q.y; t[j][2] = q.z; t[j][3] = q.w;
        }
        const float2 awh = L.anchors_wh[ai];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int pos = grp * 4 + v;
            const int row = pos / L.w, colx = pos - row * L.w;
            const float cx = (sigmoidf_rn(t[0][v]) + (float)colx) * L.stride;
            const float cy = (sigmoidf_rn(t[1][v]) + (float)row) * L.stride;
            const float tw = (t[2][v] > g.scale_clamp) ? g.scale_clamp : t[2][v];  // torch.clamp(max=): NaN stays NaN
            const float th = (t[3][v] > g.scale_clamp) ? g.scale_clamp : t[3][v];
            const float bw = expf(tw) * awh.x, bh = expf(th) * awh.y;
            box[v] = make_float4(cx - 0.5f * bw, cy - 0.5f * bh, cx + 0.5f * bw, cy + 0.5f * bh);
            score[v] = sigmoidf_rn(t[4][v]) * (C > 0 ? sigmoidf_rn(best[v]) : 1.0f);
        }
    }
    if (MODE == kModeDense) {
        const int64_t obase = (int64_t)img * g.out_img_stride + L.out_offset;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            if (!VEC && v >= m) break;
            const int64_t o = obase + (int64_t)(grp * 4 + v) * A + ai;
            st_stream(g.boxes_out + o, box[v]);
            st_stream(g.score_out + o, score[v]);
            g.class_out[o] = (int64_t)(C > 0 ? bidx[v] : 0);
        }
    } else {
        // append the passing positions to the image's candidate list: one atomic per warp when the warp works on one
        // image (almost always), slots dealt with a shuffle scan.  The list order is arbitrary; the NMS kernel
        // restores row order where it matters (ties).
        unsigned pass = 0;
        if (active) {
#pragma unroll
            for (int v = 0; v < 4; ++v) pass |= (score[v] > g.score_thresh) ? (1u << v) : 0u;
        }
        const int my = __popc(pass);
        const int lane = tid & 31;
        const int img0 = __shfl_sync(0xffffffffu, img, 0);
        int slot = 0;
        if (__all_sync(0xffffffffu, img == img0)) {
            int incl = my;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                incl += (lane >= o) ? up : 0;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            if (total) {
                int base = 0;
                if (lane == 0) base = atomicAdd(g.cand_count + (int64_t)img0 * kCountStride, total);
                slot = __shfl_sync(0xffffffffu, base, 0) + incl - my;
            }
        } else if (my) {
            slot = atomicAdd(g.cand_count + (int64_t)img * kCountStride, my);
        }
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            if (!((pass >> v) & 1u)) continue;
            if (slot < g.cand_cap) {
                const int64_t o = (int64_t)img * g.cand_cap + slot;
                g.cand_box[o] = box[v];
                g.cand_score[o] = score[v];
                g.cand_cls[o] = C > 0 ? bidx[v] : 0;
                g.cand_id[o] = (int32_t)(L.out_offset + (int64_t)(grp * 4 + v) * A + ai);
            }
            ++slot;
        }
    }
}

template <int MODE, typename T>
__global__ void __launch_bounds__(kFlatThreads) dense_decode_flat_kernel(const __grid_constant__ FlatArgs g) {
    if (MODE != kModeDense) {
        pdl_trigger();  // det_dense_detect: the NMS kernel's CTAs may move in as SM slots free up
        if (blockIdx.x == 0 && threadIdx.x == 0 && g.overflow_flag) *g.overflow_flag = 0;
    }
    long long gt = (long long)blockIdx.x * kFlatThreads + threadIdx.x;
    bool active = gt < g.thread_begin[g.num_levels];
    if (MODE == kModeDense) {
        if (!active) return;
    } else if (!active) {
        gt = 0;  // SELECT: every lane reaches the warp-collective append below
    }
    int l = 0;
#pragma unroll
    for (int q = 1; q < kMaxLevels; ++q)
        if (q < g.num_levels && gt >= g.thread_begin[q]) l = q;
    // Non-vec levels are compiled into the decode only: det_dense_detect admits vec levels alone, so the lanes of a
    // SELECT warp never split between the two forms around the warp-collective append.  threadIdx.x is read here and
    // handed down: only in the kernel itself does the compiler bound it by kFlatThreads, and the SELECT code uses that.
    if (MODE != kModeDense || g.lv[l].vec) decode_quad<MODE, T, true>(g, l, gt, active, threadIdx.x);
    else decode_quad<MODE, T, false>(g, l, gt, active, threadIdx.x);
}

// ---- candidate compaction / final gather for the unfused detector path (any candidate count: the overflow route of
// det_dense_detect and pyramids outside its limits).  One CTA per image walks the image's rows in order; a block-wide
// ballot scan keeps the candidates (score > thr) in ROW ORDER, which is what torch.nonzero gives the oracle.
constexpr int kCompactThreads = 512;

__global__ void __launch_bounds__(kCompactThreads)
threshold_compact_kernel(const float4* __restrict__ boxes, const float* __restrict__ scores,
                         const int64_t* __restrict__ classes, int64_t r, float thr, int64_t cap,
                         int64_t* __restrict__ out_rows, float4* __restrict__ out_boxes, float* __restrict__ out_scores,
                         int64_t* __restrict__ out_classes, int32_t* __restrict__ out_counts) {
    __shared__ int s_warp[kCompactThreads / 32];
    __shared__ int s_base;
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int64_t in0 = (int64_t)img * r, out0 = (int64_t)img * cap;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int64_t j0 = 0; j0 < r; j0 += kCompactThreads) {
        const int64_t j = j0 + tid;
        const float sc = j < r ? scores[in0 + j] : 0.0f;
        const bool pass = j < r && sc > thr;  // NaN never passes (torch: nan > thr is False)
        const unsigned bal = __ballot_sync(0xffffffffu, pass);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        int before = s_base, total = 0;
#pragma unroll
        for (int w = 0; w < kCompactThreads / 32; ++w) {
            const int v = s_warp[w];
            before += w < wid ? v : 0;
            total += v;
        }
        const int64_t slot = before + __popc(bal & ((1u << lane) - 1u));
        if (pass && slot < cap) {
            out_rows[out0 + slot] = j;
            out_boxes[out0 + slot] = boxes[in0 + j];
            out_scores[out0 + slot] = sc;
            out_classes[out0 + slot] = classes ? classes[in0 + j] : 0;
        }
        __syncthreads();
        if (tid == 0) s_base += total;
    }
    __syncthreads();
    if (tid == 0) out_counts[img] = (int32_t)(s_base < cap ? s_base : cap);
}

__global__ void gather_detections_kernel(const int64_t* __restrict__ keep, const int32_t* __restrict__ keep_counts,
                                         int64_t max_det, const int64_t* __restrict__ rows,
                                         const float4* __restrict__ boxes, const float* __restrict__ scores,
                                         const int64_t* __restrict__ classes, int64_t cap, int64_t n,
                                         int64_t* __restrict__ det_idx, float4* __restrict__ det_boxes,
                                         float* __restrict__ det_scores, int64_t* __restrict__ det_classes) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * max_det) return;
    const int64_t img = t / max_det, j = t - img * max_det;
    if (j >= keep_counts[img]) return;  // rows past the count stay undefined, as in det_dense_detect
    const int64_t k = keep[t];
    const int64_t src = img * cap + k;
    det_idx[t] = rows ? rows[src] : k;
    det_boxes[t] = boxes[src];
    det_scores[t] = scores[src];
    det_classes[t] = classes ? classes[src] : 0;
}

}  // namespace det


using namespace det;

template <int CAP, int T>
static int launch_detect_nms_t(const SelectArgs& sel, int n, float thr_f, int mode, int64_t max_det, int64_t* det_idx,
                               float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                               int32_t* overflow_flag, cudaStream_t st) {
    const size_t smem = sizeof(DetectSmem<CAP, T>);
    cudaError_t e = cudaFuncSetAttribute(dense_detect_nms_kernel<CAP, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(dense_detect_nms_kernel)");
    // programmatic dependent launch: the CTAs take their SM slots while the select kernel drains (see common.cuh)
    e = launch_pdl(dense_detect_nms_kernel<CAP, T>, dim3(n), dim3(T), smem, st, sel.cand_count, sel.cand_box, sel.cand_score,
                   sel.cand_cls, sel.cand_id, sel.cand_cap, thr_f, mode, max_det, det_idx,
                   reinterpret_cast<float4*>(det_boxes), det_scores, det_classes, det_count, overflow_flag, nullptr, nullptr);
    if (e != cudaSuccess) return cuda_fail(e, "dense_detect_nms_kernel");
    return DET_OK;
}

template <int CAP>
static int launch_detect_nms(const SelectArgs& sel, int n, float thr_f, int mode, int64_t max_det, int64_t* det_idx,
                             float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                             int32_t* overflow_flag, cudaStream_t st) {
    if (n <= sm_count())
        return launch_detect_nms_t<CAP, 512>(sel, n, thr_f, mode, max_det, det_idx, det_boxes, det_scores, det_classes,
                                             det_count, overflow_flag, st);
    return launch_detect_nms_t<CAP, 256>(sel, n, thr_f, mode, max_det, det_idx, det_boxes, det_scores, det_classes,
                                         det_count, overflow_flag, st);
}

int det::launch_list_nms(const SelectArgs& sel, int n, float thr_f, int mode, int64_t max_det, int64_t* det_idx,
                         float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                         int32_t* overflow_flag, cudaStream_t st) {
    if (sel.cand_cap <= 1024)
        return launch_detect_nms<1024>(sel, n, thr_f, mode, max_det, det_idx, det_boxes, det_scores, det_classes,
                                       det_count, overflow_flag, st);
    if (sel.cand_cap <= 2048)
        return launch_detect_nms<2048>(sel, n, thr_f, mode, max_det, det_idx, det_boxes, det_scores, det_classes,
                                       det_count, overflow_flag, st);
    return launch_detect_nms<4096>(sel, n, thr_f, mode, max_det, det_idx, det_boxes, det_scores, det_classes, det_count,
                                   overflow_flag, st);
}

#ifdef DET_DEBUG_PHASES
extern "C" {
__attribute__((visibility("default"))) int det_debug_read_phases_dense(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, det::g_phase_clock, sizeof(long long) * 32) == cudaSuccess ? 0 : -4;
}
__attribute__((visibility("default"))) int det_debug_read_phase_blocks_dense(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, det::g_phase_block, sizeof(long long) * 64 * 16) == cudaSuccess ? 0 : -4;
}
}  // extern "C"
#endif

// The entry points below have C linkage through their declarations in det_b200.h; the per-type implementations
// between them are C++ templates.

// a vec level streams its planes with one vector load per 4 positions: whole vectors per plane, head aligned to 4
// elements.  det_dense_detect admits vec levels only.
template <typename T>
static bool level_is_flat(const void* head, int64_t hw) {
    return hw % 4 == 0 && aligned_to(head, 4 * sizeof(T)) && hw < (1ll << 30);
}

template <typename T>
static int launch_flat(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                       float* boxes_out, float* score_out, int64_t* class_out, int64_t out_img_stride, cudaStream_t st,
                       const SelectArgs* sel = nullptr) {
    FlatArgs f;
    f.score_thresh = sel ? sel->score_thresh : 0.f; f.cand_cap = sel ? sel->cand_cap : 0;
    f.cand_count = sel ? sel->cand_count : nullptr; f.cand_box = sel ? sel->cand_box : nullptr;
    f.cand_score = sel ? sel->cand_score : nullptr; f.cand_cls = sel ? sel->cand_cls : nullptr;
    f.cand_id = sel ? sel->cand_id : nullptr; f.overflow_flag = sel ? sel->overflow_flag : nullptr;
    f.num_levels = num_levels; f.n = n; f.a = a; f.c = c; f.scale_clamp = scale_clamp; f.out_img_stride = out_img_stride;
    f.boxes_out = reinterpret_cast<float4*>(boxes_out); f.score_out = score_out; f.class_out = class_out;
    long long tb = 0;
    for (int l = 0; l < kMaxLevels; ++l) {
        DenseLevelDev& D = f.lv[l];
        f.thread_begin[l] = tb;
        if (l < num_levels) {
            const det_dense_level_t& L = levels_host[l];
            const int64_t hw = (int64_t)L.h * L.w;
            DET_CHECK_ARG(hw < (1ll << 30), "level too large (h*w >= 2^30)");
            DET_CHECK_ARG(out_img_stride >= L.out_offset + hw * a, "output slot out of range");
            D.head = L.head; D.anchors_wh = reinterpret_cast<const float2*>(L.anchors_wh);
            D.w = L.w > 0 ? L.w : 1; D.hw = (int)hw; D.vec = level_is_flat<T>(L.head, hw) ? 1 : 0;
            D.stride = (float)L.stride; D.out_offset = L.out_offset;
            tb += (long long)n * a * ((D.hw + 3) / 4);
        } else {
            D.head = nullptr; D.anchors_wh = nullptr; D.w = 1; D.hw = 4; D.vec = 1;
            D.stride = 0.f; D.out_offset = 0;
        }
    }
    for (int l = num_levels; l <= kMaxLevels; ++l) f.thread_begin[l] = tb;
    if (tb == 0) return DET_OK;
    const long long blocks = (tb + kFlatThreads - 1) / kFlatThreads;
    DET_CHECK_ARG(blocks < (1ll << 31), "too many positions");
    const unsigned grid = (unsigned)blocks;
    if (!sel) dense_decode_flat_kernel<kModeDense, T><<<grid, kFlatThreads, 0, st>>>(f);
    else if (sel->mode == kModeSelectGated) dense_decode_flat_kernel<kModeSelectGated, T><<<grid, kFlatThreads, 0, st>>>(f);
    else dense_decode_flat_kernel<kModeSelect, T><<<grid, kFlatThreads, 0, st>>>(f);
    DET_LAUNCH_OK("dense_decode_flat_kernel");
    return DET_OK;
}

template <typename T>
static int dense_decode_t(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                          float* boxes_out, float* score_out, int64_t* class_out, int64_t out_img_stride, void* stream) {
    DET_CHECK_ARG(num_levels >= 0 && n >= 0 && a >= 1 && c >= 0, "bad size");
    if (num_levels == 0 || n == 0) return DET_OK;
    DET_CHECK_ARG(levels_host && boxes_out && score_out && class_out, "null pointer");
    DET_CHECK_ARG(num_levels <= kMaxLevels, "too many levels");
    for (int l = 0; l < num_levels; ++l) {
        const det_dense_level_t& L = levels_host[l];
        DET_CHECK_ARG(L.head && L.anchors_wh && L.h >= 0 && L.w >= 0 && L.out_offset >= 0, "bad level");
    }
    if (!aligned16(boxes_out)) {
        set_error("boxes_out must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    return launch_flat<T>(levels_host, num_levels, n, a, c, scale_clamp, boxes_out, score_out, class_out, out_img_stride,
                          as_stream(stream));
}

int det_dense_decode_level(const float* head, int n, int a, int c, int h, int w, int stride, const float* anchors_wh,
                           float scale_clamp, float* boxes_out, float* score_out, int64_t* class_out,
                           int64_t out_img_stride, int64_t out_offset, void* stream) {
    DET_CHECK_ARG(n >= 0 && a >= 1 && c >= 0 && h >= 0 && w >= 0, "bad size");
    const int64_t hw = (int64_t)h * w;
    if (n == 0 || hw == 0) return DET_OK;
    DET_CHECK_ARG(head && anchors_wh && boxes_out && score_out && class_out, "null pointer");
    DET_CHECK_ARG(out_offset >= 0 && out_img_stride >= hw * a + out_offset, "output slot out of range");
    const det_dense_level_t L = {head, anchors_wh, h, w, stride, 0, out_offset};
    return dense_decode_t<float>(&L, 1, n, a, c, scale_clamp, boxes_out, score_out, class_out, out_img_stride, stream);
}

int det_dense_decode(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                     float* boxes_out, float* score_out, int64_t* class_out, int64_t out_img_stride, void* stream) {
    return dense_decode_t<float>(levels_host, num_levels, n, a, c, scale_clamp, boxes_out, score_out, class_out,
                                 out_img_stride, stream);
}

int det_dense_decode_typed(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                           float* boxes_out, float* score_out, int64_t* class_out, int64_t out_img_stride,
                           int head_dtype, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, dense_decode_t, levels_host, num_levels, n, a, c, scale_clamp, boxes_out, score_out,
                      class_out, out_img_stride, stream);
}

int64_t det_dense_detect_workspace_bytes(int n, int64_t cand_cap) {
    if (n <= 0 || cand_cap <= 0) return 256;
    return (int64_t)n * kCountStride * 4 + (int64_t)n * cand_cap * (16 + 4 + 4 + 4);
}

int64_t det_dense_detect_counter_bytes(int n) { return n <= 0 ? 0 : (int64_t)n * kCountStride * 4; }

int det::bind_select_workspace(SelectArgs& sel, int n, int64_t cand_cap, void* workspace, int64_t workspace_bytes,
                               bool counters_zero, cudaStream_t st) {
    const int64_t need = det_dense_detect_workspace_bytes(n, cand_cap);
    if (!workspace || workspace_bytes < need) {
        set_error("workspace too small: need %lld bytes", (long long)need);
        return DET_ERR_WORKSPACE;
    }
    if (!aligned16(workspace)) {
        set_error("workspace must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    unsigned char* w = static_cast<unsigned char*>(workspace);
    sel.cand_cap = (int)cand_cap;
    sel.cand_count = reinterpret_cast<int32_t*>(w);
    w += (int64_t)n * kCountStride * 4;
    sel.cand_box = reinterpret_cast<float4*>(w);
    w += (int64_t)n * cand_cap * 16;
    sel.cand_score = reinterpret_cast<float*>(w);
    w += (int64_t)n * cand_cap * 4;
    sel.cand_cls = reinterpret_cast<int32_t*>(w);
    w += (int64_t)n * cand_cap * 4;
    sel.cand_id = reinterpret_cast<int32_t*>(w);
    // The NMS CTA of an image puts the image's counter back to zero once it has read it and the select kernel clears
    // the overflow word itself, so a call on a workspace whose counters are known to be zero (gate bit 1: zeroed once by
    // the caller, then only ever used by this call) is exactly two launches; otherwise the counters are cleared here.
    if (!counters_zero) {
        cudaError_t e = cudaMemsetAsync(sel.cand_count, 0, sizeof(int32_t) * (size_t)n * kCountStride, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    }
    return DET_OK;
}

template <typename T>
static int dense_detect_t(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                          float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap, int64_t max_det,
                          int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes,
                          int32_t* det_count, int32_t* overflow_flag, void* workspace, int64_t workspace_bytes,
                          void* stream) {
    DET_CHECK_ARG(num_levels >= 0 && n >= 0 && a >= 1 && c >= 0, "bad size");
    DET_CHECK_ARG(mode >= DET_NMS_AUTO && mode <= DET_NMS_OFFSET_TRICK, "unknown mode");
    DET_CHECK_ARG(cand_cap >= 1 && cand_cap <= 4096, "cand_cap must be in [1, 4096]");
    DET_CHECK_ARG(max_det >= 1, "max_det must be positive");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(det_idx && det_boxes && det_scores && det_classes && det_count, "null output");
    DET_CHECK_ARG(num_levels <= kMaxLevels, "too many levels");
    DET_CHECK_ARG(num_levels == 0 || levels_host, "null pointer");
    cudaStream_t st = as_stream(stream);
    if (!aligned16(det_boxes)) {
        set_error("det_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    int64_t rows = 0;
    for (int l = 0; l < num_levels; ++l) {
        const det_dense_level_t& L = levels_host[l];
        DET_CHECK_ARG(L.head && L.anchors_wh && L.h >= 0 && L.w >= 0 && L.out_offset >= 0, "bad level");
        if (!level_is_flat<T>(L.head, (int64_t)L.h * L.w)) {
            set_error("det_dense_detect needs h*w %% 4 == 0 and heads aligned to 4 elements (level %d: %d x %d)", l, L.h,
                      L.w);
            return DET_ERR_UNSUPPORTED;
        }
        rows = L.out_offset + (int64_t)L.h * L.w * a > rows ? L.out_offset + (int64_t)L.h * L.w * a : rows;
    }
    DET_CHECK_ARG(rows < (1ll << 31), "too many rows per image");
    SelectArgs sel;
    int rc = bind_select_workspace(sel, n, cand_cap, workspace, workspace_bytes, gate & 2, st);
    if (rc != DET_OK) return rc;
    sel.mode = (gate & 1) ? kModeSelectGated : kModeSelect;
    sel.overflow_flag = overflow_flag;
    sel.score_thresh = score_thresh;
    rc = launch_flat<T>(levels_host, num_levels, n, a, c, scale_clamp, nullptr, nullptr, nullptr, rows, st, &sel);
    if (rc != DET_OK) return rc;
    return launch_list_nms(sel, n, float_threshold_below(iou_threshold), mode, max_det, det_idx, det_boxes, det_scores,
                           det_classes, det_count, overflow_flag, st);
}

int det_dense_detect(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                     float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap, int64_t max_det,
                     int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                     int32_t* overflow_flag, void* workspace, int64_t workspace_bytes, void* stream) {
    return dense_detect_t<float>(levels_host, num_levels, n, a, c, scale_clamp, score_thresh, iou_threshold, mode, gate,
                                 cand_cap, max_det, det_idx, det_boxes, det_scores, det_classes, det_count, overflow_flag,
                                 workspace, workspace_bytes, stream);
}

int det_dense_detect_typed(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                           float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap,
                           int64_t max_det, int64_t* det_idx, float* det_boxes, float* det_scores,
                           int64_t* det_classes, int32_t* det_count, int32_t* overflow_flag, void* workspace,
                           int64_t workspace_bytes, int head_dtype, void* stream) {
    DET_HEAD_DISPATCH(head_dtype, dense_detect_t, levels_host, num_levels, n, a, c, scale_clamp, score_thresh,
                      iou_threshold, mode, gate, cand_cap, max_det, det_idx, det_boxes, det_scores, det_classes, det_count,
                      overflow_flag, workspace, workspace_bytes, stream);
}

int det_threshold_compact(const float* boxes, const float* scores, const int64_t* classes, int n, int64_t r,
                          float score_thresh, int64_t cap, int64_t* cand_rows, float* cand_boxes, float* cand_scores,
                          int64_t* cand_classes, int32_t* cand_counts, void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && cap >= 1, "bad size");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(boxes && scores && cand_rows && cand_boxes && cand_scores && cand_classes && cand_counts, "null pointer");
    if (!aligned16(boxes) || !aligned16(cand_boxes)) {
        set_error("boxes / cand_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    threshold_compact_kernel<<<n, kCompactThreads, 0, as_stream(stream)>>>(
        reinterpret_cast<const float4*>(boxes), scores, classes, r, score_thresh, cap, cand_rows,
        reinterpret_cast<float4*>(cand_boxes), cand_scores, cand_classes, cand_counts);
    DET_LAUNCH_OK("threshold_compact_kernel");
    return DET_OK;
}

int det_gather_detections(const int64_t* keep, const int32_t* keep_counts, int n, int64_t max_det, const int64_t* cand_rows,
                          const float* cand_boxes, const float* cand_scores, const int64_t* cand_classes, int64_t cap,
                          int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes, void* stream) {
    DET_CHECK_ARG(n >= 0 && max_det >= 1 && cap >= 1, "bad size");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(keep && keep_counts && cand_boxes && cand_scores && det_idx && det_boxes && det_scores && det_classes,
                  "null pointer");
    if (!aligned16(cand_boxes) || !aligned16(det_boxes)) {
        set_error("cand_boxes / det_boxes must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    const int64_t total = (int64_t)n * max_det;
    gather_detections_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        keep, keep_counts, max_det, cand_rows, reinterpret_cast<const float4*>(cand_boxes), cand_scores, cand_classes, cap, n,
        det_idx, reinterpret_cast<float4*>(det_boxes), det_scores, det_classes);
    DET_LAUNCH_OK("gather_detections_kernel");
    return DET_OK;
}
