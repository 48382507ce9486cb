// Large path of the batched NMS: images with up to 131071 boxes each, any number of images per call.
//
// Data layout in the caller's workspace (HBM), all arrays image-major with a padded row of Mp = roundup(m_max,
// 2048) slots: two u64 key buffers (ping-pong for the merge passes), boxes in sorted order (float4) + their
// areas, one state byte and one kept-list slot per position, and two segment work lists.
// Launch sequence: [stats] -> keys -> tile sort -> log2(Mp/2048) merge passes -> gather (+segment discovery)
//   -> warp segments (persistent, atomic work counter) -> CTA segments (persistent) -> re-key kept -> sort -> emit.
#pragma once
#include <cooperative_groups.h>
#include "nms_core.cuh"
#include "nms_list.cuh"

namespace det {

constexpr int kLargeIdxBits = 17;
constexpr int kTile = 2048;
constexpr int kSortThreads = 256;
constexpr int kVT = kTile / kSortThreads;
constexpr int kLargeWarpSegMax = 256;  // segments up to this length are swept by one warp
constexpr int kSegThreads = 256;   // candidates per chunk of the CTA sweep
constexpr int kSegCtaThreads = 1024;  // threads of the CTA that runs it: 4 groups share the list tests and bit rows
constexpr int kHugeSeg = 4096;     // longer segments are swept by the whole grid (cooperative kernel)
constexpr int kHugeChunk = 512;    // positions resolved per step by the segment's leader CTA
constexpr int kTierCap = 4096;     // top-k tier: capacity of an image's candidate list
constexpr int kTierMaxWant = 3072; // ... and the largest tier size tried (1.25 * max_out + 32)

struct LargeImg {
    int32_t cnt;
    int32_t trick;
    int32_t fast;
    float span;
    int32_t nkept;
    int32_t bad;
    int32_t nsurv;
    int32_t nonan;  // no box coordinate of the image is NaN: min/max in the predicate are single FMNMX instructions
    int32_t skip;   // the top-k tier already produced this image's output: nothing to do, nothing to write
    int32_t pad_[7];
};

struct LargeLayout {
    int n;
    int64_t m_max, mp, segcap;
    int64_t off_info, off_ctr, off_keys_a, off_keys_b, off_sbox, off_sarea, off_state, off_klist, off_seg_small,
        off_seg_large, off_seg_huge, off_huge_nk, hugecap, total;
    int64_t off_tier_count, off_tier_box, off_tier_score, off_tier_cls, off_tier_id, off_tier_full, off_tier_todo;
    LargeLayout(int n_, int64_t m_) : n(n_), m_max(m_) {
        mp = (m_max + kTile - 1) / kTile * kTile;
        segcap = mp < 32768 ? mp : 32768;
        int64_t o = 0;
        auto take = [&](int64_t bytes) {
            int64_t at = o;
            o += (bytes + 255) / 256 * 256;
            return at;
        };
        off_info = take((int64_t)sizeof(LargeImg) * n);
        off_ctr = take(64);
        off_keys_a = take(8 * n * mp);
        off_keys_b = take(8 * n * mp);
        off_sbox = take(16 * n * mp);
        off_sarea = take(4 * n * mp);
        off_state = take(n * mp);
        off_klist = take(4 * n * mp);
        off_seg_small = take(16 * n * segcap);
        off_seg_large = take(16 * n * segcap);
        hugecap = (int64_t)n * (mp / kHugeSeg + 1 > 16 ? mp / kHugeSeg + 1 : 16);  // RPN: up to 16 levels per image
        off_seg_huge = take(16 * hugecap);
        off_huge_nk = take(8 * 3 * hugecap);
        // top-k tier (max_out << boxes): candidate lists of the best-scored boxes of each image
        off_tier_count = take((int64_t)n * kCountStride * 4);
        off_tier_box = take((int64_t)16 * n * kTierCap);
        off_tier_score = take((int64_t)4 * n * kTierCap);
        off_tier_cls = take((int64_t)4 * n * kTierCap);
        off_tier_id = take((int64_t)4 * n * kTierCap);
        off_tier_full = take((int64_t)sizeof(FullStats) * n);
        off_tier_todo = take((int64_t)4 * n);
        total = o;
    }
};

struct LargeWs {
    LargeImg* info;
    int32_t* ctr;  // [0] #small segs, [1] #large segs, [2] next small, [3] next large, [4] #huge segs, [6] next large (spatial index)
    uint64_t *keys_a, *keys_b;
    float4* sbox;
    float* sarea;
    uint8_t* state;
    int32_t* klist;
    int4 *seg_small, *seg_large, *seg_huge;
    int2* huge_nk;  // [3][#huge]: running kept count, then the kept range of the chunk resolved in even / odd steps
    int32_t *tier_count, *tier_cls, *tier_id, *tier_todo;
    float4* tier_box;
    float* tier_score;
    FullStats* tier_full;
    LargeWs(const LargeLayout& l, void* base) {
        char* b = static_cast<char*>(base);
        info = reinterpret_cast<LargeImg*>(b + l.off_info);
        ctr = reinterpret_cast<int32_t*>(b + l.off_ctr);
        keys_a = reinterpret_cast<uint64_t*>(b + l.off_keys_a);
        keys_b = reinterpret_cast<uint64_t*>(b + l.off_keys_b);
        sbox = reinterpret_cast<float4*>(b + l.off_sbox);
        sarea = reinterpret_cast<float*>(b + l.off_sarea);
        state = reinterpret_cast<uint8_t*>(b + l.off_state);
        klist = reinterpret_cast<int32_t*>(b + l.off_klist);
        seg_small = reinterpret_cast<int4*>(b + l.off_seg_small);
        seg_large = reinterpret_cast<int4*>(b + l.off_seg_large);
        seg_huge = reinterpret_cast<int4*>(b + l.off_seg_huge);
        huge_nk = reinterpret_cast<int2*>(b + l.off_huge_nk);
        tier_count = reinterpret_cast<int32_t*>(b + l.off_tier_count);
        tier_box = reinterpret_cast<float4*>(b + l.off_tier_box);
        tier_score = reinterpret_cast<float*>(b + l.off_tier_score);
        tier_cls = reinterpret_cast<int32_t*>(b + l.off_tier_cls);
        tier_id = reinterpret_cast<int32_t*>(b + l.off_tier_id);
        tier_full = reinterpret_cast<FullStats*>(b + l.off_tier_full);
        tier_todo = reinterpret_cast<int32_t*>(b + l.off_tier_todo);
    }
};

using KLL = KeyLayout<kLargeIdxBits>;

// ---- per-image mode + coordinate statistics ------------------------------------------------------
static __global__ void __launch_bounds__(256)
large_stats_kernel(const float4* __restrict__ boxes, const int64_t* __restrict__ cats,
                   const int32_t* __restrict__ counts, int64_t m_max, float thr_f, int mode, LargeImg* info,
                   const int32_t* __restrict__ todo = nullptr) {
    __shared__ float r_max[8], r_min[8];
    __shared__ int r_flag[8];
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int cnt = counts ? counts[img] : (int)m_max;
    cnt = max(0, min(cnt, (int)m_max));
    const bool skip = todo && todo[img] == 0;  // the top-k tier has written this image's result
    if (skip) cnt = 0;
    const bool trick = (mode == DET_NMS_AUTO) ? (cnt <= 1000) : (mode == DET_NMS_OFFSET_TRICK);
    float mx = -INFINITY, mn = INFINITY;
    int fin = 1, maxcat = 0;
    if (trick) {
        for (int i = tid; i < cnt; i += 256) {
            const float4 b = boxes[(int64_t)img * m_max + i];
            mx = max_nan(mx, max_nan(max_nan(b.x, b.y), max_nan(b.z, b.w)));
            mn = min_nan(mn, min_nan(min_nan(b.x, b.y), min_nan(b.z, b.w)));
            fin &= (int)(isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w));
            if (cats) maxcat = max(maxcat, (int)cats[(int64_t)img * m_max + i]);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        fin &= __shfl_xor_sync(0xffffffffu, fin, o);
        maxcat = max(maxcat, __shfl_xor_sync(0xffffffffu, maxcat, o));
    }
    if (lane == 0) {
        r_max[wid] = mx;
        r_min[wid] = mn;
        r_flag[wid] = fin | (maxcat << 1);
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 8; ++w) {
            mx = max_nan(mx, r_max[w]);
            mn = min_nan(mn, r_min[w]);
            fin &= r_flag[w] & 1;
            maxcat = max(maxcat, r_flag[w] >> 1);
        }
        LargeImg li;
        li.cnt = cnt;
        li.trick = trick ? 1 : 0;
        li.span = trick ? mx + 1.0f : 0.f;
        const float far = mx + (float)maxcat * li.span;
        li.fast = (!trick) || (fin && mn > -1.0f && thr_f >= 0.0f && isfinite(far));
        li.nkept = 0;
        li.bad = 0;
        li.nsurv = cnt;
        li.nonan = 1;  // cleared by the gather kernel if it meets a NaN coordinate
        li.skip = skip ? 1 : 0;
        info[img] = li;
    }
}

// ---- top-k tier: the best-scored `want` boxes of an image -> candidate list ----------------------------------------------
// Only max_out survivors are wanted and a box can only be suppressed by a better-scored one, so when max_out is a small
// part of the image the NMS first runs on the want = 1.25 * max_out + 32 best boxes (list_nms_kernel, nms_list.cuh);
// max_out survivors there are exactly the first max_out of the full result.  The cut is the want-th best score to 24
// bits (three radix passes); every box at or above it joins the list, so ties never straddle the cut.  The reference's
// branch rule and the offset trick's span are defined on the whole image: FullStats.  tier_count = -1 hands the
// image to the full path (too few boxes for a tier, a category outside the key range, or a list overflow).
static __global__ void __launch_bounds__(1024)
large_topk_select_kernel(const float4* __restrict__ boxes, const float* __restrict__ scores,
                         const int64_t* __restrict__ cats, const int32_t* __restrict__ counts, int64_t m_max, int mode,
                         int want, int32_t* __restrict__ tier_count, float4* __restrict__ cand_box,
                         float* __restrict__ cand_score, int32_t* __restrict__ cand_cls, int32_t* __restrict__ cand_id,
                         FullStats* __restrict__ full) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix;
    __shared__ int s_want, s_n, s_bad;
    __shared__ float r_max[32], r_min[32];
    __shared__ int r_flag[32];
    constexpr int T = 1024;
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int cnt = counts ? counts[img] : (int)m_max;
    cnt = max(0, min(cnt, (int)m_max));
    int32_t* my_count = tier_count + (int64_t)img * kCountStride;
    if (cnt < want + (want >> 1)) {
        if (tid == 0) *my_count = -1;
        return;
    }
    const float* sc = scores + (int64_t)img * m_max;
    const float4* bx = boxes + (int64_t)img * m_max;
    const int64_t* ct = cats ? cats + (int64_t)img * m_max : nullptr;
    if (tid == 0) {
        s_prefix = 0u;
        s_want = want;
        s_n = 0;
        s_bad = 0;
    }
    for (int shift = 24; shift >= 8; shift -= 8) {
        for (int b = tid; b < 256; b += T) hist[b] = 0u;
        __syncthreads();
        const uint32_t prefix = s_prefix, himask = (shift == 24) ? 0u : (0xffffffffu << (shift + 8));
        for (int i = tid; i < cnt; i += T) {
            const uint32_t key = score_desc_key(sc[i]);
            if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (wid == 0) {
            uint32_t c8[8], tot = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                c8[q] = hist[lane * 8 + q];
                tot += c8[q];
            }
            uint32_t incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                incl += (lane >= o) ? up : 0u;
            }
            const uint32_t w = (uint32_t)s_want, before = incl - tot;
            if (before < w && w <= incl) {
                uint32_t run = before;
                int q = 0;
                for (; q < 7 && run + c8[q] < w; ++q) run += c8[q];
                s_prefix = prefix | ((uint32_t)(lane * 8 + q) << shift);
                s_want = (int)(w - run);
            }
        }
        __syncthreads();
    }
    const uint32_t cut = s_prefix | 0xffu;
    // statistics of the whole image, needed only where the offset trick applies
    const bool trick = (mode == DET_NMS_AUTO) ? (cnt <= 1000) : (mode == DET_NMS_OFFSET_TRICK);
    float mx = -INFINITY, mn = INFINITY;
    int fin = 1, maxcat = 0;
    if (trick) {
        for (int i = tid; i < cnt; i += T) {
            const float4 b = bx[i];
            mx = max_nan(mx, max_nan(max_nan(b.x, b.y), max_nan(b.z, b.w)));
            mn = min_nan(mn, min_nan(min_nan(b.x, b.y), min_nan(b.z, b.w)));
            fin &= (int)(isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w));
        }
    }
    // compaction; every category of the image is looked at (one outside the key range makes the result -1)
    int bad = 0;
    for (int i0 = 0; i0 < cnt; i0 += T) {
        const int i = i0 + tid;
        bool in = false;
        int64_t c = 0;
        float s = 0.f;
        if (i < cnt) {
            c = ct ? ct[i] : 0;
            bad |= (c < 0 || c >= (1 << kSegBits) - 1) ? 1 : 0;
            maxcat = max(maxcat, (int)min(max(c, (int64_t)0), (int64_t)65535));
            s = sc[i];
            in = score_desc_key(s) <= cut;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        int pos = 0;
        if (lane == 0 && bal) pos = atomicAdd(&s_n, __popc(bal));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(bal & ((1u << lane) - 1u));
        if (in && pos < kTierCap) {
            const int64_t o = (int64_t)img * kTierCap + pos;
            cand_box[o] = bx[i];
            cand_score[o] = s;
            cand_cls[o] = (int32_t)c;
            cand_id[o] = i;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        fin &= __shfl_xor_sync(0xffffffffu, fin, o);
        maxcat = max(maxcat, __shfl_xor_sync(0xffffffffu, maxcat, o));
        bad |= __shfl_xor_sync(0xffffffffu, bad, o);
    }
    if (lane == 0) {
        r_max[wid] = mx;
        r_min[wid] = mn;
        r_flag[wid] = fin | (maxcat << 1);
        if (bad) s_bad = 1;
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < T / 32; ++w) {
            mx = max_nan(mx, r_max[w]);
            mn = min_nan(mn, r_min[w]);
            fin &= r_flag[w] & 1;
            maxcat = max(maxcat, r_flag[w] >> 1);
        }
        FullStats f;
        f.count = cnt; f.mx = mx; f.mn = mn; f.fin = fin; f.maxcat = maxcat;
        full[img] = f;
        *my_count = (s_bad || s_n > kTierCap) ? -1 : s_n;
    }
}

// ---- keys ----------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
large_keys_kernel(const float* __restrict__ scores, const int64_t* __restrict__ cats, int64_t m_max, int64_t mp,
                  LargeImg* info, uint64_t* __restrict__ keys) {
    const int img = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= mp) return;
    const LargeImg li = info[img];
    if (li.skip) return;
    uint64_t k = kSentinelKey;
    if (i < li.cnt) {
        const int64_t c = cats ? cats[(int64_t)img * m_max + i] : 0;
        if (c < 0 || c >= (1 << kSegBits) - 1) info[img].bad = 1;
        const bool by_cat = !li.trick || li.fast;
        k = KLL::make(by_cat ? (uint32_t)(c & ((1 << kSegBits) - 1)) : 0u, scores[(int64_t)img * m_max + i], (uint32_t)i);
    }
    keys[(int64_t)img * mp + i] = k;
}

// ---- sort: 2048-key tiles in shared memory, then merge-path passes ------------------------------------
static __global__ void __launch_bounds__(kSortThreads)
sort_tiles_kernel(uint64_t* __restrict__ keys, int64_t mp, const LargeImg* __restrict__ info) {
    __shared__ uint64_t s[kTile];
    if (info && info[blockIdx.y].skip) return;  // nobody reads this image's keys
    uint64_t* g = keys + (int64_t)blockIdx.y * mp + (int64_t)blockIdx.x * kTile;
#pragma unroll
    for (int v = 0; v < kVT; ++v) s[threadIdx.x + v * kSortThreads] = g[threadIdx.x + v * kSortThreads];
    __syncthreads();
    cta_bitonic_sort<kSortThreads>(s, kTile);
#pragma unroll
    for (int v = 0; v < kVT; ++v) g[threadIdx.x + v * kSortThreads] = s[threadIdx.x + v * kSortThreads];
}

// first index a in [lo,hi] of the merge path crossing diagonal d of (A[0..na), B[0..nb)); keys are unique
template <typename P>
__device__ __forceinline__ int64_t merge_path(P A, int64_t na, P B, int64_t nb, int64_t d) {
    int64_t lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (A[mid] < B[d - 1 - mid]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

static __global__ void __launch_bounds__(kSortThreads)
merge_pass_kernel(const uint64_t* __restrict__ in, uint64_t* __restrict__ out, int64_t mp, int64_t len, int64_t width,
                  const LargeImg* __restrict__ info) {
    __shared__ uint64_t s[kTile];
    __shared__ int64_t s_cut[2];
    if (info && info[blockIdx.y].skip) return;
    const uint64_t* kin = in + (int64_t)blockIdx.y * mp;
    uint64_t* kout = out + (int64_t)blockIdx.y * mp;
    const int64_t out0 = (int64_t)blockIdx.x * kTile;
    const int64_t lo = out0 / (2 * width) * (2 * width);
    const int64_t a_len = min(width, len - lo);
    const int64_t b_lo = lo + a_len;
    const int64_t b_len = max((int64_t)0, min(width, len - b_lo));
    const uint64_t* A = kin + lo;
    const uint64_t* B = kin + b_lo;
    const int64_t d0 = out0 - lo, d1 = min(d0 + (int64_t)kTile, a_len + b_len);
    if (threadIdx.x < 2) s_cut[threadIdx.x] = merge_path(A, a_len, B, b_len, threadIdx.x ? d1 : d0);
    __syncthreads();
    const int64_t a0 = s_cut[0], a1 = s_cut[1];
    const int64_t b0 = d0 - a0, b1 = d1 - a1;
    const int na = (int)(a1 - a0), nb = (int)(b1 - b0);
    for (int t = threadIdx.x; t < na; t += kSortThreads) s[t] = A[a0 + t];
    for (int t = threadIdx.x; t < nb; t += kSortThreads) s[na + t] = B[b0 + t];
    __syncthreads();
    const uint64_t* sa = s;
    const uint64_t* sb = s + na;
    const int total = na + nb;
    const int diag = min((int)threadIdx.x * kVT, total);
    int ai = (int)merge_path(sa, (int64_t)na, sb, (int64_t)nb, (int64_t)diag);
    int bi = diag - ai;
    uint64_t r[kVT];
#pragma unroll
    for (int v = 0; v < kVT; ++v) {
        const bool has = diag + v < total;
        const bool take_a = has && (bi >= nb || (ai < na && sa[ai] < sb[bi]));
        r[v] = has ? (take_a ? sa[ai] : sb[bi]) : 0;
        ai += (has && take_a) ? 1 : 0;
        bi += (has && !take_a) ? 1 : 0;
    }
#pragma unroll
    for (int v = 0; v < kVT; ++v)
        if (diag + v < total) kout[out0 + diag + v] = r[v];
}

// sorts the first `len` keys (a multiple of kTile; default: all mp) of every image's row ascending; rows are mp keys
// apart; returns the buffer that holds the result
static uint64_t* sort_rows(uint64_t* a, uint64_t* b, int n, int64_t mp, cudaStream_t st,
                           const LargeImg* info = nullptr, int64_t len = 0) {
    if (len <= 0) len = mp;
    dim3 grid((unsigned)(len / kTile), (unsigned)n);
    sort_tiles_kernel<<<grid, kSortThreads, 0, st>>>(a, mp, info);
    uint64_t *src = a, *dst = b;
    for (int64_t width = kTile; width < len; width *= 2) {
        merge_pass_kernel<<<grid, kSortThreads, 0, st>>>(src, dst, mp, len, width, info);
        uint64_t* t = src;
        src = dst;
        dst = t;
    }
    return src;
}

// push segment [s,e) of image img on the short, long or huge work list
// warp_max: longest segment handed to a single warp.  A lone warp needs > 100 us for 256 boxes (latency-bound), which
// is right when there are thousands of segments and wrong when there are a few hundred (RPN levels): those go to CTAs.
__device__ __forceinline__ void push_segment(int img, int s, int e, int32_t* ctr, int4* seg_small, int4* seg_large,
                                             int4* seg_huge, int2* huge_nk, int warp_max = kLargeWarpSegMax,
                                             int cta_max = kHugeSeg) {
    if (e - s <= warp_max) {
        const int slot = atomicAdd(&ctr[0], 1);
        seg_small[slot] = make_int4(img, s, e, 0);
    } else if (e - s <= cta_max) {
        const int slot = atomicAdd(&ctr[1], 1);
        seg_large[slot] = make_int4(img, s, e, 0);
    } else {
        const int slot = atomicAdd(&ctr[4], 1);
        seg_huge[slot] = make_int4(img, s, e, 0);
        huge_nk[slot] = make_int2(0, 0);
    }
}

// upper end of the segment that starts at p: first position in (p, cnt) whose segment field differs
__device__ __forceinline__ int segment_end(const uint64_t* k, int p, int cnt, uint32_t sg) {
    int lo = p + 1, hi = cnt;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (KLL::seg(k[mid]) > sg) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// ---- gather boxes into sorted order (+ coordinate offset), discover segments -------------------------
static __global__ void __launch_bounds__(256)
large_gather_kernel(const float4* __restrict__ boxes, const int64_t* __restrict__ cats, int64_t m_max, int64_t mp,
                    LargeImg* info, const uint64_t* __restrict__ keys, float4* __restrict__ sbox,
                    float* __restrict__ sarea, uint8_t* __restrict__ state, int32_t* ctr, int4* seg_small,
                    int4* seg_large, int4* seg_huge, int2* huge_nk) {
    const int img = blockIdx.y;
    const int p = blockIdx.x * 256 + threadIdx.x;
    const LargeImg li = info[img];
    if (p >= li.cnt) return;
    const uint64_t* k = keys + (int64_t)img * mp;
    const uint64_t key = k[p];
    const int i = (int)KLL::idx(key);
    float4 b = boxes[(int64_t)img * m_max + i];
    if (li.trick) {
        const int64_t c = cats ? cats[(int64_t)img * m_max + i] : 0;
        const float off = (float)c * li.span;
        b.x += off; b.y += off; b.z += off; b.w += off;
    }
    sbox[(int64_t)img * mp + p] = b;
    sarea[(int64_t)img * mp + p] = box_area(b);
    state[(int64_t)img * mp + p] = 0;
    if (!((b.x == b.x) && (b.y == b.y) && (b.z == b.z) && (b.w == b.w))) info[img].nonan = 0;
    const uint32_t sg = KLL::seg(key);
    if (p == 0 || KLL::seg(k[p - 1]) != sg) push_segment(img, p, segment_end(k, p, li.cnt, sg), ctr, seg_small, seg_large, seg_huge, huge_nk);
}

// ---- persistent segment kernels ---------------------------------------------------------------------------
static __global__ void __launch_bounds__(128)
large_warp_segments_kernel(int64_t mp, const LargeImg* __restrict__ info, const float4* __restrict__ sbox,
                           const float* __restrict__ sarea, uint8_t* state, int32_t* klist, int32_t* ctr,
                           const int4* __restrict__ seg_small, float thr_f, int max_keep) {
    const int lane = threadIdx.x & 31;
    const int total = ctr[0];
    while (true) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&ctr[2], 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= total) break;
        const int4 sg = seg_small[i];
        const int64_t o = (int64_t)sg.x * mp;
        if (info[sg.x].nonan)
            warp_segment_nms<int32_t, true>(sbox + o, sarea + o, state + o, klist + o, sg.y, sg.z, thr_f, max_keep);
        else
            warp_segment_nms<int32_t, false>(sbox + o, sarea + o, state + o, klist + o, sg.y, sg.z, thr_f, max_keep);
    }
}

// stage boxes + areas of positions [s, e) in shared memory; returns pointers that are indexed with the GLOBAL position
struct StagedBoxes {
    const float4* box;
    const float* area;
};
__device__ __forceinline__ StagedBoxes stage_boxes(const float4* __restrict__ sbox, const float* __restrict__ sarea, int s,
                                                   int e, float4* sm_box, float* sm_area) {
    for (int p = s + (int)threadIdx.x; p < e; p += (int)blockDim.x) {
        sm_box[p - s] = sbox[p];
        sm_area[p - s] = sarea[p];
    }
    __syncthreads();
    return StagedBoxes{sm_box - s, sm_area - s};
}

// segments of 257 .. kHugeSeg boxes: one CTA each, the whole segment staged in shared memory (80 KB) so that the
// kept-list tests and the chunk bit rows never wait for L2
static __global__ void __launch_bounds__(kSegCtaThreads)
large_cta_segments_kernel(int64_t mp, const LargeImg* __restrict__ info, const float4* __restrict__ sbox,
                          const float* __restrict__ sarea, uint8_t* state, int32_t* klist, int32_t* ctr,
                          const int4* __restrict__ seg_large, float thr_f, int max_keep) {
    extern __shared__ __align__(16) unsigned char seg_smem[];
    float4* sm_box = reinterpret_cast<float4*>(seg_smem);
    float* sm_area = reinterpret_cast<float*>(sm_box + kHugeSeg);
    __shared__ uint32_t rowbits[kSegThreads * (kSegThreads / 32)];
    __shared__ uint32_t amask[kSegThreads / 32], deadmask[kSegThreads / 32];
    __shared__ int s_nk, s_next;
    const int total = ctr[1];
#ifdef DET_DEBUG_PHASES
    if (total == 0) return;
#endif
    DET_MARK(0);
#ifdef DET_DEBUG_PHASES
    if (blockIdx.x < 64 && threadIdx.x == 0) g_phase_block[blockIdx.x][2] = g_phase_block[blockIdx.x][3] = 0;
#endif
    while (true) {
        if (threadIdx.x == 0) s_next = atomicAdd(&ctr[3], 1);
        __syncthreads();
        const int i = s_next;
        __syncthreads();
        if (i >= total) break;
        const int4 sg = seg_large[i];
        if (sg.w != 0) continue;  // done by large_bin_segments_kernel
#ifdef DET_DEBUG_PHASES
        if (blockIdx.x < 64 && threadIdx.x == 0) {
            g_phase_block[blockIdx.x][2] += 1;
            g_phase_block[blockIdx.x][3] += sg.z - sg.y;
        }
#endif
        const int64_t o = (int64_t)sg.x * mp;
        const StagedBoxes sb = stage_boxes(sbox + o, sarea + o, sg.y, sg.z, sm_box, sm_area);
        if (info[sg.x].nonan)
            cta_segment_nms<kSegThreads, int32_t, true>(sb.box, sb.area, state + o, klist + o, sg.y, sg.z, thr_f, max_keep,
                                                        rowbits, amask, deadmask, &s_nk);
        else
            cta_segment_nms<kSegThreads, int32_t, false>(sb.box, sb.area, state + o, klist + o, sg.y, sg.z, thr_f, max_keep,
                                                         rowbits, amask, deadmask, &s_nk);
        __syncthreads();
    }
    DET_MARK(1);
}

// ---- CTA-class segments through a spatial index (most pairs of a long segment never overlap) -----------------------------
// The sweep above tests every candidate against every kept box before it: O(kept x boxes) pair tests and a serial chain
// of 256-box chunks -- 190 us for the ~960 best level-0 proposals of an RPN image, 90 % of which survive.  For an IoU
// threshold of at least 0.5 a suppressing pair is confined in space: inter / union > 0.5 means that the intersection
// covers more than half of EITHER box in x and in y, hence it contains both centres; in particular
//     box j suppresses box i  =>  the centre of j lies inside box i.
// So every candidate is filed under the grid cell of its centre (one linked-list node per box), and box i only meets the
// boxes filed in the cells its own extent reaches, and of those only the better-scored ones whose centre it contains:
//   1  stage the segment; bounding range of the centres, largest |coordinate|; a segment with a non-finite coordinate or
//      an area outside [1e-30, 1e30] (where the rounding of the areas could defeat the argument) is left to the sweep
//   2  file the candidates by centre cell (GB x GB cells over the range of the centres; the cell function is monotone in
//      the coordinate, and the query extent is widened by m = 2^-16 x the largest |coordinate|, far more than the
//      rounding of the centre and of the IoU quotient can move anything)
//   3  every candidate collects its SUPPRESSORS -- better-scored boxes j with nms_suppresses(j, i), the same predicate
//      on the same operands as the sweep -- up to kBinEdges of them; one with more re-walks its cells when asked
//   4  greedy order without a chain over the boxes: a candidate with no suppressor is kept; in rounds, an undecided
//      candidate dies if one of its suppressors is kept and is kept once all of them are dead.  The best undecided
//      candidate is always decidable, so this terminates with exactly the sweep's result; after kBinRounds rounds
//      (a long dependency chain) the segment is left to the sweep
//   5  the first max_keep kept positions get state 2, as the sweep would leave them
// Segments handled here are marked in seg_large[i].w; large_cta_segments_kernel skips them.
constexpr int kBinThreads = 512;
constexpr int kBinEdges = 4;
constexpr int kBinRounds = 48;
constexpr int kBinCells = 32;     // cells per axis for segments of more than kBinFineSeg boxes, half that for shorter ones
constexpr int kBinFineSeg = 1024;  // passed as the kernel's bin_fine: compiled in, it changed the kernel's schedule and
                                   // cost 6 % on clustered RPN proposals (2.02 vs 1.90 ms per 64 images, B200 at 1000 W)

struct BinSmem {
    float4 box[kHugeSeg];
    uint16_t next[kHugeSeg];
    uint16_t edge[kHugeSeg * kBinEdges];
    uint8_t meta[kHugeSeg];  // bits 0-2: stored suppressors, bit 3: there are more, bits 4-5: 0 undecided 1 dead 2 kept
    int head[kBinCells * kBinCells];
};

struct BinGrid {
    float x0, y0, ix, iy, m, top;
    int gb;
    __device__ __forceinline__ int cx(float x) const { return (int)fminf(fmaxf((x - x0) * ix, 0.0f), top); }
    __device__ __forceinline__ int cy(float y) const { return (int)fminf(fmaxf((y - y0) * iy, 0.0f), top); }
};

// walks the better-scored boxes filed in the cells box q reaches; f(j, box_j) -> true stops the walk
template <typename F>
__device__ __forceinline__ void bin_walk(const BinSmem& sm, const BinGrid& g, int q, const float4 bi, F f) {
    const float lx = bi.x - g.m, hx = bi.z + g.m, ly = bi.y - g.m, hy = bi.w + g.m;
    const int c0 = g.cx(lx), c1 = g.cx(hx), r0 = g.cy(ly), r1 = g.cy(hy);
    for (int r = r0; r <= r1; ++r)
        for (int c = c0; c <= c1; ++c)
            for (int j = sm.head[r * g.gb + c]; j >= 0; j = (sm.next[j] == 0xFFFFu) ? -1 : (int)sm.next[j]) {
                if (j >= q) continue;
                const float4 bj = sm.box[j];
                const float xj = 0.5f * (bj.x + bj.z), yj = 0.5f * (bj.y + bj.w);
                if (xj < lx || xj > hx || yj < ly || yj > hy) continue;
                if (f(j, bj)) return;
            }
}

static __global__ void __launch_bounds__(kBinThreads, 2)
large_bin_segments_kernel(int64_t mp, const float4* __restrict__ sbox, uint8_t* state, int32_t* ctr, int4* seg_large,
                          float thr_f, int max_keep, int bin_fine, const LargeImg* __restrict__ info,
                          const float* __restrict__ sarea, int32_t* klist, const int4* __restrict__ seg_small) {
    extern __shared__ __align__(16) unsigned char bin_smem[];
    BinSmem& sm = *reinterpret_cast<BinSmem*>(bin_smem);
    __shared__ float s_red[kBinThreads / 32][5];
    __shared__ int s_bad[kBinThreads / 32], s_wc[kBinThreads / 32];
    __shared__ int s_next;
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    constexpr int NW = kBinThreads / 32;
    const int total = ctr[1];
    while (true) {
        __syncthreads();
        if (tid == 0) s_next = atomicAdd(&ctr[6], 1);
        __syncthreads();
        const int i = s_next;
        if (i >= total) break;
        const int4 sg = seg_large[i];
        const int n = sg.z - sg.y;
        const int64_t o = (int64_t)sg.x * mp + sg.y;
        // ---- 1: stage, statistics
        float xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY, amax = 0.0f;
        int bad = 0;
        for (int q = tid; q < n; q += kBinThreads) {
            const float4 b = sbox[o + q];
            const bool cand = state[o + q] == 0;
            sm.box[q] = b;
            sm.meta[q] = cand ? 0 : (1u << 4);
            if (cand) {
                const float a = box_area(b);
                const bool fin = isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w);
                if (!fin || (a > 0.0f && a < 1e-30f) || a > 1e30f) bad = 1;
                const float xc = 0.5f * (b.x + b.z), yc = 0.5f * (b.y + b.w);
                xmin = fminf(xmin, xc); xmax = fmaxf(xmax, xc);
                ymin = fminf(ymin, yc); ymax = fmaxf(ymax, yc);
                amax = fmaxf(amax, fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w))));
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            xmin = fminf(xmin, __shfl_xor_sync(FULL, xmin, d)); xmax = fmaxf(xmax, __shfl_xor_sync(FULL, xmax, d));
            ymin = fminf(ymin, __shfl_xor_sync(FULL, ymin, d)); ymax = fmaxf(ymax, __shfl_xor_sync(FULL, ymax, d));
            amax = fmaxf(amax, __shfl_xor_sync(FULL, amax, d));
            bad |= __shfl_xor_sync(FULL, bad, d);
        }
        if (lane == 0) {
            s_red[wid][0] = xmin; s_red[wid][1] = xmax; s_red[wid][2] = ymin; s_red[wid][3] = ymax; s_red[wid][4] = amax;
            s_bad[wid] = bad;
        }
        for (int c = tid; c < kBinCells * kBinCells; c += kBinThreads) sm.head[c] = -1;
        __syncthreads();
        for (int w = 0; w < NW; ++w) {
            xmin = fminf(xmin, s_red[w][0]); xmax = fmaxf(xmax, s_red[w][1]);
            ymin = fminf(ymin, s_red[w][2]); ymax = fmaxf(ymax, s_red[w][3]);
            amax = fmaxf(amax, s_red[w][4]);
            bad |= s_bad[w];
        }
        // (coordinates of at least 1e-20 keep the widening m far above the absolute error of denormal extents)
        if (bad || !(amax < 1e15f) || !(amax > 1e-20f)) continue;  // the barrier at the top of the loop separates the iterations
        BinGrid g;
        g.gb = n > bin_fine ? kBinCells : kBinCells / 2;
        g.top = (float)(g.gb - 1);
        g.x0 = xmin; g.y0 = ymin;
        const float rx = xmax - xmin, ry = ymax - ymin;
        g.ix = (rx > 0.0f && (float)g.gb / rx < 1e30f) ? (float)g.gb / rx : 0.0f;
        g.iy = (ry > 0.0f && (float)g.gb / ry < 1e30f) ? (float)g.gb / ry : 0.0f;
        g.m = amax * 1.52587890625e-05f;
        // ---- 2: file the candidates under the cell of their centre
        for (int q = tid; q < n; q += kBinThreads) {
            if (sm.meta[q]) continue;
            const float4 b = sm.box[q];
            const int cell = g.cy(0.5f * (b.y + b.w)) * g.gb + g.cx(0.5f * (b.x + b.z));
            const int old = atomicExch(&sm.head[cell], q);
            sm.next[q] = old < 0 ? (uint16_t)0xFFFFu : (uint16_t)old;
        }
        __syncthreads();
        // ---- 3: suppressors of every candidate
        for (int q = tid; q < n; q += kBinThreads) {
            if (sm.meta[q]) continue;
            const float4 bi = sm.box[q];
            const float ai = box_area(bi);
            int cnt = 0;
            bool more = false;
            bin_walk(sm, g, q, bi, [&](int j, const float4 bj) {
                if (!nms_suppresses<true>(bj, box_area(bj), bi, ai, thr_f)) return false;
                if (cnt == kBinEdges) {
                    more = true;
                    return true;
                }
                sm.edge[q * kBinEdges + cnt++] = (uint16_t)j;
                return false;
            });
            sm.meta[q] = (uint8_t)(cnt | (more ? 8 : 0) | (cnt == 0 ? (2 << 4) : 0));
        }
        __syncthreads();
        // ---- 4: rounds
        const volatile uint8_t* vmeta = sm.meta;
        int pending_any = 1;
        for (int round = 0; round < kBinRounds && pending_any; ++round) {
            int pending = 0;
            for (int q = tid; q < n; q += kBinThreads) {
                const unsigned mq = vmeta[q];
                if (mq >> 4) continue;
                bool kept_sup = false, open_sup = false;
                const int cnt = (int)(mq & 7u);
                for (int k = 0; k < cnt; ++k) {
                    const unsigned st = vmeta[sm.edge[q * kBinEdges + k]] >> 4;
                    kept_sup |= st == 2u;
                    open_sup |= st == 0u;
                }
                if (!kept_sup && (mq & 8u)) {  // more suppressors than the list holds: look at all of them again
                    const float4 bi = sm.box[q];
                    const float ai = box_area(bi);
                    bin_walk(sm, g, q, bi, [&](int j, const float4 bj) {
                        const unsigned st = vmeta[j] >> 4;
                        if (st == 1u || !nms_suppresses<true>(bj, box_area(bj), bi, ai, thr_f)) return false;
                        if (st == 2u) {
                            kept_sup = true;
                            return true;
                        }
                        open_sup = true;
                        return false;
                    });
                }
                if (kept_sup) sm.meta[q] = (uint8_t)(mq | (1u << 4));
                else if (!open_sup) sm.meta[q] = (uint8_t)(mq | (2u << 4));
                else pending = 1;
            }
            pending_any = __syncthreads_or(pending);
        }
        if (pending_any) continue;
        // ---- 5: the first max_keep kept positions
        int running = 0;
        for (int base = 0; base < n && running < max_keep; base += kBinThreads) {
            const int q = base + tid;
            const bool k = q < n && (sm.meta[q] >> 4) == 2u;
            const unsigned bal = __ballot_sync(FULL, k);
            if (lane == 0) s_wc[wid] = __popc(bal);
            __syncthreads();
            int pre = 0, tot = 0;
            for (int w = 0; w < NW; ++w) {
                const int v = s_wc[w];
                pre += w < wid ? v : 0;
                tot += v;
            }
            const int rank = running + pre + __popc(bal & ((1u << lane) - 1u));
            if (k && rank < max_keep) state[o + q] = 2;
            running += tot;
            __syncthreads();
        }
        if (tid == 0) seg_large[i].w = 1;
    }
    // The short segments (one warp each, large_warp_segments_kernel's loop) ride in the CTAs that have run out of long
    // ones: the lists are disjoint, and a launch of its own cost 8-12 us of mostly latency in front of this kernel.
    if (seg_small) {
        const int total_s = ctr[0];
        while (true) {
            int i = 0;
            if (lane == 0) i = atomicAdd(&ctr[2], 1);
            i = __shfl_sync(FULL, i, 0);
            if (i >= total_s) break;
            const int4 sg = seg_small[i];
            const int64_t o = (int64_t)sg.x * mp;
            if (info[sg.x].nonan)
                warp_segment_nms<int32_t, true>(sbox + o, sarea + o, state + o, klist + o, sg.y, sg.z, thr_f, max_keep);
            else
                warp_segment_nms<int32_t, false>(sbox + o, sarea + o, state + o, klist + o, sg.y, sg.z, thr_f, max_keep);
        }
    }
}

// ---- huge segments (one category with many thousands of boxes): the whole grid works on them together ----------
// Greedy NMS in score order, kHugeChunk positions per step.  In step `it`
//   * the segment's leader CTA first applies the kept boxes of chunk it-1 to the positions of chunk it, then resolves
//     chunk it internally (cta_segment_nms on a shared-memory copy) and appends its survivors to the kept list;
//   * meanwhile every other CTA (and the leaders once done) applies the kept boxes of chunk it-1 to the still-alive
//     positions BEHIND chunk it;
// then one grid-wide barrier.  The serial part (a 1024-box resolve) is thus hidden behind the O(kept x remaining) bulk
// of the previous chunk, which is spread over all SMs.  All huge segments (typically one per image) advance in lock
// step; a segment stops as soon as it has max_keep survivors.
// huge_nk[h] = (kept so far, first kept of the newest chunk); huge_prev[h] (second int2) = the same pair one step ago.
template <bool NONAN>
__device__ __forceinline__ void huge_apply(const float4* __restrict__ sbox, const float* __restrict__ sarea, uint8_t* state,
                                           const int32_t* klist_seg, int k0, int k1, int p, int pe, float thr_f) {
    // one position per thread of the CTA (p may be >= pe for the tail): warp-collective
    bool alive = p < pe && state[p] == 0;
    float4 mb = make_float4(0.f, 0.f, 0.f, 0.f);
    float ma = 0.f;
    if (alive) {
        mb = sbox[p];
        ma = sarea[p];
    }
    const bool was = alive;
    alive = alive_after_kept<int32_t, NONAN>(sbox, sarea, klist_seg, k0, k1, mb, ma, alive, thr_f);
    if (was && !alive) state[p] = 1;
}

static __global__ void __launch_bounds__(kSegCtaThreads)
large_huge_segments_kernel(int64_t mp, const LargeImg* __restrict__ info, const float4* __restrict__ sbox,
                           const float* __restrict__ sarea, uint8_t* state, int32_t* klist,
                           const int32_t* __restrict__ ctr, const int4* __restrict__ seg_huge, int2* huge_nk, float thr_f,
                           int max_keep) {
    namespace cg = cooperative_groups;
    __shared__ __align__(16) float4 sm_box[kHugeChunk];
    __shared__ float sm_area[kHugeChunk];
    __shared__ uint32_t rowbits[kSegThreads * (kSegThreads / 32)];
    __shared__ uint32_t amask[kSegThreads / 32], deadmask[kSegThreads / 32];
    __shared__ int s_nk;
    const int nh = ctr[4];
    if (nh == 0) return;  // grid-uniform
    cg::grid_group grid = cg::this_grid();
    int max_chunks = 0;
    for (int h = 0; h < nh; ++h) {
        const int4 sg = seg_huge[h];
        max_chunks = max(max_chunks, (sg.z - sg.y + kHugeChunk - 1) / kHugeChunk);
    }
    // kept ranges are double-buffered by step parity: range[it & 1] is written by the leader in step it and read by
    // everybody in step it + 1
    int2* range0 = huge_nk;            // [nh]: x = kept so far (running), y unused
    int2* ranges = huge_nk + nh;       // [2][nh]: (first, last) kept entry of the chunk resolved in that step
    for (int it = 0; it < max_chunks; ++it) {
        const int2* prev = ranges + ((it + 1) & 1) * nh;  // written in step it - 1
        int2* cur = ranges + (it & 1) * nh;
        // ---- leaders: bring chunk `it` up to date, resolve it
        for (int h = blockIdx.x; h < nh; h += gridDim.x) {
            const int4 sg = seg_huge[h];
            const int64_t o = (int64_t)sg.x * mp;
            const int base = sg.y + it * kHugeChunk;
            const int nk0 = range0[h].x;
            __syncthreads();
            if (base >= sg.z || nk0 >= max_keep) {
                if (threadIdx.x == 0) cur[h] = make_int2(nk0, nk0);  // nothing new to apply next step
                continue;
            }
            const int end = min(base + kHugeChunk, sg.z);
            if (it > 0 && prev[h].y > prev[h].x)
                for (int p0 = base; p0 < end; p0 += kSegCtaThreads) {
                    if (info[sg.x].nonan)
                        huge_apply<true>(sbox + o, sarea + o, state + o, klist + o + sg.y, prev[h].x, prev[h].y,
                                         p0 + (int)threadIdx.x, end, thr_f);
                    else
                        huge_apply<false>(sbox + o, sarea + o, state + o, klist + o + sg.y, prev[h].x, prev[h].y,
                                          p0 + (int)threadIdx.x, end, thr_f);
                }
            __syncthreads();
            const StagedBoxes sb = stage_boxes(sbox + o, sarea + o, base, end, sm_box, sm_area);
            // kept list of the segment lives at klist[o + sg.y ...]; the chunk appends at entry nk0
            int32_t* kl = klist + o + (sg.y + nk0 - base);
            const int nk = info[sg.x].nonan
                               ? cta_segment_nms<kSegThreads, int32_t, true>(sb.box, sb.area, state + o, kl, base, end, thr_f,
                                                                             max_keep - nk0, rowbits, amask, deadmask, &s_nk)
                               : cta_segment_nms<kSegThreads, int32_t, false>(sb.box, sb.area, state + o, kl, base, end, thr_f,
                                                                              max_keep - nk0, rowbits, amask, deadmask, &s_nk);
            __syncthreads();
            if (threadIdx.x == 0) {
                cur[h] = make_int2(nk0, nk0 + nk);
                range0[h].x = nk0 + nk;
            }
        }
        // ---- everybody: kept boxes of chunk it-1 against the alive positions behind chunk it
        if (it > 0) {
            int unit0 = 0;
            for (int h = 0; h < nh; ++h) {
                const int4 sg = seg_huge[h];
                const int2 pr = prev[h];
                const int first = sg.y + (it + 1) * kHugeChunk;
                const int rem = sg.z - first;
                if (rem <= 0 || pr.y <= pr.x) continue;
                const int units = (rem + kSegCtaThreads - 1) / kSegCtaThreads;
                const int64_t o = (int64_t)sg.x * mp;
                // rotate the starting CTA from segment to segment so that short tails do not land on the same CTAs
                const bool nn = info[sg.x].nonan != 0;
                for (int u = (int)((blockIdx.x + gridDim.x - unit0 % gridDim.x) % gridDim.x); u < units; u += gridDim.x) {
                    const int p = first + u * kSegCtaThreads + (int)threadIdx.x;
                    if (nn) huge_apply<true>(sbox + o, sarea + o, state + o, klist + o + sg.y, pr.x, pr.y, p, sg.z, thr_f);
                    else huge_apply<false>(sbox + o, sarea + o, state + o, klist + o + sg.y, pr.x, pr.y, p, sg.z, thr_f);
                }
                unit0 += units;
            }
        }
        grid.sync();
    }
}

// ---- kept -> output keys, count -----------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
large_rekey_kernel(int64_t mp, LargeImg* info, const uint64_t* __restrict__ keys, const uint8_t* __restrict__ state,
                   uint64_t* __restrict__ keys_out) {
    const int img = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (info[img].skip) return;
    const int cnt = info[img].cnt;
    bool kept = false;
    if (p < mp) {
        kept = (p < cnt) && state[(int64_t)img * mp + p] == 2;
        keys_out[(int64_t)img * mp + p] = kept ? KLL::strip_seg(keys[(int64_t)img * mp + p]) : kSentinelKey;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, kept);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&info[img].nkept, __popc(bal));
}

static __global__ void __launch_bounds__(256)
large_emit_kernel(int64_t mp, const LargeImg* __restrict__ info, const uint64_t* __restrict__ keys, int64_t max_out,
                  int64_t* __restrict__ keep, int32_t* __restrict__ keep_counts) {
    const int img = blockIdx.y;
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const LargeImg li = info[img];
    if (li.skip) return;
    const int64_t nout = li.bad ? 0 : min((int64_t)li.nkept, max_out);
    if (j < nout) keep[(int64_t)img * max_out + j] = (int64_t)KLL::idx(keys[(int64_t)img * mp + j]);
    if (j == 0) keep_counts[img] = li.bad ? -1 : (int32_t)nout;
}

static int launch_list_nms_ext(const int32_t* tier_count, const float4* box, const float* score, const int32_t* cls,
                               const int32_t* id, int n, float thr_f, int mode, int64_t max_out, int64_t* keep,
                               int32_t* keep_counts, const FullStats* full, int32_t* todo, cudaStream_t st) {
    constexpr int T = 512;  // 180 KB of shared memory per CTA: one CTA per SM either way
    const size_t smem = sizeof(DetectSmem<kTierCap, T>);
    static thread_local bool attr_set = false;
    if (!attr_set) {
        cudaError_t ea = cudaFuncSetAttribute(dense_detect_nms_kernel<kTierCap, T>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (ea != cudaSuccess) return cuda_fail(ea, "cudaFuncSetAttribute(list nms)");
        attr_set = true;
    }
    dense_detect_nms_kernel<kTierCap, T><<<n, T, smem, st>>>(const_cast<int32_t*>(tier_count), box, score, cls, id, kTierCap, thr_f, mode,
                                                             max_out, keep, nullptr, nullptr, nullptr, keep_counts,
                                                             nullptr, full, todo);
    DET_LAUNCH_OK("list_nms_kernel(ext)");
    return DET_OK;
}

// runs the two persistent segment kernels over the lists built by a gather kernel
// few_small: the caller knows that short segments are few (RPN levels: at most a couple per image) -- they then ride in
// large_bin_segments_kernel; thousands of short segments (per-category NMS) keep their own launch at twice the resident warps
static int run_segment_kernels(const LargeLayout& lay, const LargeWs& ws, float thr_f, int max_keep, cudaStream_t st,
                               bool few_small = false) {
    const int sms = sm_count();
    const bool bins = thr_f >= 0.5f;  // spatial index: needs "a suppressor's centre lies inside the box" (IoU > 1/2)
    if (!(bins && few_small)) {  // otherwise the short segments ride in large_bin_segments_kernel
        large_warp_segments_kernel<<<sms * 8, 128, 0, st>>>(lay.mp, ws.info, ws.sbox, ws.sarea, ws.state, ws.klist, ws.ctr,
                                                            ws.seg_small, thr_f, max_keep);
        DET_LAUNCH_OK("large_warp_segments_kernel");
    }
    const int seg_smem = kHugeSeg * 20;
    static thread_local bool attr_set = false;
    if (!attr_set) {
        cudaError_t ea = cudaFuncSetAttribute(large_cta_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, seg_smem);
        if (ea != cudaSuccess) return cuda_fail(ea, "cudaFuncSetAttribute(large_cta_segments_kernel)");
        ea = cudaFuncSetAttribute(large_bin_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BinSmem));
        if (ea != cudaSuccess) return cuda_fail(ea, "cudaFuncSetAttribute(large_bin_segments_kernel)");
        attr_set = true;
    }
    if (bins) {
        large_bin_segments_kernel<<<sms * 2, kBinThreads, sizeof(BinSmem), st>>>(lay.mp, ws.sbox, ws.state, ws.ctr, ws.seg_large,
                                                                              thr_f, max_keep, kBinFineSeg, ws.info, ws.sarea, ws.klist,
                                                                              few_small ? ws.seg_small : nullptr);
        DET_LAUNCH_OK("large_bin_segments_kernel");
    }
    large_cta_segments_kernel<<<sms * 2, kSegCtaThreads, seg_smem, st>>>(lay.mp, ws.info, ws.sbox, ws.sarea, ws.state, ws.klist, ws.ctr,
                                                                      ws.seg_large, thr_f, max_keep);
    DET_LAUNCH_OK("large_cta_segments_kernel");
    // cooperative launch: every CTA must be resident (grid barriers); it returns at once when there is no huge segment
    static thread_local int per_sm = 0;
    if (per_sm == 0) {
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, large_huge_segments_kernel, kSegCtaThreads, 0);
        if (e != cudaSuccess || per_sm < 1) return cuda_fail(e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
        if (per_sm > 4) per_sm = 4;
    }
    int64_t mp_arg = lay.mp;
    const LargeImg* info_arg = ws.info;
    const float4* sbox_arg = ws.sbox;
    const float* sarea_arg = ws.sarea;
    uint8_t* state_arg = ws.state;
    int32_t* klist_arg = ws.klist;
    const int32_t* ctr_arg = ws.ctr;
    const int4* huge_arg = ws.seg_huge;
    int2* nk_arg = ws.huge_nk;
    void* args[] = {&mp_arg, &info_arg, &sbox_arg, &sarea_arg, &state_arg, &klist_arg, &ctr_arg, &huge_arg, &nk_arg, &thr_f, &max_keep};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)large_huge_segments_kernel, dim3((unsigned)(sms * per_sm)),
                                                dim3(kSegCtaThreads), args, 0, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchCooperativeKernel(large_huge_segments_kernel)");
    return DET_OK;
}

static int large_nms_run(const LargeLayout& lay, void* workspace, const float* boxes, const float* scores,
                         const int64_t* cats, const int32_t* counts, float thr_f, int mode, int64_t max_out,
                         int64_t* keep, int32_t* keep_counts, cudaStream_t st) {
    LargeWs ws(lay, workspace);
    const int n = lay.n;
    const int64_t mp = lay.mp;
    auto b4 = reinterpret_cast<const float4*>(boxes);
    cudaError_t e = cudaMemsetAsync(ws.ctr, 0, 64, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    // top-k tier: when max_out is a small part of the image, sweep the best-scored boxes first (see
    // large_topk_select_kernel); images that get their max_out survivors there skip everything below
    // the list holds twice the first tier (capped): list_nms_kernel sweeps the best 1.25 * max_out + 32 of it first and
    // the whole list if those fall short (low survival, e.g. one category), before an image goes to the full path
    const int64_t tier1 = max_out + (max_out >> 2) + 32;
    const int64_t want = tier1 * 2 < kTierMaxWant ? tier1 * 2 : (tier1 < kTierMaxWant ? kTierMaxWant : tier1);
    const int32_t* todo = nullptr;
    if (max_out >= 1 && want <= kTierMaxWant && want + (want >> 1) <= lay.m_max) {
        large_topk_select_kernel<<<n, 1024, 0, st>>>(b4, scores, cats, counts, lay.m_max, mode, (int)want, ws.tier_count,
                                                     ws.tier_box, ws.tier_score, ws.tier_cls, ws.tier_id, ws.tier_full);
        DET_LAUNCH_OK("large_topk_select_kernel");
        const int rc = launch_list_nms_ext(ws.tier_count, ws.tier_box, ws.tier_score, ws.tier_cls, ws.tier_id, n, thr_f,
                                           mode, max_out, keep, keep_counts, ws.tier_full, ws.tier_todo, st);
        if (rc != DET_OK) return rc;
        todo = ws.tier_todo;
    }
    large_stats_kernel<<<n, 256, 0, st>>>(b4, cats, counts, lay.m_max, thr_f, mode, ws.info, todo);
    DET_LAUNCH_OK("large_stats_kernel");
    dim3 grid_e((unsigned)((mp + 255) / 256), (unsigned)n);
    large_keys_kernel<<<grid_e, 256, 0, st>>>(scores, cats, lay.m_max, mp, ws.info, ws.keys_a);
    DET_LAUNCH_OK("large_keys_kernel");
    uint64_t* sorted = sort_rows(ws.keys_a, ws.keys_b, n, mp, st, ws.info);
    uint64_t* other = (sorted == ws.keys_a) ? ws.keys_b : ws.keys_a;
    DET_LAUNCH_OK("sort_rows");
    large_gather_kernel<<<grid_e, 256, 0, st>>>(b4, cats, lay.m_max, mp, ws.info, sorted, ws.sbox, ws.sarea, ws.state,
                                                ws.ctr, ws.seg_small, ws.seg_large, ws.seg_huge, ws.huge_nk);
    DET_LAUNCH_OK("large_gather_kernel");
    const int max_keep = (int)min(max_out, (int64_t)lay.m_max);
    int rc = run_segment_kernels(lay, ws, thr_f, max_keep, st);
    if (rc != DET_OK) return rc;
    large_rekey_kernel<<<grid_e, 256, 0, st>>>(mp, ws.info, sorted, ws.state, other);
    DET_LAUNCH_OK("large_rekey_kernel");
    uint64_t* final_keys = sort_rows(other, sorted, n, mp, st, ws.info);
    DET_LAUNCH_OK("sort_rows(2)");
    dim3 grid_o((unsigned)((min(max_out, lay.m_max) + 255) / 256), (unsigned)n);
    large_emit_kernel<<<grid_o, 256, 0, st>>>(mp, ws.info, final_keys, max_out, keep, keep_counts);
    DET_LAUNCH_OK("large_emit_kernel");
    return DET_OK;
}

}  // namespace det
