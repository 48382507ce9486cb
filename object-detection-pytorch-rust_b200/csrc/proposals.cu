// RPN proposal selection for the whole batch in one call (subsystem 3, reference row a7).
//
// Replaces find_top_rpn_proposals (python/src/models/utils.py:9-109), which sorts every level fully, gathers, and then
// loops over the images in Python with >= 4 host synchronisations each.  Here:
//   per-level radix select of the pre_nms_topk best keys (level | descending logit | anchor index) into a compact row
//   (one CTA per (image, level), the level's keys staged in shared memory) -> sort of that row only (one tile sort per
//   (image, level); tile sort + merge passes when a level keeps more than a tile) -> gather with the finite / clip /
//   min-size filters fused in -> tier cut: per-(image, level) greedy NMS (nms_core.cuh / nms_large.cuh) above a global
//   score cut first, full segments only if that falls short of post_nms_topk -> finish: the kept keys of a level are a
//   sorted run, the output order is the merge of the runs (rank by binary search), boxes + logits written in place
//   (rekey / pad / sort / emit kernels when an image's kept keys do not fit into shared memory).
// No host synchronisation; the "training diverged" condition (models/utils.py:79-84) is reported through a device flag.
#include <algorithm>
#include "nms_large.cuh"

namespace det {

constexpr int kMaxLevels = 16;
constexpr int kRpnWarpSegMax = 32;  // at most 16 segments per image: longer ones are swept by whole CTAs,
constexpr int kRpnCtaSegMax = kHugeSeg;  // (routing segments > 512 to the grid-wide kernel was measured slower:
                                         //  0.69 vs 0.57 ms per 64 images -- its grid barriers cost more than they save)
struct LevelTable {
    int num_levels;
    int64_t off[kMaxLevels + 1];
};

__device__ __forceinline__ int level_of(const LevelTable& t, int64_t i) {
    int l = 0;
#pragma unroll
    for (int k = 1; k < kMaxLevels; ++k)
        if (k < t.num_levels && i >= t.off[k]) l = k;
    return l;
}

// ---- per-level top-k by radix select ---------------------------------------------------------------------------------------
// The reference sorts every level fully and narrows to pre_nms_topk (models/utils.py:56-58).  Here the pre_nms_topk
// best keys (level | descending logit | anchor index -- unique, so "best k" is exact and stable) of every level are
// found with a radix select (4 byte-passes over the 32-bit logit keys; when equal logits straddle the cut the lower
// anchor indices win, ranked in index order) and written, in arrival order, to a compact row [coff[l], coff[l] + take_l) per level.  Only that row -- a few
// tiles instead of all R keys -- is sorted afterwards.  One CTA per (image, level).
// one step of the radix select, by one warp: from the 256-bin histogram of the keys that share *prefix, find the bin that
// holds the *want-th of them, extend the prefix by it and reduce *want to the rank inside the bin
__device__ __forceinline__ void radix_decide(const uint32_t* hist, int lane, int shift, uint32_t* s_prefix, int* s_want,
                                             int* s_done) {
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
    const uint32_t prefix = *s_prefix, w = (uint32_t)*s_want, before = incl - tot;
    __syncwarp();  // every lane has read the state the owner lane is about to replace
    if (before < w && w <= incl) {
        uint32_t run = before;
        int q = 0;
        for (; q < 7 && run + c8[q] < w; ++q) run += c8[q];
        uint32_t np = prefix | ((uint32_t)(lane * 8 + q) << shift);
        if (run + c8[q] == w) {  // the whole bin is wanted: everything that shares the prefix is in
            np |= (shift == 0) ? 0u : ((1u << shift) - 1u);
            *s_done = 1;
        }
        *s_prefix = np;
        *s_want = (int)(w - run);
    }
}

static __global__ void __launch_bounds__(1024)
rpn_select_kernel(const float* __restrict__ logits, int64_t r, int64_t mp, LevelTable lt, LevelTable ct, int64_t len1,
                  LargeImg* info, uint64_t* __restrict__ keys, int stage_cap) {
    // the keys of a level that needs a selection are read from global memory once and staged here (up to stage_cap of
    // them): the radix passes and the final compaction then run out of shared memory
    extern __shared__ __align__(16) uint32_t staged_keys[];
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix;
    __shared__ int s_want, s_slot, s_done, s_warp[32];
    constexpr int T = 1024;
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const float* lg = logits + (int64_t)img * r;
    uint64_t* out = keys + (int64_t)img * mp;
    // grid (images, levels): one CTA per (image, level) -- the levels of an image are independent selections into
    // disjoint ranges of the compact row; blockIdx.y = 0 (the largest level of a pyramid) is dispatched first.  (One CTA
    // per image walking the levels took 0.199 / 0.256 / 0.560 ms per 16 / 64 / 256 images against 0.179 / 0.237 / 0.541.)
    if (blockIdx.y == 0) {
        if (tid == 0) {
            LargeImg li;
            li.cnt = (int32_t)ct.off[ct.num_levels]; li.trick = 0; li.fast = 1; li.span = 0.f; li.nkept = 0; li.bad = 0;
            li.nsurv = 0; li.nonan = 1; li.skip = 0;  // non-finite boxes are dropped by the gather kernel
            for (int q = 0; q < 7; ++q) li.pad_[q] = 0;
            info[img] = li;
        }
        for (int64_t j = ct.off[ct.num_levels] + tid; j < len1; j += T) out[j] = kSentinelKey;
    }
    const int l = blockIdx.y;
    const int64_t i0 = lt.off[l], size = lt.off[l + 1] - i0;
    const int take = (int)(ct.off[l + 1] - ct.off[l]);
    if (take == 0) return;
    // cut: keys with score key < cut are in; in tie mode those == cut only while `tie_want` lasts (index order),
    // otherwise every key <= cut is in
    uint32_t cut = 0xffffffffu;
    bool tie_mode = false;
    int tie_want = 0;
    const bool staged = take < size && size <= (int64_t)stage_cap;
    auto count_top_byte = [&](bool valid, uint32_t key) {
        // (counting lanes that share a bin with one atomic -- match.any -- was measured slower than letting the
        //  shared-memory atomics serialise: 82 vs 58 us per 64 images with one CTA per image)
        if (valid) atomicAdd(&hist[key >> 24], 1u);
    };
    if (staged) {
        // one pass over the level: keys into the staging area + the histogram of the first radix pass, eight
        // loads of a thread in flight together
        const int sz = (int)size;
        const float* lgl = lg + i0;
        for (int b = tid; b < 256; b += T) hist[b] = 0u;
        __syncthreads();
        for (int base = 0; base < sz; base += 8 * T) {
            uint32_t kk[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = base + u * T + tid;
                kk[u] = i < sz ? score_desc_key(lgl[i]) : 0u;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = base + u * T + tid;
                if (i < sz) {
                    staged_keys[i] = kk[u];
                    atomicAdd(&hist[kk[u] >> 24], 1u);
                }
            }
        }
        if (tid == 0) {
            s_prefix = 0u;
            s_want = take;
            s_done = 0;
            s_slot = 0;
        }
        // the remaining passes and the compaction read the copy four keys at a time
        const uint4* s4 = reinterpret_cast<const uint4*>(staged_keys);
        const int n4 = sz >> 2;
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (shift != 24) {
                for (int b = tid; b < 256; b += T) hist[b] = 0u;
                __syncthreads();
                if (s_done) break;
                const uint32_t prefix = s_prefix, himask = 0xffffffffu << (shift + 8);
                for (int j = tid; j < n4; j += T) {
                    const uint4 v = s4[j];
                    if ((v.x & himask) == prefix) atomicAdd(&hist[(v.x >> shift) & 255u], 1u);
                    if ((v.y & himask) == prefix) atomicAdd(&hist[(v.y >> shift) & 255u], 1u);
                    if ((v.z & himask) == prefix) atomicAdd(&hist[(v.z >> shift) & 255u], 1u);
                    if ((v.w & himask) == prefix) atomicAdd(&hist[(v.w >> shift) & 255u], 1u);
                }
                if (tid < (sz & 3)) {
                    const uint32_t key = staged_keys[(n4 << 2) + tid];
                    if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
                }
            }
            __syncthreads();
            if (wid == 0) radix_decide(hist, lane, shift, &s_prefix, &s_want, &s_done);
            __syncthreads();
        }
        __syncthreads();
        cut = s_prefix;
        tie_mode = s_done == 0;
        tie_want = s_want;
        if (!tie_mode) {
            const uint64_t lvl = (uint64_t)l << KLL::kSegShift;
            uint64_t* o = out + ct.off[l];
            const uint32_t a0 = (uint32_t)i0;
            const unsigned lt_mask = (1u << lane) - 1u;
            for (int j0 = 0; j0 < n4; j0 += T) {
                const int j = j0 + tid;
                uint4 v = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
                if (j < n4) v = s4[j];
                const bool i0n = j < n4 && v.x <= cut, i1n = j < n4 && v.y <= cut, i2n = j < n4 && v.z <= cut,
                           i3n = j < n4 && v.w <= cut;
                const unsigned b0 = __ballot_sync(0xffffffffu, i0n), b1 = __ballot_sync(0xffffffffu, i1n),
                               b2 = __ballot_sync(0xffffffffu, i2n), b3 = __ballot_sync(0xffffffffu, i3n);
                const int c0 = __popc(b0), c1 = __popc(b1), c2 = __popc(b2), c3 = __popc(b3);
                if (c0 + c1 + c2 + c3 == 0) continue;  // warp-uniform
                int pos = 0;
                if (lane == 0) pos = atomicAdd(&s_slot, c0 + c1 + c2 + c3);
                pos = __shfl_sync(0xffffffffu, pos, 0);
                const uint32_t a = a0 + (uint32_t)(j << 2);
                int q = pos + __popc(b0 & lt_mask);
                if (i0n && q < take) o[q] = lvl | ((uint64_t)v.x << KLL::kScoreShift) | (uint64_t)a;
                q = pos + c0 + __popc(b1 & lt_mask);
                if (i1n && q < take) o[q] = lvl | ((uint64_t)v.y << KLL::kScoreShift) | (uint64_t)(a + 1u);
                q = pos + c0 + c1 + __popc(b2 & lt_mask);
                if (i2n && q < take) o[q] = lvl | ((uint64_t)v.z << KLL::kScoreShift) | (uint64_t)(a + 2u);
                q = pos + c0 + c1 + c2 + __popc(b3 & lt_mask);
                if (i3n && q < take) o[q] = lvl | ((uint64_t)v.w << KLL::kScoreShift) | (uint64_t)(a + 3u);
            }
            if (tid < (sz & 3)) {
                const int i = (n4 << 2) + tid;
                const uint32_t key = staged_keys[i];
                if (key <= cut) {
                    const int q = atomicAdd(&s_slot, 1);
                    if (q < take) o[q] = lvl | ((uint64_t)key << KLL::kScoreShift) | (uint64_t)(a0 + (uint32_t)i);
                }
            }
            return;
        }
        // ties at the cut: the index-ordered walk below (cut / tie_mode / tie_want are set)
    }
    auto key_at = [&](int64_t i) -> uint32_t { return staged ? staged_keys[i] : score_desc_key(lg[i0 + i]); };
    if (take < size && !staged) {
        // radix select of the take-th best 32-bit descending-logit key, one byte per pass
        if (tid == 0) {
            s_prefix = 0u;
            s_want = take;
            s_done = 0;
        }
        for (int shift = 24; shift >= 0; shift -= 8) {
            {
                for (int b = tid; b < 256; b += T) hist[b] = 0u;
                __syncthreads();
                if (s_done) break;
                const uint32_t prefix = s_prefix, himask = (shift == 24) ? 0u : (0xffffffffu << (shift + 8));
                if (shift == 24) {
                    for (int64_t base = 0; base < size; base += T)
                        count_top_byte(base + tid < size, base + tid < size ? key_at(base + tid) : 0u);
                } else {
                    for (int64_t i = tid; i < size; i += T) {
                        const uint32_t key = key_at(i);
                        if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
                    }
                }
                __syncthreads();
            }
            if (wid == 0) radix_decide(hist, lane, shift, &s_prefix, &s_want, &s_done);
            __syncthreads();
        }
        __syncthreads();
        cut = s_prefix;
        // not done after the last byte: several anchors share the cut logit and only s_want of them fit -- the
        // reference's stable sort keeps the lower indices
        tie_mode = s_done == 0;
        tie_want = s_want;
    }
    if (tid == 0) s_slot = 0;
    __syncthreads();
    const uint64_t lvl = (uint64_t)l << KLL::kSegShift;
    int tie_seen = 0;  // equal-logit anchors already passed, in index order (block-uniform)
    for (int64_t base = 0; base < size; base += T) {
        const int64_t i = base + tid;
        uint32_t k32 = 0xffffffffu;
        bool in = false, eq = false;
        if (i < size) {
            k32 = key_at(i);
            in = tie_mode ? (k32 < cut) : (k32 <= cut);
            eq = tie_mode && k32 == cut;
        }
        if (tie_mode) {  // block-uniform branch: rank the equal keys of this step in index order
            const unsigned be = __ballot_sync(0xffffffffu, eq);
            if (lane == 0) s_warp[wid] = __popc(be);
            __syncthreads();
            int before = tie_seen, total = 0;
            for (int w = 0; w < T / 32; ++w) {
                const int v = s_warp[w];
                before += (w < wid) ? v : 0;
                total += v;
            }
            if (eq && before + __popc(be & ((1u << lane) - 1u)) < tie_want) in = true;
            tie_seen += total;
            __syncthreads();
        }
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        int pos = 0;
        if (lane == 0 && bal) pos = atomicAdd(&s_slot, __popc(bal));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(bal & ((1u << lane) - 1u));
        if (in && pos < take)
            out[ct.off[l] + pos] = lvl | ((uint64_t)k32 << KLL::kScoreShift) | (uint64_t)(uint32_t)(i0 + i);
    }
}

// ---- per-level sort of the compact row -------------------------------------------------------------------------------------
// The selected keys of level l lie in [coff[l], coff[l] + take_l) and carry the level in their top bits, so sorting every
// level's range by itself IS the sort of the row.  With take_l <= kTile that is one shared-memory tile sort per
// (image, level) and no merge passes (sort_rows: tile sort + two merge passes over 8192 keys per image at 2000 per level).
constexpr int kLevelSortThreads = 512;  // 4 keys per thread: 16 warps hide the shuffle latency of the network better than 8

static __global__ void __launch_bounds__(kLevelSortThreads, 2)
rpn_sort_levels_kernel(uint64_t* __restrict__ keys, int64_t mp, LevelTable ct) {
    __shared__ uint64_t s[kTile];
    const int l = blockIdx.x, img = blockIdx.y;
    const int take = (int)(ct.off[l + 1] - ct.off[l]);
    if (take <= 1) return;
    uint64_t* g = keys + (int64_t)img * mp + ct.off[l];
    const int n2 = next_pow2(take);
    for (int i = threadIdx.x; i < max(n2, kLevelSortThreads); i += kLevelSortThreads) s[i] = i < take ? g[i] : kSentinelKey;
    __syncthreads();
    cta_bitonic_sort<kLevelSortThreads>(s, n2);
    for (int i = threadIdx.x; i < take; i += kLevelSortThreads) g[i] = s[i];
}

__device__ __forceinline__ float4 clip_box(float4 b, float w, float h) {
    // Boxes.clip, structures/boxes.py:62-65 (inputs are finite here)
    b.x = fminf(fmaxf(b.x, 0.f), w); b.z = fminf(fmaxf(b.z, 0.f), w);
    b.y = fminf(fmaxf(b.y, 0.f), h); b.w = fminf(fmaxf(b.w, 0.f), h);
    return b;
}

static __global__ void __launch_bounds__(256)
rpn_gather_kernel(const float4* __restrict__ boxes, const float* __restrict__ logits, int64_t r, int64_t rc, int64_t mp,
                  LevelTable lt, int64_t pre_nms_topk, const int32_t* __restrict__ image_sizes, float min_size,
                  LargeImg* info, const uint64_t* __restrict__ keys, float4* __restrict__ sbox,
                  float* __restrict__ sarea, uint8_t* __restrict__ state, int32_t* __restrict__ nonfinite_flag) {
    const int img = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    bool survivor = false;
    if (p < rc) {  // lt is the COMPACT level table here: level l occupies [lt.off[l], lt.off[l+1]) of the sorted row
        const uint64_t key = keys[(int64_t)img * mp + p];
        const int64_t i = KLL::idx(key);
        const int l = (int)KLL::seg(key);
        const int64_t rank = p - lt.off[l];  // a level's keys occupy the same slot range after the sort
        const int64_t take = min(lt.off[l + 1] - lt.off[l], pre_nms_topk);
        uint8_t st = 1;
        if (rank < take) {
            float4 b = boxes[(int64_t)img * r + i];
            const float sc = logits[(int64_t)img * r + i];
            const bool fin = isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w) && isfinite(sc);
            if (!fin) {
                if (nonfinite_flag) *nonfinite_flag = 1;
            } else {
                b = clip_box(b, (float)image_sizes[2 * img + 1], (float)image_sizes[2 * img]);
                if ((b.z - b.x) > min_size && (b.w - b.y) > min_size) {  // Boxes.nonempty, boxes.py:67-80
                    st = 0;
                    survivor = true;
                    sbox[(int64_t)img * mp + p] = b;
                    sarea[(int64_t)img * mp + p] = box_area(b);
                }
            }
        }
        state[(int64_t)img * mp + p] = st;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, survivor);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&info[img].nsurv, __popc(bal));
}

// images with <= 1000 surviving boxes take torchvision's coordinate-offset branch: box + level * (max + 1) in fp32
static __global__ void __launch_bounds__(256)
rpn_offset_kernel(int64_t r, int64_t mp, const LargeImg* __restrict__ info, const uint64_t* __restrict__ keys,
                  float4* __restrict__ sbox, float* __restrict__ sarea, const uint8_t* __restrict__ state) {
    __shared__ float s_max[8];
    const int img = blockIdx.x, tid = threadIdx.x;
    const int ns = info[img].nsurv;
    if (ns == 0 || ns > 1000) return;
    float mx = -INFINITY;
    for (int64_t p = tid; p < r; p += 256)
        if (state[(int64_t)img * mp + p] == 0) {
            const float4 b = sbox[(int64_t)img * mp + p];
            mx = fmaxf(mx, fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w)));
        }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) s_max[tid >> 5] = mx;
    __syncthreads();
    mx = s_max[0];
    for (int w = 1; w < 8; ++w) mx = fmaxf(mx, s_max[w]);
    const float span = mx + 1.0f;
    for (int64_t p = tid; p < r; p += 256)
        if (state[(int64_t)img * mp + p] == 0) {
            const float off = (float)KLL::seg(keys[(int64_t)img * mp + p]) * span;
            float4 b = sbox[(int64_t)img * mp + p];
            b.x += off; b.y += off; b.z += off; b.w += off;
            sbox[(int64_t)img * mp + p] = b;
            sarea[(int64_t)img * mp + p] = box_area(b);
        }
}

// ---- tier cut --------------------------------------------------------------------------------------------------------------
// Only post_nms_topk proposals are wanted and a box can only be suppressed by a better-scored box of its level, so the
// per-level sweeps first run on the candidates above a global score cut -- the (1.25 * post_nms_topk + 32)-th best
// logit among the image's valid candidates, found exactly with a 4-pass radix select; ties with the cut are included.
// Inside a level the candidates are sorted by logit, so "above the cut" is a PREFIX of the level's segment.  If the
// prefixes yield post_nms_topk survivors, those are exactly the first post_nms_topk of the full result; otherwise
// rpn_tier_check_kernel resets the image and queues its full segments for a second run of the segment kernels.
// pass 0: decide + push prefixes (or full segments when a tier is not worth it);  pass 1: check + push full segments.
static __global__ void __launch_bounds__(1024)
rpn_tier_kernel(int pass, int64_t r, int64_t mp, LevelTable lt, int64_t pre_nms_topk, int64_t post_nms_topk,
                LargeImg* info, const uint64_t* __restrict__ keys, uint8_t* __restrict__ state, int32_t* ctr,
                int4* seg_small, int4* seg_large, int4* seg_huge, int2* huge_nk) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix;
    __shared__ int s_want, s_kept;
    constexpr int T = 1024;
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint64_t* k = keys + (int64_t)img * mp;
    uint8_t* stt = state + (int64_t)img * mp;
    const int want = (int)min(post_nms_topk + (post_nms_topk >> 2) + 32, (int64_t)1 << 30);
    if (pass == 1) {
        if (!info[img].pad_[0]) return;  // no tier was cut for this image: its full segments have been swept
        if (tid == 0) s_kept = 0;
        __syncthreads();
        int kept = 0;
        for (int l = 0; l < lt.num_levels; ++l) {
            const int64_t s0 = lt.off[l], take = min(lt.off[l + 1] - lt.off[l], pre_nms_topk);
            for (int64_t p = s0 + tid; p < s0 + take; p += T) kept += stt[p] == 2 ? 1 : 0;
        }
        kept = warp_sum(kept);
        if (lane == 0 && kept) atomicAdd(&s_kept, kept);
        __syncthreads();
        if (s_kept >= post_nms_topk) return;
        for (int l = 0; l < lt.num_levels; ++l) {  // fell short: forget the prefix sweep, queue the full segments
            const int64_t s0 = lt.off[l], take = min(lt.off[l + 1] - lt.off[l], pre_nms_topk);
            for (int64_t p = s0 + tid; p < s0 + take; p += T)
                if (stt[p] == 2) stt[p] = 0;
            if (tid == 0 && take > 0) push_segment(img, (int)s0, (int)(s0 + take), ctr, seg_small, seg_large, seg_huge, huge_nk, kRpnWarpSegMax, kRpnCtaSegMax);
        }
        return;
    }
    const bool tier = info[img].nsurv >= want + (want >> 1);
    if (tid == 0) info[img].pad_[0] = tier ? 1 : 0;
    if (!tier) {
        if (tid < lt.num_levels) {
            const int64_t s0 = lt.off[tid], take = min(lt.off[tid + 1] - lt.off[tid], pre_nms_topk);
            if (take > 0) push_segment(img, (int)s0, (int)(s0 + take), ctr, seg_small, seg_large, seg_huge, huge_nk, kRpnWarpSegMax, kRpnCtaSegMax);
        }
        return;
    }
    if (tid == 0) {
        s_prefix = 0u;
        s_want = want;
    }
    // the valid candidates' score keys are read ONCE (up to 8 per thread, all loads in flight together): the four radix
    // passes were four dependent global round trips per trip of the loop, 20 us of pure latency per launch
    constexpr int kHeld = 8;
    const bool held = r <= (int64_t)kHeld * T;  // the compact row [0, r) is level after level without gaps
    uint32_t myk[kHeld];
    unsigned myv = 0u;
    if (held) {
#pragma unroll
        for (int u = 0; u < kHeld; ++u) {
            const int64_t p = (int64_t)u * T + tid;
            const bool in = p < r;
            const uint8_t st8 = in ? stt[p] : (uint8_t)1;
            const uint64_t k64 = in ? k[p] : 0ull;
            myk[u] = (uint32_t)(k64 >> KLL::kScoreShift);
            myv |= (st8 == 0) ? (1u << u) : 0u;
        }
    }
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int b = tid; b < 256; b += T) hist[b] = 0u;
        __syncthreads();
        const uint32_t prefix = s_prefix, himask = (shift == 24) ? 0u : (0xffffffffu << (shift + 8));
        if (held) {
#pragma unroll
            for (int u = 0; u < kHeld; ++u)
                if (((myv >> u) & 1u) && (myk[u] & himask) == prefix) atomicAdd(&hist[(myk[u] >> shift) & 255u], 1u);
        } else {
            for (int l = 0; l < lt.num_levels; ++l) {
                const int64_t s0 = lt.off[l], take = min(lt.off[l + 1] - lt.off[l], pre_nms_topk);
                for (int64_t p = s0 + tid; p < s0 + take; p += T) {
                    if (stt[p] != 0) continue;
                    const uint32_t key = (uint32_t)(k[p] >> KLL::kScoreShift);
                    if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
                }
            }
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
    const uint32_t cut = s_prefix;  // exact descending-logit key of the want-th best valid candidate
    if (tid < lt.num_levels) {
        const int64_t s0 = lt.off[tid], take = min(lt.off[tid + 1] - lt.off[tid], pre_nms_topk);
        int64_t lo = s0, hi = s0 + take;  // first position of the level whose key is worse than the cut
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((uint32_t)(k[mid] >> KLL::kScoreShift) > cut) hi = mid; else lo = mid + 1;
        }
        if (lo > s0) push_segment(img, (int)s0, (int)lo, ctr, seg_small, seg_large, seg_huge, huge_nk, kRpnWarpSegMax, kRpnCtaSegMax);
    }
}

// kept candidates -> output keys (descending logit | index), COMPACTED to the front of the row: at most
// min(sum of the levels' top-k, levels * post_nms_topk) boxes survive, so the output sort only touches a few tiles
static __global__ void __launch_bounds__(256)
rpn_rekey_compact_kernel(int64_t r, int64_t mp, LargeImg* info, const uint64_t* __restrict__ keys,
                         const uint8_t* __restrict__ state, uint64_t* __restrict__ keys_out) {
    const int img = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const bool kept = (p < r) && state[(int64_t)img * mp + p] == 2;
    const unsigned bal = __ballot_sync(0xffffffffu, kept);
    if (!bal) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(&info[img].nkept, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (kept) keys_out[(int64_t)img * mp + base + __popc(bal & ((1u << lane) - 1u))] = KLL::strip_seg(keys[(int64_t)img * mp + p]);
}

static __global__ void __launch_bounds__(256)
rpn_pad_kernel(int64_t mp, int64_t len, const LargeImg* __restrict__ info, uint64_t* __restrict__ keys_out) {
    const int img = blockIdx.y;
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j < len && j >= info[img].nkept) keys_out[(int64_t)img * mp + j] = kSentinelKey;
}

static __global__ void __launch_bounds__(256)
rpn_emit_kernel(const float4* __restrict__ boxes, const float* __restrict__ logits, int64_t r, int64_t mp,
                const LargeImg* __restrict__ info, const uint64_t* __restrict__ keys,
                const int32_t* __restrict__ image_sizes, int64_t post_nms_topk, float4* __restrict__ out_boxes,
                float* __restrict__ out_logits, int32_t* __restrict__ out_counts) {
    const int img = blockIdx.y;
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t nout = min((int64_t)info[img].nkept, post_nms_topk);
    if (j < nout) {
        const int64_t i = KLL::idx(keys[(int64_t)img * mp + j]);
        out_boxes[(int64_t)img * post_nms_topk + j] =
            clip_box(boxes[(int64_t)img * r + i], (float)image_sizes[2 * img + 1], (float)image_sizes[2 * img]);
        out_logits[(int64_t)img * post_nms_topk + j] = logits[(int64_t)img * r + i];
    }
    if (j == 0) out_counts[img] = (int32_t)nout;
}

// ---- kept candidates -> proposals, one CTA per image ------------------------------------------------------------------------
// Inside a level the candidates are sorted by (descending logit, index), so the kept ones of a level form a sorted run
// and the output order is the MERGE of the levels' runs: an order-preserving compaction of the kept keys into shared
// memory (one block scan over the compact row), then every kept key finds its output slot as its position in its own
// run plus, by binary search, the number of smaller keys in every other run -- and writes its clipped box and logit
// there if the slot is below post_nms_topk.  Replaces rekey + pad + tile sort + merge pass + emit (5 launches).
static __global__ void __launch_bounds__(1024)
rpn_finish_kernel(const float4* __restrict__ boxes, const float* __restrict__ logits, int64_t r, int rc, int64_t mp,
                  LevelTable ct, int cap, const uint64_t* __restrict__ keys, const uint8_t* __restrict__ state,
                  const int32_t* __restrict__ image_sizes, int64_t post_nms_topk, float4* __restrict__ out_boxes,
                  float* __restrict__ out_logits, int32_t* __restrict__ out_counts) {
    extern __shared__ uint64_t fk[];  // kept keys without the level field, run after run
    __shared__ int s_warp[32], s_lvl[kMaxLevels + 1], s_total;
    constexpr int T = 1024;
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint64_t* k = keys + (int64_t)img * mp;
    const uint8_t* stt = state + (int64_t)img * mp;
    int run = 0;  // kept so far (block-uniform)
    for (int base0 = 0; base0 < rc; base0 += 4 * T) {
        uint8_t st4[4];
        uint64_t k4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {  // the loads of four trips in flight together
            const int p = base0 + u * T + tid;
            st4[u] = p < rc ? stt[p] : (uint8_t)0;
            k4[u] = p < rc ? k[p] : 0ull;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (base0 + u * T >= rc) break;
            const int p = base0 + u * T + tid;
            const bool kept = p < rc && st4[u] == 2;
            const unsigned bal = __ballot_sync(0xffffffffu, kept);
            if (lane == 0) s_warp[wid] = __popc(bal);
            __syncthreads();
            if (wid == 0) {  // exclusive scan of the 32 warp counts
                const int v = s_warp[lane];
                int incl = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int up = __shfl_up_sync(0xffffffffu, incl, o);
                    incl += (lane >= o) ? up : 0;
                }
                s_warp[lane] = incl - v;
                if (lane == 31) s_total = incl;
            }
            __syncthreads();
            const int before = run + s_warp[wid], total = s_total;
            const int slot = before + __popc(bal & ((1u << lane) - 1u));
            if (kept && slot < cap) fk[slot] = KLL::strip_seg(k4[u]);
            if (p < rc)
                for (int l = 0; l < ct.num_levels; ++l)
                    if ((int64_t)p == ct.off[l]) s_lvl[l] = slot;  // first slot of level l's run
            run += total;  // (no barrier: a warp's count is only rewritten by the warp itself, s_total behind the next barrier)
        }
    }
    if (tid == 0)
        for (int l = 0; l <= ct.num_levels; ++l)
            if (ct.off[l] >= (int64_t)rc) s_lvl[l] = run;
    __syncthreads();
    const int nk = min(run, cap);
    const float iw = (float)image_sizes[2 * img + 1], ih = (float)image_sizes[2 * img];
    for (int j = tid; j < nk; j += T) {
        const uint64_t key = fk[j];
        int rank = 0;
        for (int l0 = 0; l0 < ct.num_levels; l0 += 4) {  // four runs searched side by side (independent chains)
            int lo[4], hi[4], a[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool real = l0 + u < ct.num_levels;
                a[u] = real ? s_lvl[l0 + u] : 0;
                const int b = real ? s_lvl[l0 + u + 1] : 0;
                const bool own = j >= a[u] && j < b;  // its own run: the position is the count
                lo[u] = own ? j : a[u];
                hi[u] = own ? j : b;
            }
            for (;;) {
                bool any = false;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (lo[u] < hi[u]) {  // keys are unique: number of keys of the run below `key`
                        const int mid = (lo[u] + hi[u]) >> 1;
                        if (fk[mid] < key) lo[u] = mid + 1; else hi[u] = mid;
                        any = true;
                    }
                if (!any) break;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) rank += lo[u] - a[u];
        }
        if (rank < post_nms_topk) {
            const int64_t i = KLL::idx(key);
            out_boxes[(int64_t)img * post_nms_topk + rank] = clip_box(boxes[(int64_t)img * r + i], iw, ih);
            out_logits[(int64_t)img * post_nms_topk + rank] = logits[(int64_t)img * r + i];
        }
    }
    if (tid == 0) out_counts[img] = (int32_t)min((int64_t)nk, post_nms_topk);
}

}  // namespace det

using namespace det;

extern "C" {

int64_t det_rpn_proposals_workspace_bytes(int n, int64_t r) {
    if (n <= 0 || r <= 0) return 256;
    return LargeLayout(n, r).total;
}

int det_rpn_proposals(const float* boxes, const float* logits, int n, int64_t r, const int64_t* level_sizes_host,
                      int num_levels, const int32_t* image_sizes, double nms_thresh, int64_t pre_nms_topk,
                      int64_t post_nms_topk, float min_box_size, float* out_boxes, float* out_logits,
                      int32_t* out_counts, int32_t* nonfinite_flag, void* workspace, int64_t workspace_bytes,
                      void* stream) {
    DET_CHECK_ARG(n >= 0 && r >= 0 && pre_nms_topk >= 0 && post_nms_topk >= 0, "negative size");
    DET_CHECK_ARG(num_levels >= 1 && num_levels <= kMaxLevels && level_sizes_host, "1..16 levels");
    if (n == 0) return DET_OK;
    DET_CHECK_ARG(out_counts, "null output");
    cudaStream_t st = as_stream(stream);
    if (r == 0 || post_nms_topk == 0 || pre_nms_topk == 0) {
        cudaError_t e = cudaMemsetAsync(out_counts, 0, sizeof(int32_t) * (size_t)n, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
        return DET_OK;
    }
    DET_CHECK_ARG(boxes && logits && image_sizes && out_boxes && out_logits, "null pointer");
    DET_CHECK_ARG(n <= 65535, "n > 65535");
    if (r > (1 << kLargeIdxBits) - 1) {
        set_error("r %lld exceeds the limit 131071 anchors per image", (long long)r);
        return DET_ERR_UNSUPPORTED;
    }
    LevelTable lt;
    lt.num_levels = num_levels;
    int64_t acc = 0;
    for (int l = 0; l <= kMaxLevels; ++l) {
        lt.off[l] = acc;
        if (l < num_levels) {
            DET_CHECK_ARG(level_sizes_host[l] >= 0, "negative level size");
            acc += level_sizes_host[l];
        }
    }
    DET_CHECK_ARG(acc == r, "level sizes must sum to r");
    if (!aligned16(boxes) || !aligned16(out_boxes) || !aligned16(workspace)) {
        set_error("boxes/out_boxes/workspace must be 16-byte aligned");
        return DET_ERR_ALIGN;
    }
    LargeLayout lay(n, r);
    if (!workspace || workspace_bytes < lay.total) {
        set_error("workspace too small: need %lld bytes", (long long)lay.total);
        return DET_ERR_WORKSPACE;
    }
    LargeWs ws(lay, workspace);
    const int64_t mp = lay.mp;
    const float thr_f = float_threshold_below(nms_thresh);
    auto b4 = reinterpret_cast<const float4*>(boxes);
    cudaError_t e = cudaMemsetAsync(ws.ctr, 0, 64, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    // compact level table: level l keeps its best take_l = min(size_l, pre_nms_topk) keys at [coff[l], coff[l+1])
    LevelTable ct;
    ct.num_levels = num_levels;
    int64_t rc = 0;
    for (int l = 0; l <= kMaxLevels; ++l) {
        ct.off[l] = rc;
        if (l < num_levels) rc += std::min(level_sizes_host[l], pre_nms_topk);
    }
    const int64_t len1 = (rc + kTile - 1) / kTile * kTile;  // <= mp
    // staging area of the select kernel: the largest level that needs a selection, if it fits (200 KB at most)
    int64_t stage = 0;
    for (int l = 0; l < num_levels; ++l)
        if (pre_nms_topk < level_sizes_host[l] && level_sizes_host[l] <= 50 * 1024) stage = std::max(stage, level_sizes_host[l]);
    if (stage * 4 > 40 * 1024) {  // (the 48 KB default covers static + dynamic shared memory: leave room for the 2 KB of statics)
        cudaError_t ea = cudaFuncSetAttribute(rpn_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(stage * 4));
        if (ea != cudaSuccess) return cuda_fail(ea, "cudaFuncSetAttribute(rpn_select_kernel)");
    }
    // A cluster of four CTAs per (image, level) exchanging radix histograms through distributed shared memory was built and
    // measured: 45.8 us instead of 54.8 us for 64 images but 163 us instead of 140 us for 256 (ten cluster barriers per CTA); a
    // second form with two visits per key (keys below the cut's top byte written at once, the rest listed) executed MORE
    // instructions than these seven tight visits (336 k vs 292 k warp-instructions per image) -- both rejected.
    rpn_select_kernel<<<dim3((unsigned)n, (unsigned)num_levels), 1024, (size_t)(stage * 4), st>>>(logits, r, mp, lt, ct, len1, ws.info, ws.keys_a, (int)stage);
    DET_LAUNCH_OK("rpn_select_kernel");
    uint64_t* sorted;
    if (std::min(*std::max_element(level_sizes_host, level_sizes_host + num_levels), pre_nms_topk) <= kTile) {
        rpn_sort_levels_kernel<<<dim3((unsigned)num_levels, (unsigned)n), kLevelSortThreads, 0, st>>>(ws.keys_a, mp, ct);
        sorted = ws.keys_a;
    } else {
        sorted = sort_rows(ws.keys_a, ws.keys_b, n, mp, st, nullptr, len1);
    }
    uint64_t* other = (sorted == ws.keys_a) ? ws.keys_b : ws.keys_a;
    DET_LAUNCH_OK("sort_rows");
    dim3 grid_e((unsigned)((len1 + 255) / 256), (unsigned)n);
    rpn_gather_kernel<<<grid_e, 256, 0, st>>>(b4, logits, r, rc, mp, ct, pre_nms_topk, image_sizes, min_box_size, ws.info,
                                              sorted, ws.sbox, ws.sarea, ws.state, nonfinite_flag);
    DET_LAUNCH_OK("rpn_gather_kernel");
    rpn_offset_kernel<<<n, 256, 0, st>>>(rc, mp, ws.info, sorted, ws.sbox, ws.sarea, ws.state);
    DET_LAUNCH_OK("rpn_offset_kernel");
    DET_CHECK_ARG(num_levels <= 32, "levels");
    rpn_tier_kernel<<<n, 1024, 0, st>>>(0, rc, mp, ct, pre_nms_topk, post_nms_topk, ws.info, sorted, ws.state, ws.ctr,
                                        ws.seg_small, ws.seg_large, ws.seg_huge, ws.huge_nk);
    DET_LAUNCH_OK("rpn_tier_kernel");
    int status = run_segment_kernels(lay, ws, thr_f, (int)min(post_nms_topk, r), st, true);
    if (status != DET_OK) return status;
    // images whose tier fell short of post_nms_topk survivors are swept again in full (usually none: empty lists)
    e = cudaMemsetAsync(ws.ctr, 0, 64, st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    rpn_tier_kernel<<<n, 1024, 0, st>>>(1, rc, mp, ct, pre_nms_topk, post_nms_topk, ws.info, sorted, ws.state, ws.ctr,
                                        ws.seg_small, ws.seg_large, ws.seg_huge, ws.huge_nk);
    DET_LAUNCH_OK("rpn_tier_kernel(check)");
    status = run_segment_kernels(lay, ws, thr_f, (int)min(post_nms_topk, r), st, true);
    if (status != DET_OK) return status;
    int64_t kept_bound = 0;
    for (int l = 0; l < num_levels; ++l) kept_bound += std::min({level_sizes_host[l], pre_nms_topk, post_nms_topk});
    if (kept_bound * 8 <= 200 * 1024) {  // the kept keys of an image fit into shared memory
        const size_t smem = (size_t)kept_bound * 8;
        if (smem > 40 * 1024) {  // (static + dynamic share the 48 KB default)
            cudaError_t ea = cudaFuncSetAttribute(rpn_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (ea != cudaSuccess) return cuda_fail(ea, "cudaFuncSetAttribute(rpn_finish_kernel)");
        }
        rpn_finish_kernel<<<n, 1024, smem, st>>>(b4, logits, r, (int)rc, mp, ct, (int)kept_bound, sorted, ws.state, image_sizes,
                                                 post_nms_topk, reinterpret_cast<float4*>(out_boxes), out_logits, out_counts);
        DET_LAUNCH_OK("rpn_finish_kernel");
        return DET_OK;
    }
    const int64_t len2 = std::min(mp, (kept_bound + kTile - 1) / kTile * kTile);
    rpn_rekey_compact_kernel<<<grid_e, 256, 0, st>>>(rc, mp, ws.info, sorted, ws.state, other);
    DET_LAUNCH_OK("rpn_rekey_compact_kernel");
    dim3 grid_p((unsigned)((len2 + 255) / 256), (unsigned)n);
    rpn_pad_kernel<<<grid_p, 256, 0, st>>>(mp, len2, ws.info, other);
    DET_LAUNCH_OK("rpn_pad_kernel");
    uint64_t* final_keys = sort_rows(other, sorted, n, mp, st, nullptr, len2);
    DET_LAUNCH_OK("sort_rows(2)");
    dim3 grid_o((unsigned)((min(post_nms_topk, r) + 255) / 256), (unsigned)n);
    rpn_emit_kernel<<<grid_o, 256, 0, st>>>(b4, logits, r, mp, ws.info, final_keys, image_sizes, post_nms_topk,
                                            reinterpret_cast<float4*>(out_boxes), out_logits, out_counts);
    DET_LAUNCH_OK("rpn_emit_kernel");
    return DET_OK;
}

#ifdef DET_DEBUG_PHASES
__attribute__((visibility("default"))) int det_debug_read_phase_blocks_proposals(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, det::g_phase_block, sizeof(long long) * 64 * 16) == cudaSuccess ? 0 : -4;
}
__attribute__((visibility("default"))) int det_debug_read_acc_proposals(long long* out_host, int reset) {
    if (cudaMemcpyFromSymbol(out_host, det::g_phase_acc, sizeof(long long) * 16) != cudaSuccess) return -4;
    if (reset) {
        long long z[16] = {0};
        if (cudaMemcpyToSymbol(det::g_phase_acc, z, sizeof(z)) != cudaSuccess) return -4;
    }
    return 0;
}
#endif

}  // extern "C"
