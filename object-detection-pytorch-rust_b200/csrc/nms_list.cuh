// NMS over per-image candidate LISTS (box, score, class, id) of at most CAP entries: one CTA per image, built on
// small_nms_body.  Two users:
//   * det_dense_detect (dense_decode.cu): the lists are the positions of a dense head that passed the score threshold;
//   * det_nms_batched, large path with max_out << boxes (nms_large.cuh): the lists are the best-scored boxes of each
//     image, chosen by large_topk_select_kernel ("external tier": statistics of the full image come with the list, and
//     an image whose list does not yield max_out survivors is handed on to the full path through todo[]).
#pragma once
#include "nms_core.cuh"
#include "nms_small.cuh"

namespace det {

constexpr int kCountStride = 32;  // one 128-byte line per image counter: same-line atomics serialise in L2

// T = 256 threads (several CTAs per SM) for large batches; 512 when there are no more images than SMs, where the
// latency of the single CTA that owns an image is all that counts.
template <int CAP, int T>
struct DetectSmem {
    SmallSmem<CAP, T> nms;
    uint16_t perm[CAP];  // i-th candidate handed to the NMS -> slot in the image's list
    uint32_t hist[256];
    FullStats full;
    uint32_t sel_prefix;
    int sel_want, sub_count;
};

struct ListCandidates {
    const float4* boxes;
    const float* scores;
    const int32_t* cls;
    const uint16_t* perm;  // null: identity
    __device__ __forceinline__ int slot(int i) const { return perm ? (int)perm[i] : i; }
    __device__ __forceinline__ float4 box(int i) const { return boxes[slot(i)]; }
    __device__ __forceinline__ float score(int i) const { return scores[slot(i)]; }
    __device__ __forceinline__ int64_t cat(int i) const { return (int64_t)cls[slot(i)]; }
};

// ---- fast form for det_dense_detect: no tier, no bitonic sort, no chain over the boxes -----------------------------------
// dense_detect_nms_kernel's general body is a chain of CTA-wide steps (tier select, two bitonic sorts, chunked sweeps):
// 38 k cycles per image whatever the other SMs do, which is what holds the dense head at small batches below its stream
// time.  For a list of finite boxes with valid categories the same result comes out of far fewer dependent steps; the
// candidates stay in LIST order in shared memory and only learn their rank:
//   1  one pass over the list: keys (descending score | row id: the oracle's order including ties), boxes, categories,
//      coordinate statistics, category bucket sizes
//   2  counting sort of the keys on a 256-bin histogram of their upper bits, rank inside a bin by direct comparison
//   3  offset-trick shift in place, candidates grouped by category bucket (category mod 256)
//   4  every candidate collects its suppressors: better-ranked boxes of its category with nms_suppresses true (up to
//      kFastEdges are stored); with the offset trick and coordinates below -1 also the pairs (box reaching below -1 in x
//      and y, box of a lower category) -- the only pairs of different categories whose shifted boxes can intersect
//      (nms_small.cuh, phase 0) -- where a hit only flags the worse-ranked box
//   5  decision rounds (see large_bin_segments_kernel): dead if a suppressor is kept, kept once all suppressors are dead
//   6  the first max_det kept candidates, in rank order
// Anything else -- a non-finite coordinate, a category outside the valid range, a negative threshold, an offset-trick
// image whose categories cannot be separated, a long suppressor chain, a crowded category -- returns kFastNo and the
// general body runs on the untouched list.
constexpr int kFastNo = -2;
constexpr int kFastEdges = 4;
constexpr int kFastRounds = 40;
constexpr int kFastReach = 64;  // most boxes reaching below -1 (offset trick) the fast form takes on

template <int CAP>
struct DetectFastSmem {
    union {
        uint64_t key[CAP];                // steps 1-2: keys in list order
        uint16_t edge[CAP * kFastEdges];  // steps 4-5: stored suppressors (slots)
    };
    union {
        uint64_t bkey[CAP];  // step 2: keys grouped by bin
        struct {             // steps 3-5
            uint32_t members[CAP];  // category buckets: slot | rank << 12 | (category >> 8) << 24
            uint8_t ecnt[CAP];      // suppressors found per slot (only ever touched with atomic add / sub on its word)
        };
    };
    float4 box[CAP];                    // list order; shifted in step 3
    uint16_t slot_a[CAP], slot_b[CAP];  // bin-grouped position / rank -> slot
    uint16_t cat[CAP], rank[CAP];
    // bit 3 more suppressors than edge[] holds (or one of another category), bits 4-5: 0 undecided 1 dead 2 kept,
    // bit 6: reaches below -1
    uint8_t meta[CAP];
    union {
        struct {
            int hist[256], start[256];  // step 2 (start runs up to the END of its bin while the bin is filled)
        };
        struct {  // steps 3-5: the boxes that reach below -1 (shifted box, slot | rank << 12, category)
            float4 rbox[kFastReach];
            float2 rraw[kFastReach];  // unshifted x1, y1
            uint32_t rsr[kFastReach];
            uint16_t rcat[kFastReach];
        };
    };
    int bsize[256], bstart[256];  // bstart runs up to the END of its bucket while the bucket is filled
    float red_f[32][2];
    int red_i[32][5];
    int wc[32];
    struct {
        int ok, trick, cross, nreach, pmin, shift;
        float span, lim;
        unsigned work;
    } c;
};

// one out-of-line copy of the predicate: the fast form runs once per image on a cold instruction cache, so the size of
// the code it walks through counts for more than the call
static __device__ __noinline__ bool fast_suppresses(const float4 a, const float4 b, float thr_f) {
    return nms_suppresses<true>(a, box_area(a), b, box_area(b), thr_f);
}

// candidate `threadIdx.x` of the list, loaded before the count is known (slot tid < cand_cap always exists in the workspace)
struct FastFirst {
    float4 b;
    float s;
    int c, id;
};

template <int CAP, int T>
__device__ int detect_fast(DetectFastSmem<CAP>& fs, int cnt, const float4* __restrict__ cbox, const float* __restrict__ cscore,
                           const int32_t* __restrict__ ccls, const int32_t* __restrict__ cid, float thr_f, int mode,
                           int cap_out, int64_t out0, int64_t* __restrict__ det_idx, float4* __restrict__ det_boxes,
                           float* __restrict__ det_scores, int64_t* __restrict__ det_classes, const FastFirst& first) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    constexpr int NW = T / 32;
    static_assert(T >= 256, "one thread per histogram bin");
    if (cnt > CAP || !(thr_f >= 0.0f)) return kFastNo;
    for (int b = tid; b < 256; b += T) {
        fs.hist[b] = 0;
        fs.bsize[b] = 0;
    }
    __syncthreads();
    // ---- 1: the list, once
    float mx = -INFINITY, mn = INFINITY;
    int fin = 1, maxcat = 0, mincat = 0, pmin = 0x7fffffff, pmax = 0;
    auto take = [&](int i, const float4 b, int c, float sc, int id) {
        const uint64_t k = ((uint64_t)score_desc_key(sc) << 32) | (uint64_t)(uint32_t)id;
        fs.key[i] = k;
        fs.box[i] = b;
        fs.cat[i] = (uint16_t)c;
        atomicAdd(&fs.bsize[c & 255], 1);
        mx = fmaxf(mx, fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w)));
        mn = fminf(mn, fminf(fminf(b.x, b.y), fminf(b.z, b.w)));
        fin &= (int)(isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w));
        maxcat = max(maxcat, c);
        mincat = min(mincat, c);
        const int p16 = (int)(k >> 48);
        pmin = min(pmin, p16);
        pmax = max(pmax, p16);
    };
    for (int i = tid; i < cnt; i += 2 * T) {  // two candidates per trip: both sets of loads are in flight together
        const int i2 = i + T;
        const bool two = i2 < cnt;
        const bool pre = i == tid;  // candidate `tid` was requested together with the count (FastFirst)
        const float4 b0 = pre ? first.b : cbox[i];
        const int c0 = pre ? first.c : ccls[i], id0 = pre ? first.id : cid[i];
        const float s0 = pre ? first.s : cscore[i];
        float4 b1 = b0;
        int c1 = 0, id1 = 0;
        float s1 = 0.0f;
        if (two) {
            b1 = cbox[i2];
            c1 = ccls[i2];
            id1 = cid[i2];
            s1 = cscore[i2];
        }
        take(i, b0, c0, s0, id0);
        if (two) take(i2, b1, c1, s1, id1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));
        mn = fminf(mn, __shfl_xor_sync(FULL, mn, o));
        fin &= __shfl_xor_sync(FULL, fin, o);
        maxcat = max(maxcat, __shfl_xor_sync(FULL, maxcat, o));
        mincat = min(mincat, __shfl_xor_sync(FULL, mincat, o));
        pmin = min(pmin, __shfl_xor_sync(FULL, pmin, o));
        pmax = max(pmax, __shfl_xor_sync(FULL, pmax, o));
    }
    if (lane == 0) {
        fs.red_f[wid][0] = mx; fs.red_f[wid][1] = mn;
        fs.red_i[wid][0] = fin; fs.red_i[wid][1] = maxcat; fs.red_i[wid][2] = mincat; fs.red_i[wid][3] = pmin;
        fs.red_i[wid][4] = pmax;
    }
    __syncthreads();
    if (wid == 0) {
        const int w = lane < NW ? lane : 0;
        mx = fs.red_f[w][0]; mn = fs.red_f[w][1];
        fin = fs.red_i[w][0]; maxcat = fs.red_i[w][1]; mincat = fs.red_i[w][2]; pmin = fs.red_i[w][3]; pmax = fs.red_i[w][4];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));
            mn = fminf(mn, __shfl_xor_sync(FULL, mn, o));
            fin &= __shfl_xor_sync(FULL, fin, o);
            maxcat = max(maxcat, __shfl_xor_sync(FULL, maxcat, o));
            mincat = min(mincat, __shfl_xor_sync(FULL, mincat, o));
            pmin = min(pmin, __shfl_xor_sync(FULL, pmin, o));
            pmax = max(pmax, __shfl_xor_sync(FULL, pmax, o));
        }
    }
    if (tid == 0) {
        // reference CPU rule: boxes.numel() <= 4000 -> coordinate-offset trick (torchvision/ops/boxes.py batched_nms)
        const bool trick = (mode == DET_NMS_AUTO) ? (cnt <= 1000) : (mode == DET_NMS_OFFSET_TRICK);
        int ok = fin && mincat >= 0 && maxcat < (1 << kSegBits) - 1;
        int cross = 0;
        float span = 0.0f, lim = 0.0f;
        if (ok && trick && cnt > 0) {  // the conditions of small_nms_body, phase 0
            span = mx + 1.0f;          // max_coordinate + torch.tensor(1).to(boxes)
            const float far = mx + (float)maxcat * span;
            if (!isfinite(far)) {
                ok = 0;
            } else if (!(mn > -1.0f)) {
                if (mx > -1.0f) {
                    cross = 1;
                    lim = -1.0f + far * 4e-6f;
                } else {
                    ok = 0;
                }
            }
        }
        fs.c.ok = ok; fs.c.trick = trick ? 1 : 0; fs.c.cross = cross; fs.c.span = span; fs.c.lim = lim;
        fs.c.nreach = 0;
        fs.c.pmin = pmin;
        const int range = pmax - pmin;
        fs.c.shift = range > 0 ? max(0, 32 - __clz(range) - 8) : 0;
    } else if (wid == 1) {  // category buckets: offsets, and the pair tests their sizes imply
        int h8[8], tot = 0, big = 0;
        unsigned sq = 0u;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            h8[q] = fs.bsize[lane * 8 + q];
            tot += h8[q];
            sq += (unsigned)h8[q] * (unsigned)h8[q];
            big |= h8[q] > 200;  // keeps the per-slot suppressor counters (bytes, atomic add / sub) far from a carry
        }
        if (__any_sync(FULL, big)) sq = 0xffffffffu;
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, incl, o);
            incl += (lane >= o) ? up : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned v = __shfl_xor_sync(FULL, sq, o);
            sq = sq + v < sq ? 0xffffffffu : sq + v;
        }
        int run = incl - tot;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            fs.bstart[lane * 8 + q] = run;
            run += h8[q];
        }
        if (lane == 0) fs.c.work = sq;
    }
    __syncthreads();
    if (!fs.c.ok || fs.c.work > (unsigned)cnt * 192u) return kFastNo;
    DET_MARK(1);
    const bool trick = fs.c.trick != 0, cross = fs.c.cross != 0;
    const float span = fs.c.span, lim = fs.c.lim;
    const int kpmin = fs.c.pmin, kshift = fs.c.shift;
    // ---- 2: counting sort by the keys' upper bits (ascending key = descending score), then the rank inside the bin
    for (int i = tid; i < cnt; i += T) atomicAdd(&fs.hist[((int)(fs.key[i] >> 48) - kpmin) >> kshift], 1);
    __syncthreads();
    if (wid == 0) {
        int h8[8], tot = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            h8[q] = fs.hist[lane * 8 + q];
            tot += h8[q];
        }
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, incl, o);
            incl += (lane >= o) ? up : 0;
        }
        int run = incl - tot;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            fs.start[lane * 8 + q] = run;
            run += h8[q];
        }
    }
    __syncthreads();
    for (int i = tid; i < cnt; i += T) {
        const uint64_t k = fs.key[i];
        const int bin = ((int)(k >> 48) - kpmin) >> kshift;
        const int pos = atomicAdd(&fs.start[bin], 1);
        fs.bkey[pos] = k;
        fs.slot_a[pos] = (uint16_t)i;
    }
    __syncthreads();
    int my_slot[(CAP + T - 1) / T], my_rank[(CAP + T - 1) / T];
#pragma unroll
    for (int u = 0; u < (CAP + T - 1) / T; ++u) {
        const int t = tid + u * T;
        my_slot[u] = -1;
        my_rank[u] = 0;
        if (t < cnt) {
            const uint64_t k = fs.bkey[t];
            const int bin = ((int)(k >> 48) - kpmin) >> kshift;
            const int b1 = fs.start[bin], b0 = b1 - fs.hist[bin];
            int r = b0;
            for (int j = b0; j < b1; ++j) r += (fs.bkey[j] < k) ? 1 : 0;  // the keys are distinct (row ids)
            my_slot[u] = (int)fs.slot_a[t];
            my_rank[u] = r;
        }
    }
    __syncthreads();  // bkey is dead: its storage becomes the bucket member lists
    DET_MARK(2);
    // ---- 3: rank table, shift, category buckets
#pragma unroll
    for (int u = 0; u < (CAP + T - 1) / T; ++u) {
        const int i = my_slot[u];
        if (i < 0) continue;
        const int r = my_rank[u];
        fs.rank[i] = (uint16_t)r;
        fs.slot_b[r] = (uint16_t)i;
        float4 b = fs.box[i];
        const int c = (int)fs.cat[i];
        const bool reaches = cross && c >= 1 && b.x < lim && b.y < lim;
        const float2 raw_xy = make_float2(b.x, b.y);
        if (trick) {
            const float off = (float)c * span;  // idxs.to(boxes) * (max_coordinate + 1)
            b.x += off; b.y += off; b.z += off; b.w += off;
            fs.box[i] = b;
        }
        if (reaches) {
            const int a = atomicAdd(&fs.c.nreach, 1);
            if (a < kFastReach) {
                fs.rbox[a] = b;
                fs.rraw[a] = raw_xy;
                fs.rsr[a] = (uint32_t)i | ((uint32_t)r << 12);
                fs.rcat[a] = (uint16_t)c;
            }
        }
        fs.meta[i] = reaches ? 64 : 0;
        fs.ecnt[i] = 0;
        fs.members[atomicAdd(&fs.bstart[c & 255], 1)] = (uint32_t)i | ((uint32_t)r << 12) | ((uint32_t)(c >> 8) << 24);
    }
    __syncthreads();
    const int nreach = fs.c.nreach;
    if (nreach > kFastReach) return kFastNo;
    DET_MARK(3);
    // the better-ranked boxes that may suppress slot i (rank p, category c): the members of its bucket, and across
    // categories the pairs named above.  f(j, box_j) -> true ends the walk
    auto walk_same = [&](int p, int c, auto f) {
        const int m1 = fs.bstart[c & 255], m0 = m1 - fs.bsize[c & 255];
        const uint32_t want_hi = (uint32_t)(c >> 8);
        uint32_t e = fs.members[m0];
        float4 bj = fs.box[e & 4095u];
        for (int q = m0; q < m1; ++q) {
            const uint32_t cur = e;
            const float4 bcur = bj;
            if (q + 1 < m1) {  // the next member and its box are on their way while this one is tested
                e = fs.members[q + 1];
                bj = fs.box[e & 4095u];
            }
            if ((int)((cur >> 12) & 4095u) < p && (cur >> 24) == want_hi && f((int)(cur & 4095u), bcur)) return true;
        }
        return false;
    };
    auto walk_cross = [&](int p, int c, bool reaches, auto f) {
        for (int a = 0; a < nreach; ++a)
            if ((int)fs.rcat[a] > c && (int)(fs.rsr[a] >> 12) < p && f((int)(fs.rsr[a] & 4095u), fs.rbox[a])) return true;
        if (reaches)
            for (int j = 0; j < cnt; ++j)
                if ((int)fs.cat[j] < c && (int)fs.rank[j] < p && f(j, fs.box[j])) return true;
        return false;
    };
    // ---- 4: suppressors.  Inside a bucket every unordered pair is tested exactly once, one thread per member: member r
    // meets member (r + d) mod m for d = 1 .. m/2 (distance-m/2 pairs of an even m from the lower half only), and a hit
    // is appended to the worse-ranked box's list
    auto add_edge = [&](int hi, int lo) {
        unsigned* w = reinterpret_cast<unsigned*>(fs.ecnt) + (hi >> 2);
        const int sh = (hi & 3) * 8;
        const int k = (int)((atomicAdd(w, 1u << sh) >> sh) & 255u);
        if (k < kFastEdges) {
            fs.edge[hi * kFastEdges + k] = (uint16_t)lo;
        } else {
            atomicSub(w, 1u << sh);
            atomicOr(reinterpret_cast<unsigned*>(fs.meta) + (hi >> 2), 8u << sh);
        }
    };
    for (int q = tid; q < cnt; q += T) {
        const uint32_t e = fs.members[q];
        const int i = (int)(e & 4095u), p = (int)((e >> 12) & 4095u);
        const float4 bi = fs.box[i];
        const int c = (int)fs.cat[i];
        const int m = fs.bsize[c & 255], m0 = fs.bstart[c & 255] - m, r = q - m0, half = m >> 1;
        const int dmax = (((m & 1) == 0) && r >= half) ? half - 1 : half;
        for (int d = 1; d <= dmax; ++d) {
            int r2 = r + d;
            r2 = r2 >= m ? r2 - m : r2;
            const uint32_t e2 = fs.members[m0 + r2];
            if ((e2 >> 24) != (e >> 24)) continue;  // another category of the same bucket
            const int j = (int)(e2 & 4095u);
            const float4 bj = fs.box[j];
            // disjoint boxes (most pairs): the intersection is exactly 0 and nothing is suppressed at a threshold >= 0
            if (!(fminf(bj.z, bi.z) > fmaxf(bj.x, bi.x) && fminf(bj.w, bi.w) > fmaxf(bj.y, bi.y))) continue;
            const bool j_first = (int)((e2 >> 12) & 4095u) < p;
            if (fast_suppresses(bj, bi, thr_f)) {  // (the predicate is symmetric in its two boxes)
                if (j_first) add_edge(i, j);
                else add_edge(j, i);
            }
        }
    }
    DET_MARK(6);
#ifdef DET_DEBUG_PHASES
    if (blockIdx.x < 64 && tid == 0) g_phase_block[blockIdx.x][7] = nreach;
#endif
    // pairs of different categories: (a box reaching below -1, a box of a lower category); a hit only flags the
    // worse-ranked of the two, which then looks for itself in the rounds
    // A reaching box of category cq > c has its shifted x1 = fl(x1 + cq * span) >= fl(RX + (c + 1) * span), RX the smallest
    // raw x1 of the reaching boxes (rounding is monotone, span > 0): a box of category c whose shifted x2 does not exceed
    // that -- nearly all of them -- meets none of them (the same in y)
    float reach_x = INFINITY, reach_y = INFINITY;
    for (int a = 0; a < nreach; ++a) {
        reach_x = fminf(reach_x, fs.rraw[a].x);
        reach_y = fminf(reach_y, fs.rraw[a].y);
    }
    for (int i = tid; i < (nreach ? cnt : 0); i += T) {
        const float4 bi = fs.box[i];
        const int c = (int)fs.cat[i];
        const float next_origin = (float)(c + 1) * span;
        if (!(bi.z > reach_x + next_origin && bi.w > reach_y + next_origin)) continue;
        const int p = (int)fs.rank[i];
        for (int a = 0; a < nreach; ++a) {
            if ((int)fs.rcat[a] <= c) continue;
            const float4 bq = fs.rbox[a];
            if (!(fminf(bq.z, bi.z) > fmaxf(bq.x, bi.x) && fminf(bq.w, bi.w) > fmaxf(bq.y, bi.y))) continue;
            const uint32_t sr = fs.rsr[a];
            const bool q_first = (int)(sr >> 12) < p;
            if (fast_suppresses(bq, bi, thr_f)) {
                const int v = q_first ? i : (int)(sr & 4095u);
                atomicOr(reinterpret_cast<unsigned*>(fs.meta) + (v >> 2), 8u << ((v & 3) * 8));
            }
        }
    }
    __syncthreads();
    DET_MARK(4);
    // ---- 5: rounds
    const volatile uint8_t* vmeta = fs.meta;
    int pending_any = 1;
    for (int round = 0; round < kFastRounds && pending_any; ++round) {
        int pending = 0;
        for (int i = tid; i < cnt; i += T) {
            const unsigned mq = vmeta[i];
            if ((mq >> 4) & 3u) continue;
            bool kept_sup = false, open_sup = false;
            const int ne = (int)fs.ecnt[i];
            for (int k = 0; k < ne; ++k) {
                const unsigned st = (vmeta[fs.edge[i * kFastEdges + k]] >> 4) & 3u;
                kept_sup |= st == 2u;
                open_sup |= st == 0u;
            }
            if (!kept_sup && (mq & 8u)) {  // more suppressors than the list holds, or one of another category
                const float4 bi = fs.box[i];
                const int c = (int)fs.cat[i], p = (int)fs.rank[i];
                auto look = [&](int j, const float4 bj) {
                    const unsigned st = (vmeta[j] >> 4) & 3u;
                    if (st == 1u) return false;
                    if (!fast_suppresses(bj, bi, thr_f)) return false;
                    if (st == 2u) {
                        kept_sup = true;
                        return true;
                    }
                    open_sup = true;
                    return false;
                };
                if (!walk_same(p, c, look) && nreach) walk_cross(p, c, (mq & 64u) != 0u, look);
            }
            if (kept_sup) fs.meta[i] = (uint8_t)(mq | (1u << 4));
            else if (!open_sup) fs.meta[i] = (uint8_t)(mq | (2u << 4));
            else pending = 1;
        }
        pending_any = __syncthreads_or(pending);
    }
    if (pending_any) return kFastNo;
    DET_MARK(5);
    // ---- 6: the first cap_out kept candidates, in rank order
    int running = 0;
    for (int p0 = 0; p0 < cnt && running < cap_out; p0 += T) {
        const int p = p0 + tid;
        const int sl = p < cnt ? (int)fs.slot_b[p] : 0;
        const bool k = p < cnt && ((fs.meta[sl] >> 4) & 3u) == 2u;
        const unsigned bal = __ballot_sync(FULL, k);
        if (lane == 0) fs.wc[wid] = __popc(bal);
        __syncthreads();
        int pre = 0, tot = 0;
        for (int w = 0; w < NW; ++w) {
            const int v = fs.wc[w];
            pre += w < wid ? v : 0;
            tot += v;
        }
        const int rank = running + pre + __popc(bal & ((1u << lane) - 1u));
        if (k && rank < cap_out) {
            const int64_t o = out0 + rank;
            det_idx[o] = (int64_t)cid[sl];
            if (det_boxes) det_boxes[o] = cbox[sl];
            if (det_scores) det_scores[o] = cscore[sl];
            if (det_classes) det_classes[o] = (int64_t)ccls[sl];
        }
        running += tot;
        __syncthreads();
    }
    return min(running, cap_out);
}

template <int CAP, int T>
__global__ void __launch_bounds__(T, 512 / T)
dense_detect_nms_kernel(int32_t* cand_count, const float4* __restrict__ cand_box,
                        const float* __restrict__ cand_score, const int32_t* __restrict__ cand_cls,
                        const int32_t* __restrict__ cand_id, int cand_cap, float thr_f, int mode, int64_t max_det,
                        int64_t* __restrict__ det_idx, float4* __restrict__ det_boxes, float* __restrict__ det_scores,
                        int64_t* __restrict__ det_classes, int32_t* __restrict__ det_count,
                        int32_t* __restrict__ overflow_flag, const FullStats* __restrict__ ext_full = nullptr,
                        int32_t* __restrict__ todo = nullptr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DetectSmem<CAP, T>& sm = *reinterpret_cast<DetectSmem<CAP, T>*>(smem_raw);
    using KL = KeyLayout<kSmallIdxBits>;
    const int img = blockIdx.x, tid = threadIdx.x;
    pdl_wait();  // no-op unless launched with launch_pdl (det_dense_detect): the candidate lists are complete from here
    DET_MARK(0);
    FastFirst first;
    first.b = make_float4(0.f, 0.f, 0.f, 0.f); first.s = 0.f; first.c = 0; first.id = 0;
    if (!ext_full && tid < cand_cap) {  // in flight together with the count
        const int64_t o = (int64_t)img * cand_cap + tid;
        first.b = cand_box[o]; first.s = cand_score[o]; first.c = cand_cls[o]; first.id = cand_id[o];
    }
    const int cnt = cand_count[(int64_t)img * kCountStride];
    if (!ext_full) {  // det_dense_detect: the counter goes back to zero for the next call on this workspace
        __syncthreads();
        if (tid == 0) cand_count[(int64_t)img * kCountStride] = 0;
    }
    if (ext_full) {  // external tier: a negative count means "no usable list", the full path takes the image
        if (tid == 0) todo[img] = (cnt < 0 || cnt > cand_cap) ? 1 : 0;
        if (cnt < 0 || cnt > cand_cap) return;
    }
    if (cnt > cand_cap) {  // the list is incomplete: report, do not guess
        if (tid == 0) {
            det_count[img] = -1;
            if (overflow_flag) atomicExch(overflow_flag, 1);
        }
        return;
    }
    const int64_t base = (int64_t)img * cand_cap;
    const int cap_out = (int)min(max_det, (int64_t)CAP);
    const int lane = tid & 31, wid = tid >> 5;
    if (!ext_full) {
        static_assert(sizeof(DetectFastSmem<CAP>) <= sizeof(DetectSmem<CAP, T>), "the fast form lives in the same shared memory");
        const int r = detect_fast<CAP, T>(*reinterpret_cast<DetectFastSmem<CAP>*>(smem_raw), cnt, cand_box + base,
                                          cand_score + base, cand_cls + base, cand_id + base, thr_f, mode, cap_out,
                                          (int64_t)img * max_det, det_idx, det_boxes, det_scores, det_classes, first);
        if (r != kFastNo) {
            if (tid == 0) det_count[img] = r;
            DET_MARK(14);
            return;
        }
        __syncthreads();
    }
    ListCandidates src{cand_box + base, cand_score + base, cand_cls + base, nullptr};
    int kept = 0;
    // Tier cut: only the first max_det detections are wanted and a box can only be suppressed by a better-scored
    // one, so the NMS first runs on the ~1.25 * max_det best candidates (every score above a 16-bit radix cut, ties
    // with the cut included).  max_det survivors there are the answer; otherwise everything is swept.  The
    // reference's branch rule and the offset trick's span are defined on ALL candidates: FullStats carries them.
    const int want_sub = cap_out + (cap_out >> 2) + 32;
    for (int tier = (cnt >= want_sub + (want_sub >> 1)) ? 0 : 1; tier < 2; ++tier) {
        int m = cnt;
        const FullStats* fs = ext_full ? ext_full + img : nullptr;
        if (tier == 0) {
            float mx = -INFINITY, mn = INFINITY;
            int fin = 1, maxcat = 0;
            uint32_t* skey = reinterpret_cast<uint32_t*>(sm.nms.sarea);
            for (int i = tid; i < cnt; i += T) {
                const float4 b = cand_box[base + i];
                mx = max_nan(mx, max_nan(max_nan(b.x, b.y), max_nan(b.z, b.w)));
                mn = min_nan(mn, min_nan(min_nan(b.x, b.y), min_nan(b.z, b.w)));
                fin &= (int)(isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w));
                maxcat = max(maxcat, cand_cls[base + i]);
                skey[i] = score_desc_key(cand_score[base + i]);
            }
            for (int o = 16; o > 0; o >>= 1) {
                mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
                fin &= __shfl_xor_sync(0xffffffffu, fin, o);
                maxcat = max(maxcat, __shfl_xor_sync(0xffffffffu, maxcat, o));
            }
            if (lane == 0) {
                sm.nms.red_max[wid] = mx;
                sm.nms.red_min[wid] = mn;
                sm.nms.red_flag[wid] = fin | (maxcat << 1);
            }
            if (tid == 0) {
                sm.sel_prefix = 0u;
                sm.sel_want = want_sub;
                sm.sub_count = 0;
            }
            __syncthreads();
            if (tid == 0) {
                float gmx = sm.nms.red_max[0], gmn = sm.nms.red_min[0];
                int gfin = sm.nms.red_flag[0] & 1, gcat = sm.nms.red_flag[0] >> 1;
                for (int w = 1; w < T / 32; ++w) {
                    gmx = max_nan(gmx, sm.nms.red_max[w]);
                    gmn = min_nan(gmn, sm.nms.red_min[w]);
                    gfin &= sm.nms.red_flag[w] & 1;
                    gcat = max(gcat, sm.nms.red_flag[w] >> 1);
                }
                sm.full.count = cnt; sm.full.mx = gmx; sm.full.mn = gmn; sm.full.fin = gfin; sm.full.maxcat = gcat;
            }
            // radix select on the two upper bytes of the descending-score keys: the bin of the want_sub-th best
            for (int shift = 24; shift >= 16; shift -= 8) {
                for (int b = tid; b < 256; b += T) sm.hist[b] = 0u;
                __syncthreads();
                const uint32_t prefix = sm.sel_prefix, himask = (shift == 24) ? 0u : 0xff000000u;
                for (int i = tid; i < cnt; i += T)
                    if ((skey[i] & himask) == prefix) atomicAdd(&sm.hist[(skey[i] >> shift) & 255u], 1u);
                __syncthreads();
                if (wid == 0) {
                    uint32_t c8[8], tot = 0;
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        c8[q] = sm.hist[lane * 8 + q];
                        tot += c8[q];
                    }
                    uint32_t incl = tot;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                        incl += (lane >= o) ? up : 0u;
                    }
                    const uint32_t want = (uint32_t)sm.sel_want, before = incl - tot;
                    if (before < want && want <= incl) {  // exactly one lane (want <= number of matching keys)
                        uint32_t run = before;
                        int q = 0;
                        for (; q < 7 && run + c8[q] < want; ++q) run += c8[q];
                        sm.sel_prefix = prefix | ((uint32_t)(lane * 8 + q) << shift);
                        sm.sel_want = (int)(want - run);
                    }
                }
                __syncthreads();
            }
            const uint32_t cut = sm.sel_prefix | 0xffffu;  // every key of the chosen 16-bit bin and all better ones
            for (int i0 = 0; i0 < cnt; i0 += T) {
                const int i = i0 + tid;
                const bool in = i < cnt && skey[i] <= cut;
                const unsigned bal = __ballot_sync(0xffffffffu, in);
                int pos = 0;
                if (lane == 0 && bal) pos = atomicAdd(&sm.sub_count, __popc(bal));
                pos = __shfl_sync(0xffffffffu, pos, 0);
                if (in) sm.perm[pos + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)i;
            }
            __syncthreads();
            m = sm.sub_count;
            if (!ext_full) fs = &sm.full;  // external tier: the statistics of the whole image came with the list
            src.perm = sm.perm;
        } else {
            src.perm = nullptr;
        }
        // The list was filled in arrival order, the oracle's candidates come in row order (torch.nonzero).  The order
        // only matters where two scores tie, so the first attempt uses the list as it is and looks for ties: inside a
        // category segment (small_nms_body flags them) they may have changed the outcome and the image is redone with
        // the slots in row order (rare); ties of different segments only meet in the final list, where each run of
        // equal scores is put into row order by the thread that owns its first entry.
        const int npad = next_pow2(max(m, 2));
        for (bool presort = false;; presort = true) {
            if (presort) {
                for (int i = tid; i < npad; i += T) {
                    const int slot = (i < m) ? src.slot(i) : 0;
                    sm.nms.keys[i] = (i < m) ? (((uint64_t)(uint32_t)cand_id[base + slot] << kSmallIdxBits) | (uint64_t)slot)
                                             : kSentinelKey;
                }
                __syncthreads();
                cta_bitonic_sort<T>(sm.nms.keys, npad);
                for (int i = tid; i < m; i += T) sm.perm[i] = (uint16_t)(sm.nms.keys[i] & ((1u << kSmallIdxBits) - 1u));
                __syncthreads();
                src.perm = sm.perm;
            }
            DET_MARK(1);
            kept = small_nms_body<CAP, T>(sm.nms, src, m, thr_f, mode, cap_out, fs);
            if (presort) break;
            int redo = sm.nms.tie;
            if (!redo) {
                for (int j = tid; j + 1 < kept; j += T) {
                    const uint64_t sc = sm.nms.keys[j] >> KL::kScoreShift;
                    if ((sm.nms.keys[j + 1] >> KL::kScoreShift) != sc) continue;
                    if (j > 0 && (sm.nms.keys[j - 1] >> KL::kScoreShift) == sc) continue;  // not the head of the run
                    int len = 2;
                    while (j + len < kept && (sm.nms.keys[j + len] >> KL::kScoreShift) == sc) ++len;
                    if (len > 16) {
                        redo = 1;
                        break;
                    }
                    for (int a = 0; a + 1 < len; ++a)  // selection sort by row index; only this thread writes the run
                        for (int b = a + 1; b < len; ++b) {
                            const uint64_t ka = sm.nms.keys[j + a], kb = sm.nms.keys[j + b];
                            if (cand_id[base + src.slot((int)KL::idx(kb))] < cand_id[base + src.slot((int)KL::idx(ka))]) {
                                sm.nms.keys[j + a] = kb;
                                sm.nms.keys[j + b] = ka;
                            }
                        }
                }
            }
            if (!__syncthreads_or(redo)) break;
        }
        if (kept < 0 || kept >= cap_out) break;  // bad category, or the tier already holds max_det survivors
    }
    if (ext_full && kept >= 0 && kept < cap_out && cnt < ext_full[img].count) {
        if (tid == 0) todo[img] = 1;  // the best-scored subset fell short of max_out survivors: full path
        return;
    }
    const int nout = kept < 0 ? 0 : min(kept, cap_out);
    for (int j = tid; j < nout; j += T) {
        const int slot = src.slot((int)KL::idx(sm.nms.keys[j]));
        const int64_t o = (int64_t)img * max_det + j;
        det_idx[o] = (int64_t)cand_id[base + slot];
        if (det_boxes) det_boxes[o] = cand_box[base + slot];
        if (det_scores) det_scores[o] = cand_score[base + slot];
        if (det_classes) det_classes[o] = (int64_t)cand_cls[base + slot];
    }
    if (tid == 0) det_count[img] = kept < 0 ? -1 : nout;
    DET_MARK(14);
}

// The per-image candidate lists of a det_dense_detect / det_roi_detect workspace, and what the select kernel that fills
// them is told (mode and score_thresh: det_dense_detect's select kernel only).
struct SelectArgs {
    int mode;  // kModeSelect / kModeSelectGated
    float score_thresh;
    int cand_cap;
    int32_t* cand_count;  // one counter every kCountStride words
    float4* cand_box;
    float* cand_score;
    int32_t* cand_cls;
    int32_t* cand_id;
    int32_t* overflow_flag;
};

// Points the lists of `sel` (and its cand_cap) into `workspace`: counters (one per 128-byte line), boxes, scores,
// classes, ids -- det_dense_detect_workspace_bytes(n, cand_cap) bytes, 16-byte aligned, else DET_ERR_WORKSPACE /
// DET_ERR_ALIGN.  The counters are cleared on `st` unless `counters_zero` (gate bit 1: the NMS CTAs leave them zero).
// Defined in dense_decode.cu.
int bind_select_workspace(SelectArgs& sel, int n, int64_t cand_cap, void* workspace, int64_t workspace_bytes,
                          bool counters_zero, cudaStream_t st);

// dense_detect_nms_kernel over the n lists of `sel` (cand_cap <= 4096), launched with programmatic dependent launch
// behind the select kernel that filled them: the second launch of det_dense_detect and det_roi_detect.  The tie order
// is ascending cand_id.  Defined in dense_decode.cu.
int launch_list_nms(const SelectArgs& sel, int n, float thr_f, int mode, int64_t max_det, int64_t* det_idx,
                    float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count, int32_t* overflow_flag,
                    cudaStream_t st);

}  // namespace det
