// PAF candidate scoring + exact std::sort + greedy one-to-one matching (pafprocess.cpp:47-125) as a kernel family.
//
// Round-1 ran all of this in one block per (image, limb); the step was then bound by the block of the largest limb
// (4.4 of 5.3 ms) and by a work-queue quicksort that spent most of its instructions on bookkeeping.  The family below
// cuts the work along its natural seams, every stage a grid that balances itself:
//
//   limb_plan_kernel   (1 block)            per (image, limb): pair count, slot ranges in the two key pools, first
//                                            scoring work item; totals; zeroes the cursors
//   limb_score_kernel  (dynamic work list)   work item = 2048 consecutive (a, b) pairs of one limb; every warp scores 256
//                                            of them (10 PAF samples each, the limb's two PAF planes staged in shared
//                                            memory) and compacts the survivors IN ORDER into its slot of pool A
//   limb_gather_kernel (image x limb)        packs the warp slots into the limb's contiguous candidate list in pool B
//                                            (= the order the reference pushes candidates in), then runs the top levels
//                                            of libstdc++'s introsort in global memory until every range fits shared
//                                            memory; emits the ranges
//   range_sort_kernel  (dynamic range list)  exact introsort of one range (<= 4096 keys) in shared memory, LEVEL-
//                                            SYNCHRONOUS: all partitions of a recursion level run together, every
//                                            thread walks rows of keys, ranks come from ballots (see below)
//   limb_greedy_kernel (image x limb)        the greedy one-to-one assignment over the sorted list
//
// Exactness: the reference sorts with std::sort (unstable introsort) and exactly equal scores are common (two peaks
// refined to the same pixel), so the order of ties is observable.  Everything here reproduces __introsort_loop +
// __final_insertion_sort element for element (rank formulation of the Hoare partition, post_core.h).
#include <cstdio>
#include <vector>

#include "host_util.h"
#include "postprocess.cuh"

namespace b2p {

namespace {

__constant__ int c_lparts[kNumLimb][2] = B2P_LIMB_TABLES;
__constant__ int c_lpaf[kNumLimb][2] = B2P_LIMB_PAF_TABLES;

const int c_host_limb0[2] = {1, 2};            // parts of limb 0 (B2P_LIMB_TABLES), for the test hook
constexpr int kChunkPairs = kLimbChunkPairs;   // pairs per scoring work item
constexpr int kScoreThreads = 256;             // 8 warps x 256 pairs
constexpr int kSubPairs = 256;
constexpr int kSubPerChunk = kChunkPairs / kSubPairs;
static_assert(kSubPerChunk * 32 == kScoreThreads, "one warp per sub-chunk");

#ifndef B2P_GATHER_THREADS
#define B2P_GATHER_THREADS 512
#endif
constexpr int kGatherThreads = B2P_GATHER_THREADS, kGatherWarps = kGatherThreads / 32;
constexpr int kS = kLimbSmemRange;             // keys per shared-memory range
constexpr int kSortThreads = 512, kSortWarps = kSortThreads / 32;
constexpr int kGreedyThreads = 512, kGreedySeg = 2048, kGreedyPer = kGreedySeg / kGreedyThreads;
constexpr int kBigStack = 96;
constexpr int kBalRows = 4096;                 // ballot cache of the global-memory partitions: up to 131072 keys

__device__ __forceinline__ uint32_t key_hi(const unsigned long long* keys, int i) {
    return reinterpret_cast<const uint32_t*>(keys)[2 * i + 1];
}

// Longest-job-first: block `rank` of an image takes the limb with the rank-th largest number of (a, b) pairs.
// One warp: lane l ranks limb l.
__device__ __forceinline__ int limb_of_rank_warp(const PostBuffers& pb, int img, int rank_y) {
    const int lane = threadIdx.x & 31;
    const int mine = lane < kNumLimb ? pb.counts[img * kNumPart + c_lparts[lane][0]] * pb.counts[img * kNumPart + c_lparts[lane][1]] : -1;
    int rank = 0;
    for (int m = 0; m < kNumLimb; ++m) {
        const int pm = __shfl_sync(0xffffffffu, mine, m);
        rank += (pm > mine) || (pm == mine && m < lane);
    }
    const uint32_t hit = __ballot_sync(0xffffffffu, lane < kNumLimb && rank == rank_y);
    return hit ? __ffs(hit) - 1 : rank_y;
}

// ------------------------------------------------------------------ plan
__global__ void __launch_bounds__(1024) limb_plan_kernel(PostBuffers pb, int batch) {
    __shared__ long long s_wr[32];
    __shared__ int s_ww[32];
    __shared__ long long s_carry_reg;
    __shared__ int s_carry_work;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = batch * kNumLimb;
    const long long half = pb.pool_cap / 2;
    if (tid == 0) { s_carry_reg = 0; s_carry_work = 0; }
    __syncthreads();
    for (int base = 0; base < N; base += 1024) {
        const int i = base + tid;
        int na = 0, nb = 0, img = 0, limb = 0;
        long long reg = 0;
        if (i < N) {
            img = i / kNumLimb;
            limb = i - img * kNumLimb;
            na = pb.counts[img * kNumPart + c_lparts[limb][0]];
            nb = pb.counts[img * kNumPart + c_lparts[limb][1]];
            if (na > 0 && nb > 0) reg = (long long)na * nb + 2;       // + 2: the partition scratch needs 2 (n + 2) int32
        }
        // exclusive scan of the region sizes
        long long r = reg;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, r, o);
            if (lane >= o) r += t;
        }
        if (lane == 31) s_wr[warp] = r;
        __syncthreads();
        if (warp == 0) {
            long long w = s_wr[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            s_wr[lane] = wi - w;
        }
        __syncthreads();
        const long long reg0 = s_carry_reg + s_wr[warp] + r - reg;
        const bool fits = reg0 + reg <= half;
        if (i < N && reg > 0 && !fits) atomicOr(&pb.status[img], 2);       // candidate pool exhausted: loud
        const int nch = (reg > 0 && fits) ? (int)((reg - 2 + kChunkPairs - 1) / kChunkPairs) : 0;
        int w = nch;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        if (lane == 31) s_ww[warp] = w;
        __syncthreads();
        if (warp == 0) {
            int v = s_ww[lane], vi = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, vi, o);
                if (lane >= o) vi += t;
            }
            s_ww[lane] = vi - v;
        }
        __syncthreads();
        if (i < N) {
            LimbPlan pl;
            pl.na = (reg > 0 && fits) ? na : 0;
            pl.nb = (reg > 0 && fits) ? nb : 0;
            pl.nchunks = nch;
            pl.work0 = s_carry_work + s_ww[warp] + w - nch;
            pl.n = 0;
            pl.region = reg0;
            pb.lplan[i] = pl;
        }
        __syncthreads();
        if (tid == 1023) {          // inclusive values of the last thread = tile totals
            s_carry_reg += s_wr[31] + r;
            s_carry_work += s_ww[31] + w;
        }
        __syncthreads();
    }
    if (tid == 0) {
        pb.cursors[0] = 0;                  // scoring work cursor
        pb.cursors[1] = s_carry_work;       // scoring work items
        pb.cursors[2] = 0;                  // ranges emitted
        pb.cursors[3] = 0;                  // range cursor
    }
}

// ------------------------------------------------------------------ scoring
struct PlanePaf {          // the limb's two PAF planes in shared memory: channel 0 / 1, low resolution
    const float* pl;
    int lw, hw;
    __device__ __forceinline__ float at(int c, int y, int x) const { return pl[c * hw + (y >> 3) * lw + (x >> 3)]; }
};

__global__ void __launch_bounds__(kScoreThreads) limb_score_kernel(PostBuffers pb, PafView paf0, long p_img, int h_up,
                                                                   int lw, int lh, int paf_in_smem, int n_limbs,
                                                                   const int2* __restrict__ dims) {
    extern __shared__ float s_planes[];
    __shared__ int s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cap = pb.peak_cap;
    const int hw = lw * lh;
    const uint32_t lt = (1u << lane) - 1u;
    int staged = -1;
    constexpr int kGroup = 4;      // consecutive work items per grab: they mostly belong to one limb, whose planes stay staged
    for (int it0 = 0;; ++it0) {
        const int sub = it0 & (kGroup - 1);
        if (sub == 0) {
            __syncthreads();                 // the previous group is done with s_item
            if (tid == 0) s_item = atomicAdd(pb.cursors + 0, kGroup);
            __syncthreads();
        }
        const int item = s_item + sub;
        if (item >= pb.cursors[1]) {
            if (sub == 0) return;
            continue;                        // tail of the last group (uniform)
        }
        // the limb of this work item: last plan entry with work0 <= item
        int lo = 0, hi = n_limbs - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (pb.lplan[mid].work0 <= item) lo = mid; else hi = mid - 1;
        }
        const int li = lo;
        const LimbPlan pl = pb.lplan[li];
        const int img = li / kNumLimb, limb = li - img * kNumLimb;
        const int chunk = item - pl.work0;
        const int img_h_up = dims != nullptr ? 8 * dims[img].x : h_up;     // ragged batch: the image's own padded height
        const int pa = c_lparts[limb][0], pbp = c_lparts[limb][1];
        const int c1 = c_lpaf[limb][0], c2 = c_lpaf[limb][1];
        PafView paf = paf0;
        paf.base += img * p_img;
        if (paf_in_smem && staged != li) {
            __syncthreads();                 // every warp is done with the planes of the previous limb
            if (paf.sx == 1 && paf.sy == lw) {          // planar maps (the network's NCHW outputs): two contiguous planes
                const float* p1 = paf.base + c1 * paf.sc;
                const float* p2 = paf.base + c2 * paf.sc;
                for (int i = tid; i < hw; i += kScoreThreads) { s_planes[i] = p1[i]; s_planes[hw + i] = p2[i]; }
            } else {
                for (int i = tid; i < 2 * hw; i += kScoreThreads) {
                    const int ch = i >= hw, r = i - ch * hw;
                    s_planes[i] = paf.base[(ch ? c2 : c1) * paf.sc + (long)(r / lw) * paf.sy + (long)(r % lw) * paf.sx];
                }
            }
            staged = li;
            __syncthreads();
        }
        const int nb = pl.nb;
        const long npairs = (long)pl.na * nb;
        const long start = (long)chunk * kChunkPairs + warp * kSubPairs;
        int cnt = 0;
        if (start < npairs) {
            const int* axp = pb.peak_x + ((long)img * kNumPart + pa) * cap;
            const int* ayp = pb.peak_y + ((long)img * kNumPart + pa) * cap;
            const int* bxp = pb.peak_x + ((long)img * kNumPart + pbp) * cap;
            const int* byp = pb.peak_y + ((long)img * kNumPart + pbp) * cap;
            unsigned long long* dst = pb.pool + pl.region + start;
            long p = start + lane;
            int a = (int)(p / nb), b = (int)(p - (long)a * nb);
            const PlanePaf pp{s_planes, lw, hw};
#pragma unroll 1
            for (int it = 0; it < kSubPairs / 32; ++it, p += 32) {
                float sc = 0.f;
                bool pass = false;
                if (p < npairs) {
                    const int ax = __ldg(axp + a), ay = __ldg(ayp + a), bx = __ldg(bxp + b), by = __ldg(byp + b);
                    pass = paf_in_smem ? pair_score_t(pp, 0, 1, ax, ay, bx, by, img_h_up, &sc)
                                       : pair_score_t(paf, c1, c2, ax, ay, bx, by, img_h_up, &sc);
                }
                const unsigned m = __ballot_sync(0xffffffffu, pass);
                if (pass) dst[cnt + __popc(m & lt)] = cand_key(sc, (uint32_t)p);
                cnt += __popc(m);
                b += 32;
                while (b >= nb) { b -= nb; ++a; }
            }
        }
        if (lane == 0) pb.sub_cnt[(long)item * kSubPerChunk + warp] = cnt;
    }
}

// ------------------------------------------------------------------ block-wide exact partition in global memory
// Rank formulation of libstdc++'s __unguarded_partition_pivot (post_core.h), evaluated row-wise by the whole block:
// every warp owns a contiguous segment of rows, lanes take consecutive keys, ranks come from ballots + running counts.
struct PartShared {
    unsigned long long scan2[16];
    int ksum;
};
template <class PosT, int kThreads>
__device__ int block_rank_partition(unsigned long long* v, int f, int l, PosT* tabA, PosT* tabB, PartShared& sh,
                                    uint32_t* bal = nullptr /* optional cache of 2 x rows stop-flag ballots */) {
    constexpr int kWarps = kThreads / 32;
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u, gt = ~lt & ~(1u << lane);
    if (tid == 0) {       // __move_median_to_first(first, first+1, mid, last-1)
        const long a = f + 1, b = f + (l - f) / 2, c = l - 1;
        long m;
        if (B2P_COMP(v[a], v[b])) m = B2P_COMP(v[b], v[c]) ? b : (B2P_COMP(v[a], v[c]) ? c : a);
        else m = B2P_COMP(v[a], v[c]) ? a : (B2P_COMP(v[b], v[c]) ? c : b);
        const unsigned long long t = v[f]; v[f] = v[m]; v[m] = t;
        sh.ksum = 0;
    }
    __syncthreads();
    const uint32_t pivot = (uint32_t)(v[f] >> 32);
    const int base = f + 1;
    const int rows = (l - base + 31) >> 5;
    const int rpw = (rows + kWarps - 1) / kWarps;
    const int r0 = min(rows, wq * rpw), r1 = min(rows, r0 + rpw);
    int cA = 0, cB = 0;
    for (int r = r0; r < r1; ++r) {
        const int p = base + (r << 5) + lane;
        const uint32_t k = p < l ? (uint32_t)(v[p] >> 32) : 0u;
        const uint32_t mA = __ballot_sync(0xffffffffu, p < l && k >= pivot);
        const uint32_t mB = __ballot_sync(0xffffffffu, p < l && k <= pivot);
        if (bal != nullptr && lane == 0) { bal[2 * r] = mA; bal[2 * r + 1] = mB; }
        cA += __popc(mA);
        cB += __popc(mB);
    }
    if (lane == 0) sh.scan2[wq] = ((unsigned long long)(unsigned)cB << 32) | (unsigned)cA;
    __syncthreads();
    unsigned long long pre = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < kWarps; ++k) {
        const unsigned long long c = sh.scan2[k];
        if (k < wq) pre += c;
        tot += c;
    }
    const int offA = (int)(unsigned)pre, offB = (int)(pre >> 32);
    const int totA = (int)(unsigned)tot, totB = (int)(tot >> 32);
    int run = offA;
    for (int r = r0; r < r1; ++r) {          // lo-stops ranked from the left
        const int p = base + (r << 5) + lane;
        const uint32_t m = bal != nullptr ? bal[2 * r]
                                          : __ballot_sync(0xffffffffu, p < l && (uint32_t)(v[p] >> 32) >= pivot);
        if ((m >> lane) & 1u) tabA[run + __popc(m & lt) + 1] = (PosT)(p - f);
        run += __popc(m);
    }
    run = totB - offB - cB;                  // hi-stops ranked from the right
    for (int r = r1 - 1; r >= r0; --r) {
        const int p = base + (r << 5) + lane;
        const uint32_t m = bal != nullptr ? bal[2 * r + 1]
                                          : __ballot_sync(0xffffffffu, p < l && (uint32_t)(v[p] >> 32) <= pivot);
        if ((m >> lane) & 1u) tabB[run + __popc(m & gt) + 1] = (PosT)(p - f);
        run += __popc(m);
    }
    __syncthreads();
    const int lim = totA < totB ? totA : totB;
    int c = 0;
    for (int k = 1 + tid; k <= lim; k += kThreads) c += (tabA[k] < tabB[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0 && c) atomicAdd(&sh.ksum, c);
    __syncthreads();
    const int K = sh.ksum;
    for (int k = 1 + tid; k <= K; k += kThreads) {
        const int ia = f + (int)tabA[k], ib = f + (int)tabB[k];
        const unsigned long long t = v[ia]; v[ia] = v[ib]; v[ib] = t;
    }
    const int a_next = (K + 1 <= totA) ? f + (int)tabA[K + 1] : l;
    const int cut = (K > 0 && f + (int)tabB[K] < a_next) ? f + (int)tabB[K] : a_next;
    __syncthreads();
    return cut;
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* total, int* scratch /*[warps + 1]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) scratch[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        int w = lane < nw ? scratch[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < nw) scratch[lane] = winc - w;
        if (lane == nw - 1) scratch[nw] = winc;
    }
    __syncthreads();
    const int res = scratch[warp] + inc - v;
    *total = scratch[blockDim.x >> 5];
    __syncthreads();
    return res;
}

__device__ __forceinline__ void emit_range(const PostBuffers& pb, int img, long off, int len, int depth) {
    const int idx = atomicAdd(pb.cursors + 2, 1);
    if (idx < pb.range_cap) pb.ranges[idx] = SortRange{off, len, depth};
    else atomicOr(&pb.status[img], 2);
}

// ------------------------------------------------------------------ gather + top-level partitions
__global__ void __launch_bounds__(kGatherThreads) limb_gather_kernel(PostBuffers pb) {
    __shared__ int scan_scratch[kGatherWarps + 1];
    __shared__ PartShared s_part;
    __shared__ int s_carry;
    __shared__ int g_top, g_f[kBigStack], g_l[kBigStack], g_d[kBigStack];
    __shared__ uint32_t s_bal[2 * kBalRows];        // stop-flag ballots of a partition: passes 2 and 3 do not re-read the keys
    __shared__ int s_limb;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int img = blockIdx.x;
    if (warp == 0) {
        const int l = limb_of_rank_warp(pb, img, blockIdx.y);
        if (lane == 0) s_limb = l;
    }
    __syncthreads();
    const int limb = s_limb;
    const int li = img * kNumLimb + limb;
    const LimbPlan pl = pb.lplan[li];
    if (pl.nchunks == 0) return;                                      // no pairs (pl.n stays 0)
    const int nsub = pl.nchunks * kSubPerChunk;
    const int* cnt = pb.sub_cnt + (long)pl.work0 * kSubPerChunk;
    int* off = pb.sub_off + (long)pl.work0 * kSubPerChunk;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < nsub; base += kGatherThreads) {
        const int s = base + tid;
        const int c = s < nsub ? cnt[s] : 0;
        int tot;
        const int ex = block_exclusive_scan(c, &tot, scan_scratch);
        if (s < nsub) off[s] = s_carry + ex;
        __syncthreads();
        if (tid == 0) s_carry += tot;
        __syncthreads();
    }
    const int n = s_carry;
    const unsigned long long* src = pb.pool + pl.region;
    unsigned long long* keys = pb.pool + pb.pool_cap / 2 + pl.region;   // pool B: the contiguous list
    for (int s = warp; s < nsub; s += kGatherWarps) {
        const int c = cnt[s], o = off[s];
        for (int i = lane; i < c; i += 32) keys[o + i] = src[(long)s * kSubPairs + i];
    }
    if (tid == 0) pb.lplan[li].n = n;
    if (n <= 1) return;
    int lg = 0;
    for (int m = n; m > 1; m >>= 1) ++lg;
    const long key_off = pb.pool_cap / 2 + pl.region;
    if (n <= kS) {
        if (tid == 0) emit_range(pb, img, key_off, n, 2 * lg);
        return;
    }
    __threadfence();
    __syncthreads();
    // top levels of __introsort_loop in global memory; pool A is free again: rank -> position scratch
    int32_t* gA = reinterpret_cast<int32_t*>(pb.pool + pl.region);
    int32_t* gB = gA + n + 2;
    if (tid == 0) { g_top = 1; g_f[0] = 0; g_l[0] = n; g_d[0] = 2 * lg; }
    __syncthreads();
    for (;;) {
        __syncthreads();
        if (g_top == 0) break;
        const int t = g_top - 1;
        const int f = g_f[t], l = g_l[t], d = g_d[t];
        __syncthreads();
        if (tid == 0) g_top = t;
        if (l - f <= kS) {
            if (tid == 0) emit_range(pb, img, key_off + f, l - f, d);
        } else if (d == 0) {
            if (tid == 0) seq_heap_sort(reinterpret_cast<uint64_t*>(keys), f, l);     // depth limit: std::__partial_sort
        } else {
            const int cut = block_rank_partition<int32_t, kGatherThreads>(keys, f, l, gA, gB, s_part,
                                                          (l - f - 1 + 31) / 32 <= kBalRows ? s_bal : nullptr);
            if (tid == 0) {
                int q = g_top;
                if (q + 2 <= kBigStack) {
                    g_f[q] = f; g_l[q] = cut; g_d[q] = d - 1; ++q;
                    g_f[q] = cut; g_l[q] = l; g_d[q] = d - 1; ++q;
                    g_top = q;
                } else {        // unreachable (stack depth <= 2 + 2 log2 n): finish sequentially, exactly
                    seq_sort_range(reinterpret_cast<uint64_t*>(keys), f, cut, d - 1);
                    seq_sort_range(reinterpret_cast<uint64_t*>(keys), cut, l, d - 1);
                }
            }
        }
    }
}

// ------------------------------------------------------------------ exact introsort of one range in shared memory
// One block sorts one range of n <= kS keys with depth budget d, reproducing __introsort_loop (+ the part of
// __final_insertion_sort that falls into the range).  The recursion is walked LEVEL BY LEVEL (one block barrier per
// level; the segments of a level are independent), and a segment is partitioned by as many threads as it can feed:
//   > kWarpSeg keys   the whole block, one segment at a time (block_rank_partition: ranks from ballots + per-warp counts)
//   > kLaneT keys     ONE WARP per segment, 16 segments side by side: the stop flags of the segment's <= 32 rows are
//                     ballots held in registers (lane r keeps row r), their prefix sums are two warp scans, the rank ->
//                     position tables live in the segment's own slice of the table arrays - no block barrier, no queue
//   <= kLaneT keys    ONE LANE per segment after the last level: the sequential routine (the rest of the recursion + the
//                     insertion sort of its leaves) on hundreds of segments side by side.  A lane spends ~10 instructions
//                     per key and level where a cooperative partition spends ~50 lane slots, and below kLaneT keys
//                     there are enough segments to keep the lanes busy.
constexpr int kLaneT = B2P_LANE_SORT_KEYS;
constexpr int kWarpSeg = 1024;                 // <= 32 rows of 32 keys behind the pivot
constexpr int kSegMax = kS / (kLaneT + 1) + 2;    // segments longer than kLaneT in one level
constexpr int kSmallMax = kS / 17 + 2;            // segments handed to single lanes: disjoint, more than 16 keys each
struct Seg { uint16_t f, l; uint8_t d, pad; };
struct SortSmem {
    unsigned long long keys[kS];
    uint16_t tabA[kS + 32], tabB[kS + 32];
    Seg segs[2][kSegMax];
    Seg bigs[2][kS / kWarpSeg + 1];
    Seg small[kSmallMax];
    int nseg[2], nbig[2], nsmall;
    PartShared part;
    int range_idx, cut;
};

// Sequential exact __introsort_loop of the small segment v[first, last) with depth budget `depth`, by ONE lane: partitions
// until every part has <= 16 keys (the parts themselves are left to the final insertion pass).  post_core.h's
// seq_sort_range with 32-bit indices and a stack sized for kLaneT keys (a right part is only stacked when it has more
// than 16 keys, so a segment of n keys stacks at most n / 17 of them).
constexpr int kLaneStack = kLaneT / 17 + 2;
__device__ void lane_partition_segment(unsigned long long* v, int first, int last, int depth) {
    int sf[kLaneStack], sl[kLaneStack], sd[kLaneStack], sp = 1;
    sf[0] = first; sl[0] = last; sd[0] = depth;
    while (sp > 0) {
        --sp;
        int f = sf[sp], l = sl[sp], d = sd[sp];
        while (l - f > 16) {
            if (d == 0) { seq_heap_sort(reinterpret_cast<uint64_t*>(v), f, l); break; }
            --d;
            const int a = f + 1, b = f + (l - f) / 2, c = l - 1;
            int m;
            if (B2P_COMP(v[a], v[b])) m = B2P_COMP(v[b], v[c]) ? b : (B2P_COMP(v[a], v[c]) ? c : a);
            else m = B2P_COMP(v[a], v[c]) ? a : (B2P_COMP(v[b], v[c]) ? c : b);
            { const unsigned long long t = v[f]; v[f] = v[m]; v[m] = t; }
            const uint32_t pivot = (uint32_t)(v[f] >> 32);
            int lo = f + 1, hi = l;
            for (;;) {
                while ((uint32_t)(v[lo] >> 32) < pivot) ++lo;
                --hi;
                while (pivot < (uint32_t)(v[hi] >> 32)) --hi;
                if (!(lo < hi)) break;
                const unsigned long long t = v[lo]; v[lo] = v[hi]; v[hi] = t;
                ++lo;
            }
            if (l - lo > 16) { sf[sp] = lo; sl[sp] = l; sd[sp] = d; ++sp; }      // sp < kLaneStack: see above
            l = lo;
        }
    }
}

// files the segment [f, l) with depth budget d (one thread): next level's list, the lanes' list, or - budget spent -
// heap sort on the spot (std::__partial_sort, rare)
__device__ void push_segment(SortSmem& S, int f, int l, int d, int nx) {
    const int m = l - f;
    if (m <= 16) return;                       // a leaf: the final insertion pass sorts it
    if (m <= kLaneT) {
        const int i = atomicAdd(&S.nsmall, 1);
        S.small[i] = Seg{(uint16_t)f, (uint16_t)l, (uint8_t)d, 0};
    } else if (d == 0) {
        seq_heap_sort(reinterpret_cast<uint64_t*>(S.keys), f, l);
    } else if (m > kWarpSeg) {
        const int i = atomicAdd(&S.nbig[nx], 1);
        S.bigs[nx][i] = Seg{(uint16_t)f, (uint16_t)l, (uint8_t)d, 0};
    } else {
        const int i = atomicAdd(&S.nseg[nx], 1);
        S.segs[nx][i] = Seg{(uint16_t)f, (uint16_t)l, (uint8_t)d, 0};
    }
}

// exact partition of keys[f, l), 64 < l - f <= kWarpSeg, by one warp; returns the cut (all lanes)
__device__ int warp_rank_partition(SortSmem& S, int f, int l) {
    const int lane = threadIdx.x & 31;
    unsigned long long* v = S.keys;
    const uint32_t lt = (1u << lane) - 1u, gt = ~lt & ~(1u << lane);
    if (lane == 0) {       // __move_median_to_first(first, first+1, mid, last-1)
        const int a = f + 1, b = f + (l - f) / 2, c = l - 1;
        int m;
        if (B2P_COMP(v[a], v[b])) m = B2P_COMP(v[b], v[c]) ? b : (B2P_COMP(v[a], v[c]) ? c : a);
        else m = B2P_COMP(v[a], v[c]) ? a : (B2P_COMP(v[b], v[c]) ? c : b);
        const unsigned long long t = v[f]; v[f] = v[m]; v[m] = t;
    }
    __syncwarp();
    const uint32_t* kw = reinterpret_cast<const uint32_t*>(v);
    const uint32_t pivot = kw[2 * f + 1];
    const int base = f + 1;
    const int rows = (l - base + 31) >> 5;          // <= 32
    uint32_t myA = 0u, myB = 0u;                    // stop flags of row `lane`
    for (int r = 0; r < rows; ++r) {
        const int p = base + (r << 5) + lane;
        const uint32_t k = p < l ? kw[2 * p + 1] : 0u;
        const uint32_t bA = __ballot_sync(0xffffffffu, p < l && k >= pivot);
        const uint32_t bB = __ballot_sync(0xffffffffu, p < l && k <= pivot);
        if (lane == r) { myA = bA; myB = bB; }
    }
    const int cA = __popc(myA), cB = __popc(myB);
    int incA = cA, incB = cB;                       // inclusive prefix over rows (A), inclusive suffix (B)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int ta = __shfl_up_sync(0xffffffffu, incA, o);
        const int tb = __shfl_down_sync(0xffffffffu, incB, o);
        if (lane >= o) incA += ta;
        if (lane + o < 32) incB += tb;
    }
    const int totA = __shfl_sync(0xffffffffu, incA, 31), totB = __shfl_sync(0xffffffffu, incB, 0);
    const int preA = incA - cA, sufB = incB - cB;   // lo-stops in earlier rows, hi-stops in later rows
    uint16_t* tabA = S.tabA + f;
    uint16_t* tabB = S.tabB + f;
    for (int r = 0; r < rows; ++r) {
        const uint32_t bA = __shfl_sync(0xffffffffu, myA, r), bB = __shfl_sync(0xffffffffu, myB, r);
        const int pa = __shfl_sync(0xffffffffu, preA, r), sb = __shfl_sync(0xffffffffu, sufB, r);
        const int p = base + (r << 5) + lane;
        if ((bA >> lane) & 1u) tabA[pa + __popc(bA & lt) + 1] = (uint16_t)p;
        if ((bB >> lane) & 1u) tabB[sb + __popc(bB & gt) + 1] = (uint16_t)p;
    }
    __syncwarp();
    const int lim = totA < totB ? totA : totB;
    int c = 0;
    for (int k = 1 + lane; k <= lim; k += 32) c += (tabA[k] < tabB[k]);       // monotone: the count is K
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    const int K = c;
    for (int k = 1 + lane; k <= K; k += 32) {
        const int ia = tabA[k], ib = tabB[k];
        const unsigned long long t = v[ia]; v[ia] = v[ib]; v[ib] = t;
    }
    const int a_next = (K + 1 <= totA) ? (int)tabA[K + 1] : l;
    const int cut = (K > 0 && (int)tabB[K] < a_next) ? (int)tabB[K] : a_next;
    __syncwarp();
    return cut;
}

__device__ void smem_level_sort(SortSmem& S, int n, int depth) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        S.nseg[0] = 0; S.nseg[1] = 0; S.nbig[0] = 0; S.nbig[1] = 0; S.nsmall = 0;
        push_segment(S, 0, n, depth, 0);
    }
    __syncthreads();
    int level = 0;
    for (int cur = 0;; cur ^= 1) {
        const int cnt = S.nseg[cur], nbig = S.nbig[cur];
        if (cnt == 0 && nbig == 0) break;
        if (++level > 2 * 64 + 8) {      // every level consumes depth budget (<= 2 log2 n <= 64): a bug must trap, not hang the box
            if (tid == 0) printf("[b200pose] level-wise sort did not terminate (n=%d depth=%d)\n", n, depth);
            __trap();
        }
        const int nx = cur ^ 1;
        // segments too long for one warp: the whole block, one after the other (only the first levels have any)
        for (int i = 0; i < nbig; ++i) {
            const Seg sg = S.bigs[cur][i];
            const int cut = block_rank_partition<uint16_t, kSortThreads>(S.keys, sg.f, sg.l, S.tabA + sg.f, S.tabB + sg.f, S.part);
            if (tid == 0) {
                push_segment(S, sg.f, cut, sg.d - 1, nx);
                push_segment(S, cut, sg.l, sg.d - 1, nx);
            }
        }
        // the others: one warp each
        for (int i = warp; i < cnt; i += kSortWarps) {
            const Seg sg = S.segs[cur][i];
            const int cut = warp_rank_partition(S, sg.f, sg.l);
            if (lane == 0) {
                push_segment(S, sg.f, cut, sg.d - 1, nx);
                push_segment(S, cut, sg.l, sg.d - 1, nx);
            }
        }
        __syncthreads();
        if (tid == 0) { S.nseg[cur] = 0; S.nbig[cur] = 0; }
        __syncthreads();
    }
    // one lane per remaining segment of 17..kLaneT keys; lanes of different warps first (lanes of one warp that run
    // different data-dependent loops serialise each other)
    for (int i0 = 0; i0 < S.nsmall; i0 += kSortThreads) {
        const int i = i0 + lane * kSortWarps + warp;
        if (i < S.nsmall) {
            const Seg sg = S.small[i];
            lane_partition_segment(S.keys, sg.f, sg.l, sg.d);
        }
    }
    __syncthreads();
    // __final_insertion_sort: every part now has <= 16 keys (or is sorted), parts are ordered among each other, and an
    // insertion sort is stable - so a key's final position is its rank in the window of +-15 positions around it
    {
        const uint32_t* kw = reinterpret_cast<const uint32_t*>(S.keys);
        constexpr int kPer = kS / kSortThreads;
        unsigned long long val[kPer];
        int dst[kPer];
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
            const int p = j * kSortThreads + tid;
            dst[j] = -1;
            val[j] = 0ull;
            if (p < n) {
                val[j] = S.keys[p];
                const uint32_t kp = (uint32_t)(val[j] >> 32);
                const int lo = p - 15 > 0 ? p - 15 : 0, hi = p + 15 < n - 1 ? p + 15 : n - 1;
                int c = lo;
                for (int q = lo; q < p; ++q) c += kw[2 * q + 1] <= kp;
                for (int q = p + 1; q <= hi; ++q) c += kw[2 * q + 1] < kp;
                dst[j] = c;
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kPer; ++j)
            if (dst[j] >= 0) S.keys[dst[j]] = val[j];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kSortThreads, 3) range_sort_kernel(PostBuffers pb) {
    extern __shared__ __align__(16) unsigned char sort_smem_raw[];
    SortSmem& S = *reinterpret_cast<SortSmem*>(sort_smem_raw);
    const int tid = threadIdx.x;
    for (;;) {
        __syncthreads();
        if (tid == 0) S.range_idx = atomicAdd(pb.cursors + 3, 1);
        __syncthreads();
        const int idx = S.range_idx;
        const int total = min(pb.cursors[2], pb.range_cap);
        if (idx >= total) return;
        const SortRange rg = pb.ranges[idx];
        unsigned long long* g = pb.pool + rg.off;
        for (int i = tid; i < rg.len; i += kSortThreads) S.keys[i] = g[i];
        __syncthreads();
        smem_level_sort(S, rg.len, rg.depth);
        for (int i = tid; i < rg.len; i += kSortThreads) g[i] = S.keys[i];
    }
}

// ------------------------------------------------------------------ greedy matching (pafprocess.cpp:98-124)
// The sorted list is walked in segments of kGreedySeg candidates: all threads first drop the candidates whose end points
// were already taken by earlier segments (ordered compaction into shared memory), then one warp runs the sequential rule
// over the survivors only, 32 per step, resolving conflicts inside a chunk in candidate order.  Identical to the
// sequential loop: a candidate rejected by the pre-filter would be rejected sequentially too, survivors are examined in
// order against the live used-sets.
__device__ int greedy_warp_chunked(const unsigned long long* keys, int n, int nb, uint32_t* used_a, uint32_t* used_b,
                                   int max_conn, int nc, int* conn_a, int* conn_b, float* conn_s) {
    const int lane = threadIdx.x & 31;
    for (int base = 0; base < n && nc < max_conn; base += 32) {
        const int i = base + lane;
        unsigned long long k = 0;
        int a = -1, b = -1;
        bool free_ = false;
        if (i < n) {
            k = keys[i];
            const uint32_t pair = (uint32_t)k;
            a = pair / nb;
            b = pair - a * nb;
            free_ = !((used_a[a >> 5] >> (a & 31)) & 1u) && !((used_b[b >> 5] >> (b & 31)) & 1u);
        }
        uint32_t active = __ballot_sync(0xffffffffu, free_);
        while (active && nc < max_conn) {
            const int leader = __ffs(active) - 1;
            const int la = __shfl_sync(0xffffffffu, a, leader), lb = __shfl_sync(0xffffffffu, b, leader);
            if (lane == leader) {
                used_a[a >> 5] |= 1u << (a & 31);
                used_b[b >> 5] |= 1u << (b & 31);
                conn_a[nc] = a;
                conn_b[nc] = b;
                conn_s[nc] = key_score(k);
            }
            ++nc;
            active &= ~__ballot_sync(0xffffffffu, a == la || b == lb);
        }
        __syncwarp();
    }
    return nc;
}

__global__ void __launch_bounds__(kGreedyThreads) limb_greedy_kernel(PostBuffers pb) {
    __shared__ unsigned long long seg[kGreedySeg];
    __shared__ uint32_t used_a[64], used_b[64];          // peak_cap <= 2048
    __shared__ int scan_scratch[kGreedyThreads / 32 + 1];
    __shared__ int s_nc;
    __shared__ int s_limb;
    const int tid = threadIdx.x;
    const int img = blockIdx.x;
    if (tid < 32) {
        const int l = limb_of_rank_warp(pb, img, blockIdx.y);
        if (tid == 0) s_limb = l;
    }
    __syncthreads();
    const int limb = s_limb;
    const LimbPlan pl = pb.lplan[img * kNumLimb + limb];
    int* out_cnt = pb.conn_cnt + img * kNumLimb + limb;
    const int n = pl.n, nb = pl.nb;
    if (n == 0) {
        if (tid == 0) *out_cnt = 0;
        return;
    }
    const unsigned long long* keys = pb.pool + pb.pool_cap / 2 + pl.region;
    const int max_conn = min(pl.na, pl.nb);
    const long o = ((long)img * kNumLimb + limb) * pb.peak_cap;
    for (int i = tid; i < 64; i += kGreedyThreads) { used_a[i] = 0; used_b[i] = 0; }
    if (tid == 0) s_nc = 0;
    __syncthreads();
    for (int s0 = 0; s0 < n; s0 += kGreedySeg) {
        if (s_nc >= max_conn) break;
        unsigned long long kk[kGreedyPer];
        int keep = 0, cnt = 0;
#pragma unroll
        for (int j = 0; j < kGreedyPer; ++j) {
            const int i = s0 + tid * kGreedyPer + j;
            kk[j] = 0;
            if (i < n) {
                kk[j] = keys[i];
                const uint32_t pair = (uint32_t)kk[j];
                const int a = pair / nb, b = pair - a * nb;
                if (!((used_a[a >> 5] >> (a & 31)) & 1u) && !((used_b[b >> 5] >> (b & 31)) & 1u)) { keep |= 1 << j; ++cnt; }
            }
        }
        int m;
        int off = block_exclusive_scan(cnt, &m, scan_scratch);
#pragma unroll
        for (int j = 0; j < kGreedyPer; ++j)
            if ((keep >> j) & 1) seg[off++] = kk[j];
        __syncthreads();
        if (tid < 32) {
            const int nc = greedy_warp_chunked(seg, m, nb, used_a, used_b, max_conn, s_nc, pb.conn_a + o, pb.conn_b + o,
                                               pb.conn_s + o);
            __syncwarp();
            if (tid == 0) s_nc = nc;
        }
        __syncthreads();
    }
    if (tid == 0) {
        *out_cnt = s_nc;
        if (pb.dbg) {
            atomicMax(pb.dbg + 3, (unsigned long long)n);
            atomicAdd(pb.dbg + 4, (unsigned long long)n);
        }
    }
}

}  // namespace

#define B2P_TRY(x)                        \
    do {                                  \
        cudaError_t e_ = (x);             \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

cudaError_t post_limbs(const PostBuffers& pb, int batch, const float* paf, long p_img, long p_ch, long p_y, long p_x,
                       int shift, int h_up, int lw, int lh, cudaStream_t s, const int2* dims) {
    if (batch > pb.batch_cap) return cudaErrorInvalidValue;
    if (pb.cand_smem_cap != kS) return cudaErrorInvalidValue;
    PafView pv{paf, p_ch, p_y, p_x, shift};
    limb_plan_kernel<<<1, 1024, 0, s>>>(pb, batch);
    B2P_TRY(cudaGetLastError());
    int in_smem = 0;
    size_t smem = 0;
    if (shift == 3 && (size_t)2 * lw * lh * sizeof(float) <= 96 * 1024) {
        in_smem = 1;
        smem = (size_t)2 * lw * lh * sizeof(float);
    }
    static DynSmemOptIn optin_score, optin_sort;
    B2P_TRY(optin_score.ensure(limb_score_kernel, smem));
    int dev = 0, sms = 148;
    B2P_TRY(cudaGetDevice(&dev));
    B2P_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    limb_score_kernel<<<sms * 6, kScoreThreads, smem, s>>>(pb, pv, p_img, h_up, lw, lh, in_smem, batch * kNumLimb, dims);
    B2P_TRY(cudaGetLastError());
    limb_gather_kernel<<<dim3(batch, kNumLimb), kGatherThreads, 0, s>>>(pb);
    B2P_TRY(cudaGetLastError());
    B2P_TRY(optin_sort.ensure(range_sort_kernel, sizeof(SortSmem)));
    const int sort_blocks = batch * kNumLimb < sms * 3 ? batch * kNumLimb : sms * 3;
    range_sort_kernel<<<sort_blocks, kSortThreads, sizeof(SortSmem), s>>>(pb);
    B2P_TRY(cudaGetLastError());
    limb_greedy_kernel<<<dim3(batch, kNumLimb), kGreedyThreads, 0, s>>>(pb);
    return cudaGetLastError();
}

// Test hook: exact std::sort of `n` host keys through the product's sorting stages (limb_gather_kernel's global-memory
// partitions + range_sort_kernel), as if they were the candidates of limb 0 of image 0.
cudaError_t post_debug_sort(const PostBuffers& pb, const unsigned long long* keys, int n, unsigned long long* out,
                            cudaStream_t s) {
    if (n < 1 || (long long)n + 2 > pb.pool_cap / 2) return cudaErrorInvalidValue;
    const int nchunks = (n + kChunkPairs - 1) / kChunkPairs;
    if (nchunks > pb.work_cap) return cudaErrorInvalidValue;
    std::vector<LimbPlan> plans(kNumLimb);
    for (auto& p : plans) p = LimbPlan{0, 0, 0, nchunks, 0, 0};
    plans[0] = LimbPlan{1, n, nchunks, 0, 0, 0};
    std::vector<int> cnt((size_t)nchunks * kSubPerChunk, 0), counts(kNumPart, 0);
    for (int sidx = 0; sidx * kSubPairs < n; ++sidx) cnt[sidx] = n - sidx * kSubPairs < kSubPairs ? n - sidx * kSubPairs : kSubPairs;
    counts[c_host_limb0[0]] = 1;
    counts[c_host_limb0[1]] = 1;
    const int cur[4] = {0, 0, 0, 0};
    B2P_TRY(cudaMemcpyAsync(pb.counts, counts.data(), kNumPart * sizeof(int), cudaMemcpyHostToDevice, s));
    B2P_TRY(cudaMemcpyAsync(pb.lplan, plans.data(), plans.size() * sizeof(LimbPlan), cudaMemcpyHostToDevice, s));
    B2P_TRY(cudaMemcpyAsync(pb.sub_cnt, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    B2P_TRY(cudaMemcpyAsync(pb.cursors, cur, sizeof(cur), cudaMemcpyHostToDevice, s));
    B2P_TRY(cudaMemcpyAsync(pb.pool, keys, (size_t)n * sizeof(unsigned long long), cudaMemcpyHostToDevice, s));
    limb_gather_kernel<<<dim3(1, kNumLimb), kGatherThreads, 0, s>>>(pb);
    B2P_TRY(cudaGetLastError());
    static DynSmemOptIn optin_sort;
    B2P_TRY(optin_sort.ensure(range_sort_kernel, sizeof(SortSmem)));
    range_sort_kernel<<<148 * 3, kSortThreads, sizeof(SortSmem), s>>>(pb);
    B2P_TRY(cudaGetLastError());
    B2P_TRY(cudaMemcpyAsync(out, pb.pool + pb.pool_cap / 2, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    return cudaStreamSynchronize(s);
}

}  // namespace b2p
