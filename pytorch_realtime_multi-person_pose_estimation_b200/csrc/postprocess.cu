// Fused post-processing kernel family for sm_100a: heat-map NMS + bicubic refinement, PAF line-integral scoring
// + greedy bipartite matching, person assembly.  See postprocess.cuh for the reference lines each kernel replaces.
// HBM-side this path touches 56 x h x w x 4 B per image once (18 heat + 38 PAF planes); it is latency bound, so
// the design goal is: everything stays on the device, one block per (image, part) / (image, limb) / image, warp
// shuffles for ordered compaction and arg-max, shared memory for the plane / candidate keys.
#include <cstdio>
#include <cstdlib>

#include "host_util.h"
#include "postprocess.cuh"

namespace b2p {

namespace {

__constant__ int c_limb_parts[kNumLimb][2] = B2P_LIMB_TABLES;

// OpenCV interpolateCubic (A = -0.75) for the 8 destination phases of an x8 up-sampling; exact float32 values
// (the 8 x 4 table is pinned against OpenCV in tests/test_oracle.py).  Phases 0-3 start at tap floor(src)-1 = X/8 - 2, phases 4-7 at X/8 - 1.
__constant__ float c_cubic[8][4] = {
    {-0x1.4acp-4f, 0x1.0568p-1f, 0x1.5918p-1f, -0x1.a94p-4f}, {-0x1.9c8p-5f, 0x1.5efp-2f, 0x1.a308p-1f, -0x1.c5cp-4f},
    {-0x1.5fp-6f, 0x1.7b2p-3f, 0x1.dbb8p-1f, -0x1.7c4p-4f},   {-0x1.68p-9f, 0x1.ad8p-5f, 0x1.fba8p-1f, -0x1.518p-5f},
    {-0x1.518p-5f, 0x1.fba8p-1f, 0x1.ad8p-5f, -0x1.68p-9f},   {-0x1.7c4p-4f, 0x1.dbb8p-1f, 0x1.7b2p-3f, -0x1.5fp-6f},
    {-0x1.c5cp-4f, 0x1.a308p-1f, 0x1.5efp-2f, -0x1.9c8p-5f},  {-0x1.a94p-4f, 0x1.5918p-1f, 0x1.0568p-1f, -0x1.4acp-4f}};

// the same table as compile-time constants (immediates of the unrolled vertical pass of the interior fast path)
__device__ constexpr float k_cubic[8][4] = {
    {-0x1.4acp-4f, 0x1.0568p-1f, 0x1.5918p-1f, -0x1.a94p-4f}, {-0x1.9c8p-5f, 0x1.5efp-2f, 0x1.a308p-1f, -0x1.c5cp-4f},
    {-0x1.5fp-6f, 0x1.7b2p-3f, 0x1.dbb8p-1f, -0x1.7c4p-4f},   {-0x1.68p-9f, 0x1.ad8p-5f, 0x1.fba8p-1f, -0x1.518p-5f},
    {-0x1.518p-5f, 0x1.fba8p-1f, 0x1.ad8p-5f, -0x1.68p-9f},   {-0x1.7c4p-4f, 0x1.dbb8p-1f, 0x1.7b2p-3f, -0x1.5fp-6f},
    {-0x1.c5cp-4f, 0x1.a308p-1f, 0x1.5efp-2f, -0x1.9c8p-5f},  {-0x1.a94p-4f, 0x1.5918p-1f, 0x1.0568p-1f, -0x1.4acp-4f}};

#ifndef B2P_PEAK_THREADS
#define B2P_PEAK_THREADS 256
#endif
constexpr int kPeakThreads = B2P_PEAK_THREADS;
constexpr int kAsmThreads = 128;
constexpr int kHorStride = 40;   // (2*2+1) * 8

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ------------------------------------------------------------------ peaks
// Interior fast path of the refinement: slots J0 .. J0+NS-1 of this lane (slot j = up-sampled column (lane + 32 j) % 40 of
// peak (lane + 32 j) / 40 of the group of four).  Horizontal pass into registers, vertical pass fully unrolled, per slot the
// maximum and the smallest row-major index attaining it.  Arithmetic and operation order: OpenCV's separable INTER_CUBIC.
template <int J0, int NS>
__device__ __forceinline__ void refine_interior_slots(const float* plane, int w, const int* px, const int* py,
                                                      const uint16_t* list, int ni, int grp, int lane, float* best,
                                                      int* bidx) {
    float hv[NS][5];
    int Xs[NS];
#pragma unroll
    for (int jj = 0; jj < NS; ++jj) {
        const int c = lane + 32 * (J0 + jj);               // 0..159: column X of peak g
        const int g = c >= 120 ? 3 : (c >= 80 ? 2 : (c >= 40 ? 1 : 0));
        const int X = c - 40 * g;
        const int gi = grp * 4 + g;
        Xs[jj] = X;
        best[J0 + jj] = -INFINITY;
        bidx[J0 + jj] = 0x7fffffff;
        if (gi < ni) {
            const int pk = list[gi];
            const int x = px[pk], y = py[pk];
            const int phase = X & 7;
            const int sx = (X >> 3) + (phase < 4 ? -2 : -1);
            const int t0 = clampi(sx, 0, 4), t1 = clampi(sx + 1, 0, 4), t2 = clampi(sx + 2, 0, 4), t3 = clampi(sx + 3, 0, 4);
            const float a0 = c_cubic[phase][0], a1 = c_cubic[phase][1], a2 = c_cubic[phase][2], a3 = c_cubic[phase][3];
            const float* p0 = plane + (y - 2) * w + (x - 2);
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                const float* prow = p0 + r * w;
                float v = __fmul_rn(prow[t0], a0);
                v = __fadd_rn(v, __fmul_rn(prow[t1], a1));
                v = __fadd_rn(v, __fmul_rn(prow[t2], a2));
                v = __fadd_rn(v, __fmul_rn(prow[t3], a3));
                hv[jj][r] = v;
            }
        } else {
#pragma unroll
            for (int r = 0; r < 5; ++r) hv[jj][r] = -INFINITY;     // never wins
        }
    }
#pragma unroll
    for (int Y = 0; Y < 40; ++Y) {
        const int phase = Y & 7;
        const int sy = (Y >> 3) + (phase < 4 ? -2 : -1);
        const int r0 = sy < 0 ? 0 : (sy > 4 ? 4 : sy), r1 = sy + 1 < 0 ? 0 : (sy + 1 > 4 ? 4 : sy + 1);
        const int r2 = sy + 2 < 0 ? 0 : (sy + 2 > 4 ? 4 : sy + 2), r3 = sy + 3 < 0 ? 0 : (sy + 3 > 4 ? 4 : sy + 3);
        const float b0 = k_cubic[phase][0], b1 = k_cubic[phase][1], b2 = k_cubic[phase][2], b3 = k_cubic[phase][3];
#pragma unroll
        for (int jj = 0; jj < NS; ++jj) {
            float v = __fmul_rn(hv[jj][r3], b3);
            v = __fadd_rn(__fmul_rn(hv[jj][r2], b2), v);
            v = __fadd_rn(__fmul_rn(hv[jj][r1], b1), v);
            v = __fadd_rn(__fmul_rn(hv[jj][r0], b0), v);
            if (v > best[J0 + jj]) { best[J0 + jj] = v; bidx[J0 + jj] = Y * 40 + Xs[jj]; }
        }
    }
}

__global__ void __launch_bounds__(kPeakThreads, 512 / kPeakThreads) peaks_kernel(PostBuffers pb, const float* __restrict__ heat, long h_img,
                                                             long h_ch, long h_y, long h_x, int h, int w, float thresh,
                                                             const int2* __restrict__ dims) {
    extern __shared__ float sm_f[];
    if (dims != nullptr) {      // ragged batch: this image's own map size (its plane sits top-left in the canvas strides)
        h = dims[blockIdx.y].x;
        w = dims[blockIdx.y].y;
    }
    float* plane = sm_f;                       // [h*w]
    float* hor_all = sm_f + h * w;             // [8 warps][5][40]
    __shared__ int warp_cnt[kPeakThreads / 32];
    __shared__ int s_base, s_ni, s_nb;
    __shared__ uint16_t s_list[2048];          // peak indices: interior ones from the front, border ones from the back
    const int part = blockIdx.x, img = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int hw = h * w;
    const float* src = heat + img * h_img + part * h_ch;
    for (int i = tid; i < hw; i += kPeakThreads) plane[i] = src[(long)(i / w) * h_y + (long)(i % w) * h_x];
    if (tid == 0) s_base = 0;
    __syncthreads();

    const int cap = pb.peak_cap;
    int* px = pb.peak_x + ((long)img * kNumPart + part) * cap;
    int* py = pb.peak_y + ((long)img * kNumPart + part) * cap;
    float* ps = pb.peak_s + ((long)img * kNumPart + part) * cap;

    // find_peaks: ordered (raster) compaction
    for (int start = 0; start < hw; start += kPeakThreads) {
        const int i = start + tid;
        bool flag = false;
        int x = 0, y = 0;
        if (i < hw) {
            y = i / w;
            x = i - y * w;
            const float v = plane[i];
            flag = (v > thresh) && (y == 0 || v >= plane[i - w]) && (y == h - 1 || v >= plane[i + w]) &&
                   (x == 0 || v >= plane[i - 1]) && (x == w - 1 || v >= plane[i + 1]);
        }
        const unsigned m = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) warp_cnt[warp] = __popc(m);
        __syncthreads();
        int pre = s_base, tot = 0;
        for (int k = 0; k < kPeakThreads / 32; ++k) {
            if (k < warp) pre += warp_cnt[k];
            tot += warp_cnt[k];
        }
        const int pos = pre + __popc(m & ((1u << lane) - 1u));
        if (flag && pos < cap) {
            px[pos] = x;
            py[pos] = y;
        }
        __syncthreads();
        if (tid == 0) s_base += tot;
        __syncthreads();
    }
    int n = s_base;
    if (n > cap) {
        if (tid == 0) atomicOr(&pb.status[img], 1);
        n = cap;
    }
    if (tid == 0) pb.counts[img * kNumPart + part] = n;

    // refinement: 5x5 window (clipped) -> x8 bicubic (separable, OpenCV's operation order) -> first arg-max.
    // Peaks whose window is not clipped (all but the two outermost rows / columns of the map) take the fast path: FOUR
    // peaks per warp - their 4 x 40 up-sampled columns fill the 32 lanes exactly five times - with the horizontal results in
    // registers and the vertical pass fully unrolled (tap rows and coefficients are compile-time constants).
    if (tid == 0) { s_ni = 0; s_nb = 0; }
    __syncthreads();
    for (int pk = tid; pk < n; pk += kPeakThreads) {
        const int x = px[pk], y = py[pk];
        const bool interior = x >= 2 && x + 2 <= w - 1 && y >= 2 && y + 2 <= h - 1;
        if (interior) s_list[atomicAdd(&s_ni, 1)] = (uint16_t)pk;
        else s_list[2047 - atomicAdd(&s_nb, 1)] = (uint16_t)pk;
    }
    __syncthreads();
    const int ni = s_ni, nbd = s_nb;
    for (int grp = warp; grp * 4 < ni; grp += kPeakThreads / 32) {
        float best[5];
        int bidx[5];
        refine_interior_slots<0, 3>(plane, w, px, py, s_list, ni, grp, lane, best, bidx);
        refine_interior_slots<3, 2>(plane, w, px, py, s_list, ni, grp, lane, best, bidx);
        // per peak: maximum value, smallest row-major index among equals (= first arg-max)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            float bv = -INFINITY;
            int bi = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const int c = lane + 32 * j;
                const int gj = c >= 120 ? 3 : (c >= 80 ? 2 : (c >= 40 ? 1 : 0));
                if (gj == g && (best[j] > bv || (best[j] == bv && bidx[j] < bi))) { bv = best[j]; bi = bidx[j]; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            const int gi = grp * 4 + g;
            if (lane == 0 && gi < ni) {
                const int pk = s_list[gi];
                const int x = px[pk], y = py[pk];
                const int ay = bi / 40, ax = bi - ay * 40;
                px[pk] = 8 * (x - 2) + ax;     // == (x+0.5)*8-0.5 + (ax - ((x-x_min+0.5)*8-0.5)), paf_to_pose.py:126-139
                py[pk] = 8 * (y - 2) + ay;
                ps[pk] = bv;
            }
        }
        __syncwarp();
    }
    // border peaks (clipped window): one warp per peak, rows walked
    float* hor = hor_all + warp * 5 * kHorStride;
    for (int bi_ = warp; bi_ < nbd; bi_ += kPeakThreads / 32) {
        const int pk = s_list[2047 - bi_];
        const int x = px[pk], y = py[pk];
        const int x_min = max(0, x - 2), x_max = min(w - 1, x + 2);
        const int y_min = max(0, y - 2), y_max = min(h - 1, y + 2);
        const int pw = x_max - x_min + 1, ph = y_max - y_min + 1;
        const int W8 = pw * 8, H8 = ph * 8;
        __syncwarp();
        // horizontal pass: lanes own columns X = lane and lane + 32 (W8 <= 40), rows are walked - no divisions
        for (int xi = 0; xi < 2; ++xi) {
            const int X = lane + 32 * xi;
            if (X < W8) {
                const int phase = X & 7;
                const int sx = (X >> 3) + (phase < 4 ? -2 : -1);
                const int t0 = clampi(sx, 0, pw - 1), t1 = clampi(sx + 1, 0, pw - 1);
                const int t2 = clampi(sx + 2, 0, pw - 1), t3 = clampi(sx + 3, 0, pw - 1);
                const float a0 = c_cubic[phase][0], a1 = c_cubic[phase][1], a2 = c_cubic[phase][2], a3 = c_cubic[phase][3];
                for (int r = 0; r < ph; ++r) {
                    const float* prow = plane + (y_min + r) * w + x_min;
                    float v = __fmul_rn(prow[t0], a0);
                    v = __fadd_rn(v, __fmul_rn(prow[t1], a1));
                    v = __fadd_rn(v, __fmul_rn(prow[t2], a2));
                    v = __fadd_rn(v, __fmul_rn(prow[t3], a3));
                    hor[r * kHorStride + X] = v;
                }
            }
        }
        __syncwarp();
        // vertical pass + first arg-max (row-major index Y*W8 + X; each lane visits its indices in increasing order)
        float best = -INFINITY;
        int best_idx = 0x7fffffff;
        for (int Y = 0; Y < H8; ++Y) {
            const int phase = Y & 7;
            const int sy = (Y >> 3) + (phase < 4 ? -2 : -1);
            const float* h0 = hor + clampi(sy, 0, ph - 1) * kHorStride;
            const float* h1 = hor + clampi(sy + 1, 0, ph - 1) * kHorStride;
            const float* h2 = hor + clampi(sy + 2, 0, ph - 1) * kHorStride;
            const float* h3 = hor + clampi(sy + 3, 0, ph - 1) * kHorStride;
            const float b0 = c_cubic[phase][0], b1 = c_cubic[phase][1], b2 = c_cubic[phase][2], b3 = c_cubic[phase][3];
#pragma unroll
            for (int xi = 0; xi < 2; ++xi) {
                const int X = lane + 32 * xi;
                if (X < W8) {
                    float v = __fmul_rn(h3[X], b3);
                    v = __fadd_rn(__fmul_rn(h2[X], b2), v);
                    v = __fadd_rn(__fmul_rn(h1[X], b1), v);
                    v = __fadd_rn(__fmul_rn(h0[X], b0), v);
                    if (v > best) { best = v; best_idx = Y * W8 + X; }
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
            if (ov > best || (ov == best && oi < best_idx)) { best = ov; best_idx = oi; }
        }
        if (lane == 0) {
            const int ay = best_idx / W8, ax = best_idx - ay * W8;
            px[pk] = 8 * x_min + ax;     // == (x+0.5)*8-0.5 + (ax - ((x-x_min+0.5)*8-0.5)), paf_to_pose.py:126-139
            py[pk] = 8 * y_min + ay;
            ps[pk] = best;
        }
    }
}

// ------------------------------------------------------------------ assembly
__global__ void __launch_bounds__(kAsmThreads) assemble_kernel(PostBuffers pb) {
    extern __shared__ int sm_kept[];     // [human_cap]
    __shared__ int part_base[kNumPart + 1];
    __shared__ int s_nh, s_nrows;
    const int img = blockIdx.x, tid = threadIdx.x;
    const int cap = pb.peak_cap;
    const int id_cap = kNumPart * cap;
    if (tid == 0) {
        part_base[0] = 0;
        for (int p = 0; p < kNumPart; ++p) part_base[p + 1] = part_base[p] + pb.counts[img * kNumPart + p];
    }
    __syncthreads();
    float* id_score = pb.id_score + (long)img * id_cap;
    int* id_xy = pb.id_xy + (long)img * id_cap * 2;
    uint8_t* list_n = pb.list_n + (long)img * id_cap;
    uint8_t* alive = pb.alive + (long)img * pb.row_cap;
    const int total = part_base[kNumPart];
    for (int p = 0; p < kNumPart; ++p) {
        const int n = part_base[p + 1] - part_base[p];
        const long src = ((long)img * kNumPart + p) * cap;
        for (int i = tid; i < n; i += kAsmThreads) {
            const int id = part_base[p] + i;
            id_score[id] = pb.peak_s[src + i];
            id_xy[2 * id] = pb.peak_x[src + i];
            id_xy[2 * id + 1] = pb.peak_y[src + i];
        }
    }
    for (int i = tid; i < total; i += kAsmThreads) list_n[i] = 0;
    for (int i = tid; i < pb.row_cap; i += kAsmThreads) alive[i] = 0;
    __syncthreads();

    float* rows = pb.rows + (long)img * pb.row_cap * kRowFloats;
    __shared__ Assembler s_as;
    if (tid == 0) {
        s_as.rows = rows;
        s_as.alive = alive;
        s_as.lists = pb.lists + (long)img * id_cap * kListCap;
        s_as.list_n = list_n;
        s_as.part_base = part_base;
        s_as.peak_score = id_score;
        s_as.row_cap = pb.row_cap;
        s_as.nrows = 0;
        s_as.degraded = 0;
        s_as.overflow = 0;
    }
    __syncthreads();
    // The assembly itself is inherently sequential (pafprocess.cpp:127-185) and latency bound: one thread walks the
    // connections.  Before each limb all threads pull the lines that walk will touch (row lists of both end points,
    // the listed rows, peak scores) into L1 so the sequential part runs on L1 hits.
    for (int l = 0; l < kNumLimb; ++l) {
        const int p1 = c_limb_parts[l][0], p2 = c_limb_parts[l][1];
        const int nc = pb.conn_cnt[img * kNumLimb + l];
        const long o = ((long)img * kNumLimb + l) * cap;
        for (int c = tid; c < nc; c += kAsmThreads) {
            const int ids[2] = {part_base[p1] + pb.conn_a[o + c], part_base[p2] + pb.conn_b[o + c]};
            prefetch_l1(pb.conn_s + o + c);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int id = ids[e];
                prefetch_l1(id_score + id);
                const int n = s_as.list_n[id];
                for (int i = 0; i < n && i < kListCap; ++i) {
                    const int r = s_as.lists[id * kListCap + i];
                    prefetch_l1(rows + (long)r * kRowFloats);
                    prefetch_l1(rows + (long)r * kRowFloats + kRowFloats - 1);
                    prefetch_l1(alive + r);
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            for (int c = 0; c < nc; ++c)
                s_as.add_connection(l, p1, p2, part_base[p1] + pb.conn_a[o + c], part_base[p2] + pb.conn_b[o + c],
                                    pb.conn_s[o + c]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        Assembler& as = s_as;
        int nh = 0, st = 0;
        for (int r = 0; r < as.nrows; ++r)
            if (as.keep(r)) {
                if (nh < pb.human_cap) sm_kept[nh++] = r;
                else st |= 8;
            }
        if (as.overflow) st |= 4;
        if (as.degraded) st |= 16;
        // this block is the last writer of the image's status word: fold it into the sticky accumulator as well
        const int st_all = (st ? atomicOr(&pb.status[img], st) : pb.status[img]) | st;
        if (st_all) atomicOr(&pb.status_acc[img], st_all);
        s_nh = nh;
        s_nrows = as.nrows;
        pb.n_humans[img] = nh;
    }
    __syncthreads();
    const int nh = s_nh;
    float* out = (pb.humans_out ? pb.humans_out : pb.humans) + (long)img * pb.human_cap * kHumanFloats;
    for (int e = tid; e < nh * kHumanFloats; e += kAsmThreads) {
        const int hi = e / kHumanFloats, f = e - hi * kHumanFloats;
        const float* row = rows + sm_kept[hi] * kRowFloats;
        float v;
        if (f == 0) v = __fdiv_rn(row[18], row[19]);     // get_score, pafprocess.cpp:204-206
        else {
            const int p = (f - 1) >> 2, k = (f - 1) & 3;
            const int cid = (int)row[p];                  // get_part_cid truncation, pafprocess.cpp:200-202
            if (cid < 0) v = (k == 3) ? -1.f : 0.f;
            else v = k == 0 ? (float)id_xy[2 * cid] : k == 1 ? (float)id_xy[2 * cid + 1] : k == 2 ? id_score[cid] : (float)cid;
        }
        out[e] = v;
    }
}

}  // namespace

#define B2P_TRY(x)                        \
    do {                                  \
        cudaError_t e_ = (x);             \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

cudaError_t post_alloc(PostBuffers& pb, int batch_cap, int peak_cap, int human_cap, long pool_cap) {
    memset(&pb, 0, sizeof(pb));
    if (peak_cap > 2048 || peak_cap < 1) return cudaErrorInvalidValue;
    pb.batch_cap = batch_cap;
    pb.peak_cap = peak_cap;
    pb.human_cap = human_cap;
    pb.cand_smem_cap = kLimbSmemRange;
    pb.pool_cap = pool_cap;
    pb.row_cap = 4 * peak_cap;
    const long B = batch_cap;
    B2P_TRY(cudaMalloc(&pb.counts, B * kNumPart * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.peak_x, B * kNumPart * peak_cap * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.peak_y, B * kNumPart * peak_cap * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.peak_s, B * kNumPart * peak_cap * sizeof(float)));
    B2P_TRY(cudaMalloc(&pb.conn_cnt, B * kNumLimb * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.conn_a, B * kNumLimb * peak_cap * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.conn_b, B * kNumLimb * peak_cap * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.conn_s, B * kNumLimb * peak_cap * sizeof(float)));
    B2P_TRY(cudaMalloc(&pb.rows, B * pb.row_cap * kRowFloats * sizeof(float)));
    B2P_TRY(cudaMalloc(&pb.alive, B * pb.row_cap));
    B2P_TRY(cudaMalloc(&pb.lists, B * kNumPart * peak_cap * kListCap * sizeof(int32_t)));
    B2P_TRY(cudaMalloc(&pb.list_n, B * kNumPart * peak_cap));
    B2P_TRY(cudaMalloc(&pb.id_score, B * kNumPart * peak_cap * sizeof(float)));
    B2P_TRY(cudaMalloc(&pb.id_xy, B * kNumPart * peak_cap * 2 * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.pool, pool_cap * sizeof(unsigned long long)));
    // scoring work items: sum over limbs of ceil(pairs / 2048) <= half pool / 2048 + limbs; sort ranges: one per limb plus
    // two per global-memory partition (a partition of > 4096 keys rarely leaves a child below 512)
    pb.work_cap = (int)(pool_cap / 2 / kLimbChunkPairs + B * kNumLimb + 1);
    pb.range_cap = (int)(pool_cap / 2 / 512 + B * kNumLimb * 2);
    B2P_TRY(cudaMalloc(&pb.lplan, B * kNumLimb * sizeof(LimbPlan)));
    B2P_TRY(cudaMalloc(&pb.sub_cnt, (size_t)pb.work_cap * 8 * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.sub_off, (size_t)pb.work_cap * 8 * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.cursors, 4 * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.ranges, (size_t)pb.range_cap * sizeof(SortRange)));
    B2P_TRY(cudaMalloc(&pb.n_humans, B * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.humans, B * human_cap * kHumanFloats * sizeof(float)));
    B2P_TRY(cudaMalloc(&pb.status, B * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.status_acc, B * sizeof(int)));
    B2P_TRY(cudaMemset(pb.status_acc, 0, B * sizeof(int)));
    B2P_TRY(cudaMalloc(&pb.dbg, 16 * sizeof(unsigned long long)));
    B2P_TRY(cudaMemset(pb.dbg, 0, 16 * sizeof(unsigned long long)));
    B2P_TRY(cudaMemset(pb.status, 0, B * sizeof(int)));
    B2P_TRY(cudaMemset(pb.counts, 0, B * kNumPart * sizeof(int)));
    return cudaSuccess;
}

void post_free(PostBuffers& pb) {
    void* ptrs[] = {pb.counts, pb.peak_x, pb.peak_y, pb.peak_s,  pb.conn_cnt, pb.conn_a,      pb.conn_b,
                    pb.conn_s, pb.rows,   pb.alive,  pb.lists,   pb.list_n,   pb.id_score,    pb.id_xy,
                    pb.pool,   pb.lplan, pb.sub_cnt, pb.sub_off, pb.cursors, pb.ranges, pb.n_humans, pb.humans, pb.status, pb.status_acc, pb.dbg};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    memset(&pb, 0, sizeof(pb));
}

cudaError_t post_peaks(const PostBuffers& pb, int batch, const float* heat, long h_img, long h_ch, long h_y, long h_x,
                       int h, int w, float thresh, cudaStream_t s, const int2* dims) {
    if (batch > pb.batch_cap) return cudaErrorInvalidValue;
    const size_t smem = ((size_t)h * w + (kPeakThreads / 32) * 5 * kHorStride) * sizeof(float);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    static DynSmemOptIn optin;
    B2P_TRY(optin.ensure(peaks_kernel, smem));
    B2P_TRY(cudaMemsetAsync(pb.status, 0, batch * sizeof(int), s));
    peaks_kernel<<<dim3(kNumPart, batch), kPeakThreads, smem, s>>>(pb, heat, h_img, h_ch, h_y, h_x, h, w, thresh, dims);
    return cudaGetLastError();
}

cudaError_t post_assemble(const PostBuffers& pb, int batch, cudaStream_t s) {
    if (batch > pb.batch_cap) return cudaErrorInvalidValue;
    assemble_kernel<<<batch, kAsmThreads, pb.human_cap * sizeof(int), s>>>(pb);
    return cudaGetLastError();
}

}  // namespace b2p
