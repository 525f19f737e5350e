// Fused post-processing kernel family (device-resident replacement of NMS + pafprocess):
//   peaks_kernel    : find_peaks + NMS refinement      /root/reference/lib/utils/paf_to_pose.py:25-38, 67-145
//   limbs.cu family : candidate scoring + std::sort + greedy match  /root/reference/lib/pafprocess/pafprocess.cpp:47-125
//   assemble_kernel : person assembly + prune + getters /root/reference/lib/pafprocess/pafprocess.cpp:127-218
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "post_core.h"

namespace b2p {

constexpr int kLimbChunkPairs = 2048;    // (a, b) pairs per scoring work item
#ifndef B2P_LIMB_SMEM_RANGE
#define B2P_LIMB_SMEM_RANGE 4096
#endif
constexpr int kLimbSmemRange = B2P_LIMB_SMEM_RANGE;     // candidate keys sorted per shared-memory range
#ifndef B2P_LANE_SORT_KEYS
#define B2P_LANE_SORT_KEYS 64            // segments of at most this many keys are finished by one lane each (limbs.cu)
#endif

struct LimbPlan {         // per (image, limb), written by limb_plan_kernel
    int na, nb;           // peaks of the two parts (0 / 0: no pairs, or the candidate pool is exhausted)
    int nchunks;          // scoring work items of this limb
    int work0;            // index of its first work item
    int n;                // candidates that passed both criteria (limb_gather_kernel)
    long long region;     // first slot of the limb's na*nb + 2 slots in pool A (warp slots / partition scratch) and pool B
};
struct SortRange {        // one shared-memory sort job: pool[off, off + len), introsort depth budget
    long long off;
    int len, depth;
};

struct PostBuffers {
    // capacities
    int batch_cap, peak_cap /*per part*/, human_cap, cand_smem_cap;
    long pool_cap;   // candidate key pool (entries) for limbs whose candidate list does not fit shared memory
    // peaks (per image, per part)
    int* counts;        // [B][18]
    int* peak_x;        // [B][18][peak_cap]  full-resolution integer coordinates
    int* peak_y;
    float* peak_s;      // refined score
    // connections (per image, per limb)
    int* conn_cnt;      // [B][19]
    int* conn_a;        // [B][19][peak_cap]
    int* conn_b;
    float* conn_s;
    // assembly scratch
    float* rows;        // [B][row_cap][20]
    uint8_t* alive;     // [B][row_cap]
    int32_t* lists;     // [B][18*peak_cap][kListCap]
    uint8_t* list_n;    // [B][18*peak_cap]
    float* id_score;    // [B][18*peak_cap]   peak score by id
    int* id_xy;         // [B][18*peak_cap][2]
    int row_cap;
    // candidate keys: pool[0, pool_cap/2) = pool A, pool[pool_cap/2, pool_cap) = pool B (limbs.cu)
    unsigned long long* pool;
    LimbPlan* lplan;    // [B][19]
    int* sub_cnt;       // [work_cap][8] candidates per warp slot of a scoring work item
    int* sub_off;       // [work_cap][8] their offsets in the limb's contiguous list
    int* cursors;       // [4] scoring work cursor, scoring work items, ranges emitted, range cursor
    SortRange* ranges;  // [range_cap]
    int work_cap, range_cap;
    // results
    int* n_humans;      // [B]
    float* humans;      // [B][human_cap][1 + 18*4]: score, then per part (x, y, peak score, cid or -1)
    float* humans_out;  // where assemble_kernel writes the rows: `humans`, or (set per run) a pinned HOST buffer of the same
                        // geometry - the kernel then exports exactly the used rows over PCIe and no copy of the full-capacity
                        // buffer follows
    unsigned long long* dbg;   // [16] diagnostics: max cycles per limbs_kernel phase, candidate counts
    int* status_acc;    // [B] OR of `status` over every run since the last reset (b200pose_post_status_accum)
    int* status;        // [B] bit0 peak overflow, bit1 candidate pool overflow, bit2 row overflow, bit3 human overflow,
                        //     bit4 assembler used the slow scan, bit8.. number of limbs that needed the tie-exact sort
};

constexpr int kHumanFloats = 1 + 18 * 4;

cudaError_t post_alloc(PostBuffers& pb, int batch_cap, int peak_cap, int human_cap, long pool_cap);
void post_free(PostBuffers& pb);

// heat: fp32, value(img, part, y, x) = heat[img*h_img + part*h_ch + y*h_y + x*h_x]; low-res (h x w).
// dims (ragged batches, device array or null): image i's own low-res (h, w), its maps top-left in the h x w canvas.
cudaError_t post_peaks(const PostBuffers& pb, int batch, const float* heat, long h_img, long h_ch, long h_y, long h_x,
                       int h, int w, float thresh, cudaStream_t s, const int2* dims = nullptr);
// paf: fp32 view per image: base + img*p_img, strides (p_ch, p_y, p_x), shift (3: low-res, 0: already upsampled).
// dims (ragged batches): image i's own low-res (h, w); its length criterion uses h_up = 8 h instead of h_up.
cudaError_t post_limbs(const PostBuffers& pb, int batch, const float* paf, long p_img, long p_ch, long p_y,
                                    long p_x, int shift, int h_up, int lw, int lh, cudaStream_t s,
                                    const int2* dims = nullptr);
// Test hook (limbs.cu): exact std::sort of n host keys through the global-memory partition + shared-memory range kernels.
cudaError_t post_debug_sort(const PostBuffers& pb, const unsigned long long* keys, int n, unsigned long long* out,
                            cudaStream_t s);
// Person assembly of the connections post_limbs() left in `pb`.  Small footprint (128 threads, human_cap*4 B smem per
// image): it can run on a second stream next to the convolutions of the following batch.
cudaError_t post_assemble(const PostBuffers& pb, int batch, cudaStream_t s);
// lw x lh: dimensions of the low-resolution PAF planes (used to stage them in shared memory when shift == 3)

}  // namespace b2p
