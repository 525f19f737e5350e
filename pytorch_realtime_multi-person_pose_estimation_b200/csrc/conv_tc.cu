// tcgen05 "halo-patch" implicit-GEMM convolution for sm_100a (B200).
//
// Computes, for every conv of the rtpose VGG19 net with Cin >= 64
// (/root/reference/lib/network/rtpose_vgg.py:69-127), out = act(conv_kxk(in) + bias) with optional fused
// MaxPool2d(2,2) and "concat by construction" (the epilogue writes straight into a channel slice of the
// next layer's NHWC buffer, replacing torch.cat at rtpose_vgg.py:165,171,177,183,189).
//
// Mapping to the hardware (see DESIGN.md "conv_tc"):
//   * A CTA owns a 16x16 block of output pixels = two UMMA M=128 sub-tiles of 8 (w) x 16 (h) pixels.
//   * For each 64-channel block of the input, ONE TMA 4-D tile load brings the (16+k-1) x 24 pixel halo patch
//     (NHWC bf16, 128 B per pixel, SWIZZLE_128B, out-of-image pixels zero-filled by TMA = conv padding) into
//     shared memory.  Every one of the k*k filter taps then reads its shifted 8x16 window of that SAME patch
//     directly through the UMMA shared-memory descriptor (start address = patch + (dy*24+dx)*128 B,
//     8-row groups 24*128 B apart), so the activation tile is fetched from L2 once instead of k*k times.
//   * TMA 3-D loads bring the [n_tile x 64] weight slices (K-major, SWIZZLE_128B) of `tps` consecutive taps per stage into a
//     48 KB ring (tps: as many taps as still leave three stages - the per-stage barrier / issue cost is ~360 clk).
//   * One elected thread issues tcgen05.mma (kind::f16, bf16 x bf16 -> fp32) into TMEM; two accumulator sets
//     (2 x 256 columns) let the epilogue of tile i overlap the MMAs of tile i+1.
//   * Eight epilogue warps (two per TMEM lane quarter) read TMEM (tcgen05.ld 32x32b), add bias, ReLU, optionally 2x2 max-pool through warp
//     shuffles, convert to bf16 and store NHWC; the stage heads additionally emit the fp32 NCHW outputs.
//   * Persistent grid (one CTA per SM), static round-robin tile schedule.
//   * CTA-PAIR mode (a.pair, template kPair): the grid is launched as clusters of two CTAs on the two SMs of a TPC and the
//     MMAs are tcgen05.mma.cta_group::2 with M = 256: each CTA keeps its OWN 16x16 pixel tile (own halo patch, own TMEM
//     accumulators, own epilogue) but the two tiles share the weight slice, so each CTA loads and holds only HALF of the
//     N rows of B.  Per MMA a CTA's shared memory is read for A (4 KB) + B/2 (2 KB) instead of 8 KB, and the per-tap weight
//     TMA is 8 KB instead of 16 KB: the single-CTA kernel sits at the 128 B/clk shared-memory limit with N = 128
//     (68 % tensor-pipe activity measured), the pair does not.  Only the leader CTA issues MMAs; TMA loads of both CTAs
//     credit the leader's "full" barriers, tcgen05.commit multicasts the "empty" / "accumulator full" arrivals to both.
#include <cstdio>

#include "conv_tc.cuh"
#include "host_util.h"
#include "ptx.cuh"

namespace b2p {

#ifdef B2P_CONV_TIMELINE
__device__ unsigned long long g_conv_timeline[64 * kTlSlots];
#define B2P_TL(slot) do { if (blockIdx.x < 64) g_conv_timeline[blockIdx.x * kTlSlots + (slot)] = clock64(); } while (0)
#else
#define B2P_TL(slot) do { } while (0)
#endif

namespace {

struct TileCoord {
    int n, y0, x0, g, nt;
    bool valid;      // pair mode: the odd CTA of the last pair may have no pixel tile (it then computes on zeros)
};

// Single-CTA mode: work item t = one (pixel tile, group, n-tile).  Pair mode: work item t = one (pair of consecutive
// pixel tiles, group, n-tile); the CTA of rank r takes pixel tile 2 * pair + r.  (n-tile, group) vary fastest so that CTAs
// running at the same time read the same activation patches from L2.
template <bool kPair>
__device__ __forceinline__ TileCoord decode_tile(int t, int n_tiles, int groups, int tiles_x, int tiles_y, int n_img,
                                                 int rank, int tile_w) {
    TileCoord c;
    c.nt = t % n_tiles;
    t /= n_tiles;
    c.g = t % groups;
    t /= groups;
    c.valid = true;
    if (kPair) {
        const int pix_tiles = n_img * tiles_y * tiles_x;
        t = 2 * t + rank;
        if (t >= pix_tiles) { t = pix_tiles; c.valid = false; }     // -> n = n_img: TMA zero-fills, nothing is stored
    }
    c.x0 = (t % tiles_x) * tile_w;
    t /= tiles_x;
    c.y0 = (t % tiles_y) * kTileH;
    c.n = t / tiles_y;
    return c;
}

// Ragged batches (a.ext): input-resolution pixel (y, x) of image n lies outside that image's extent.  Extents are multiples
// of 8 and pooled layers have ext_shift <= 2, so a 2x2 pooling window lies wholly inside or wholly outside.
__device__ __forceinline__ bool outside_extent(const ConvTcArgs& a, int n, int y, int x) {
    if (a.ext == nullptr) return false;
    const int2 e = __ldg(a.ext + n);
    return y >= (e.x >> a.ext_shift) || x >= (e.y >> a.ext_shift);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

template <bool kPair, bool kChunk>
__device__ __forceinline__ void conv_tc_body(const ConvTcArgs& a) {
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B operands need 1024 B alignment.
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* patch_smem = smem;
    uint8_t* b_smem = smem + kNumPatchStages * kPatchBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_smem + kNumBStages * kBStageBytes);
    uint64_t* patch_full = bars;                          // [2]
    uint64_t* patch_empty = bars + kNumPatchStages;       // [2]
    uint64_t* b_full = bars + 2 * kNumPatchStages;        // [kMaxBStages]
    uint64_t* b_empty = b_full + kMaxBStages;             // [kMaxBStages]
    uint64_t* acc_full = b_empty + kMaxBStages;           // [2]
    uint64_t* acc_empty = acc_full + 2;                   // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) B2P_TL(0);

    // narrow mode (small batches): the CTA tile is ONE 8 x 16 sub-tile - twice the CTAs, half the MMA work each; the patch
    // box keeps its 24-pixel pitch (the right part is loaded and not read)
    const int nsub = a.narrow ? 1 : 2;
    const int tile_w = 8 * nsub;
    const int tiles_x = (a.W + tile_w - 1) / tile_w;
    const int tiles_y = (a.H + kTileH - 1) / kTileH;
    const int rank = kPair ? (int)cluster_ctarank() : 0;
    // work items of this CTA (pair mode: of this pair): first, stride, total
    const int pix_items = kPair ? (a.n_img * tiles_y * tiles_x + 1) / 2 : a.n_img * tiles_y * tiles_x;
    const int total_tiles = pix_items * a.groups * a.n_tiles;
    const int work0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int wstep = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int taps = a.ksize * a.ksize;
    const int pad = a.ksize >> 1;
    const uint32_t patch_tx = kPatchPitch * (kTileH + a.ksize - 1) * 128;
    const int b_rows = kPair ? a.n_tile / 2 : a.n_tile;      // weight rows this CTA loads per tap
    const uint32_t b_tx = b_rows * 128;
    // The weight ring is cut into stages of `tps` consecutive taps (a.tps, chosen with the tensor map's box): per stage the
    // producer pays a barrier wait + expect_tx + TMA issue and the MMA warp a barrier wait + elect + commit - about 360 clk,
    // which bounded the small-batch plans (64 clk of tensor work per tap with 32-wide n-tiles; timeline build, batch 1).
    const int tps = a.tps;
    const uint32_t b_stride = b_tx * tps;                    // multiples of 1024 B (n_tile % 16 == 0; pair: n_tile % 32 == 0)
    const uint32_t nb_fit = (kNumBStages * kBStageBytes) / b_stride;
    const uint32_t nb = nb_fit < (uint32_t)kMaxBStages ? nb_fit : (uint32_t)kMaxBStages;
    const int nterms = a.split ? 3 : 1;   // split mode: A_hi*W_hi, A_hi*W_lo, A_lo*W_hi per K block

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&a.tm_in);
        tma_prefetch_desc(&a.tm_w);
        if (a.split) tma_prefetch_desc(&a.tm_in_lo);
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < kNumPatchStages; ++i) {
                mbar_init(&patch_full[i], 1);
                mbar_init(&patch_empty[i], 1);
            }
            for (uint32_t i = 0; i < nb; ++i) {
                mbar_init(&b_full[i], 1);
                mbar_init(&b_empty[i], 1);
            }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&acc_full[i], 1);
                mbar_init(&acc_empty[i], kPair ? 16 : 8);   // one arrive per epilogue warp (of both CTAs of a pair)
            }
            fence_mbar_init();
        }
        __syncwarp();
        if (kPair) tmem_alloc_pair(tmem_slot, 512);
        else tmem_alloc(tmem_slot, 512);
    }
    tc_fence_before();
    if (kPair) cluster_sync_all();      // the peer's barriers are initialised before anything arrives on them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) B2P_TL(1);
    // PDL (no-ops unless the launch carries the attribute): let the next layer start its prologue now; everything that reads
    // or writes activations first waits for the previous layer's grid to complete (weights / bias are constants).
    pdl_launch_dependents();

    if (warp == 0) {
        // =========================== TMA producer: activation halo patches ===========================
        if (lane == 0) {
            pdl_wait();
            uint32_t pi = 0, pph = 0;
            for (int t = work0; t < total_tiles; t += wstep) {
                const TileCoord tc = decode_tile<kPair>(t, a.n_tiles, a.groups, tiles_x, tiles_y, a.n_img, rank, tile_w);
                const int ch0 = a.in_ch_base + tc.g * a.in_ch_group_stride;
                for (int cb = 0; cb < a.cin_blocks; ++cb) {
                    for (int plane = 0; plane <= a.split; ++plane) {     // hi plane, then (split mode) the residual plane
                        mbar_wait(&patch_empty[pi], pph ^ 1, 1);
                        if (kPair) {      // both patches of the pair complete on the leader's barrier
                            if (rank == 0) mbar_expect_tx(&patch_full[pi], 2 * patch_tx);
                            tma_load_4d_pair(patch_smem + pi * kPatchBytes, plane ? &a.tm_in_lo : &a.tm_in, &patch_full[pi],
                                             ch0 + cb * 64, tc.x0 - pad, tc.y0 - pad, tc.n);
                        } else {
                            mbar_expect_tx(&patch_full[pi], patch_tx);
                            tma_load_4d(patch_smem + pi * kPatchBytes, plane ? &a.tm_in_lo : &a.tm_in, &patch_full[pi],
                                        ch0 + cb * 64, tc.x0 - pad, tc.y0 - pad, tc.n);
                        }
                        if (++pi == kNumPatchStages) { pi = 0; pph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 6) {
        // =========================== TMA producer: weight slices ===========================
        if (lane == 0) {
            uint32_t bi = 0, bph = 0;
            for (int t = work0; t < total_tiles; t += wstep) {
                const TileCoord tc = decode_tile<kPair>(t, a.n_tiles, a.groups, tiles_x, tiles_y, a.n_img, rank, tile_w);
                const int wrow = (tc.g * a.n_tiles + tc.nt) * a.n_tile + rank * b_rows;   // pair: this CTA's half of N
                for (int cb = 0; cb < a.cin_blocks; ++cb) {
                    for (int term = 0; term < nterms; ++term) {          // W_hi, (split) W_lo, W_hi
                        const int wsel = (term == 1) ? taps : 0;
                        for (int tap0 = 0; tap0 < taps; tap0 += tps) {       // (the last box of a block may run past `taps`:
                            mbar_wait(&b_empty[bi], bph ^ 1, 2);             //  those slices are loaded and not read)
                            if (kPair) {
                                if (rank == 0) mbar_expect_tx(&b_full[bi], 2 * b_stride);
                                tma_load_3d_pair(b_smem + bi * b_stride, &a.tm_w, &b_full[bi], cb * 64, wrow, wsel + tap0);
                            } else {
                                mbar_expect_tx(&b_full[bi], b_stride);
                                tma_load_3d(b_smem + bi * b_stride, &a.tm_w, &b_full[bi], cb * 64, wrow, wsel + tap0);
                            }
                            if (++bi == nb) { bi = 0; bph ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1 && rank == 0) {
        // =========================== MMA issuer (pair mode: the leader CTA only) ===========================
        // The whole warp walks the loops (warp-uniform control flow, uniform registers for the descriptors); one
        // elected lane issues the tcgen05 instructions.  A divergent `if (lane == 0)` around the loop makes ptxas wrap
        // every UTCHMMA in an ELECT/BRA.U.ANY uniformisation loop (~2x the issue cost).
        {
            const uint32_t idesc = kPair ? make_idesc_bf16_m256(a.n_tile) : make_idesc_bf16_m128(a.n_tile);
            // Descriptors are built incrementally: the high words are loop invariants, the low word (address >> 4)
            // only receives small adds per tap / sub-tile / K step.
            const uint64_t adesc_hi = make_sdesc_sw128(0, kPatchPitch * 128, 0);
            const uint64_t bdesc_hi = make_sdesc_sw128(0, 1024, 0);
            const uint32_t patch_lo0 = (smem_u32(patch_smem) & 0x3FFFFu) >> 4;
            const uint32_t b_lo0 = (smem_u32(b_smem) & 0x3FFFFu) >> 4;
            const uint32_t b_tap_step = b_tx >> 4;                      // one tap's slice within a stage
            const uint32_t b_stage_step = b_stride >> 4;
            const uint32_t row_wrap = (kPatchPitch - a.ksize) * 8;      // (16-byte units) jump to the next filter row
            const bool row_chunks = kChunk && a.ksize == 7;    // K-chunked mode: one accumulator set per filter row (7x7) ...
            const bool blk_chunks = kChunk && !row_chunks;     // ... or per (channel block, term); (row chunks: tps == 1)
            uint32_t pi = 0, pph = 0, bi = 0, bph = 0, ai = 0, aph = 0;
            for (int t = work0; t < total_tiles; t += wstep) {
                if (!kChunk) {
                    mbar_wait(&acc_empty[ai], aph ^ 1, 3);
                    tc_fence_after();
                }
                uint32_t accumulate = 0;
                for (int cb = 0; cb < a.cin_blocks; ++cb) {
                    for (int term = 0; term < nterms; ++term) {
                        // term 0 and 1 read the hi patch (against W_hi, W_lo), term 2 the residual patch (against W_hi)
                        if (term != 1) mbar_wait(&patch_full[pi], pph, 4);
                        if (lane == 0 && t == work0) B2P_TL(2 + cb);        // 2, 3: patch of channel block 0 / 1 has landed
                        const bool release_patch = (term == nterms - 1) || (term == 1);
                        if (blk_chunks) {
                            mbar_wait(&acc_empty[ai], aph ^ 1, 3);
                            tc_fence_after();
                            accumulate = 0;
                        }
                        uint32_t a_lo = patch_lo0 + pi * (kPatchBytes >> 4);     // window start of the next tap, sub-tile 0
                        int dx = 0;
                        for (int tap0 = 0; tap0 < taps; tap0 += tps) {          // one weight stage = tps consecutive taps
                            const int cnt = taps - tap0 < tps ? taps - tap0 : tps;
                            if (row_chunks && dx == 0) {
                                mbar_wait(&acc_empty[ai], aph ^ 1, 3);
                                tc_fence_after();
                                accumulate = 0;
                            }
                            const uint32_t d_tmem = tmem_base + ai * 256;
                            mbar_wait(&b_full[bi], bph, 5);
                            tc_fence_after();
                            if (lane == 0 && t == work0 && cb == 0 && tap0 == 0) B2P_TL(4);   // first weight slice
                            const bool c_end = row_chunks && dx == a.ksize - 1;
                            if (elect_one()) {
                                uint32_t ta = a_lo, acc = accumulate;
                                uint32_t b_lo = b_lo0 + bi * b_stage_step;
                                int tdx = dx;
                                for (int j = 0; j < cnt; ++j) {
#pragma unroll
                                    for (int sub = 0; sub < 2; ++sub) {
                                        if (sub >= nsub) break;
#pragma unroll
                                        for (int k = 0; k < 4; ++k) {
                                            if (kPair)
                                                umma_bf16_pair(d_tmem + sub * 128, adesc_hi | (ta + sub * 64 + k * 2),
                                                               bdesc_hi | (b_lo + k * 2), idesc, k == 0 ? acc : 1u);
                                            else
                                                umma_bf16(d_tmem + sub * 128, adesc_hi | (ta + sub * 64 + k * 2),
                                                          bdesc_hi | (b_lo + k * 2), idesc, k == 0 ? acc : 1u);
                                        }
                                    }
                                    acc = 1;
                                    b_lo += b_tap_step;
                                    ta += 8;                                      // next tap: one pixel (128 B) to the right
                                    if (++tdx == a.ksize) { tdx = 0; ta += row_wrap; }
                                }
                                if (kPair) umma_commit_pair(&b_empty[bi]);
                                else umma_commit(&b_empty[bi]);
                                if (c_end) {
                                    if (kPair) umma_commit_pair(&acc_full[ai]);
                                    else umma_commit(&acc_full[ai]);
                                }
                            }
                            __syncwarp();
                            accumulate = 1;
                            if (c_end) { if (++ai == 2) { ai = 0; aph ^= 1; } }
                            if (++bi == nb) { bi = 0; bph ^= 1; }
                            dx += cnt;                                            // every lane keeps the window position
                            a_lo += cnt * 8;
                            while (dx >= a.ksize) { dx -= a.ksize; a_lo += row_wrap; }
                        }
                        if (blk_chunks || release_patch) {
                            if (elect_one()) {      // (elect.sync names the same lane every time: the one that issued the MMAs)
                                if (release_patch) {
                                    if (kPair) umma_commit_pair(&patch_empty[pi]);
                                    else umma_commit(&patch_empty[pi]);
                                }
                                if (blk_chunks) {
                                    if (kPair) umma_commit_pair(&acc_full[ai]);
                                    else umma_commit(&acc_full[ai]);
                                }
                            }
                            __syncwarp();
                        }
                        if (blk_chunks) { if (++ai == 2) { ai = 0; aph ^= 1; } }
                        if (release_patch) { if (++pi == kNumPatchStages) { pi = 0; pph ^= 1; } }
                    }
                }
                if (!kChunk) {
                    if (lane == 0 && t == work0) B2P_TL(5);                 // all MMAs of the first tile issued
                    if (elect_one()) {
                        if (kPair) umma_commit_pair(&acc_full[ai]);
                        else umma_commit(&acc_full[ai]);
                    }
                    __syncwarp();
                    if (++ai == 2) { ai = 0; aph ^= 1; }
                }
            }
        }
    } else if (warp >= 2 && warp != 6) {
        // =========================== epilogue (warps 2..5 and 7..10) ===========================
        // A warp may only touch its own quarter (warp & 3) of the 128 TMEM lanes: warps 2..5 cover quarters 2,3,0,1 and
        // warps 7..10 cover 3,0,1,2 - two warps per quarter, which split the accumulator columns in 32-column chunks
        // (even chunks / odd chunks).  With one warp per quarter the layers with little MMA work per tile (Cin = 64, the
        // 1x1 layers, the pooled layers with their shuffles) were bound by this epilogue.
        pdl_wait();               // (stores of this layer may overwrite what the previous layer still reads)
        const int q = warp & 3;   // TMEM lane quarter this warp may access
        const int half = warp >= 7 ? 1 : 0;
        const int h_in = q * 4 + (lane >> 3);
        const int w_in = lane & 7;
        const int Ho = a.pool ? a.H >> 1 : a.H;
        const int Wo = a.pool ? a.W >> 1 : a.W;
        uint32_t ai = 0, aph = 0;
        for (int t = work0; t < total_tiles; t += wstep) {
            const TileCoord tc = decode_tile<kPair>(t, a.n_tiles, a.groups, tiles_x, tiles_y, a.n_img, rank, tile_w);
            if (kChunk) {
                // ---- K-chunked accumulation (n_tile <= 64: this warp owns ONE 32-column chunk of both sub-tiles) ----
                float accr[2][32];
#pragma unroll
                for (int sub = 0; sub < 2; ++sub)
#pragma unroll
                    for (int j = 0; j < 32; ++j) accr[sub][j] = 0.f;
                const int c0 = half * 32;
                const bool mine = c0 < a.n_tile, full = c0 + 32 <= a.n_tile;
                const int nchunks = a.cin_blocks * nterms * (a.ksize == 7 ? 7 : 1);
                for (int chk = 0; chk < nchunks; ++chk) {
                    mbar_wait(&acc_full[ai], aph, 6);
                    tc_fence_after();
                    if (mine) {
#pragma unroll
                        for (int sub = 0; sub < 2; ++sub) {
                            if (sub >= nsub) break;
                            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + ai * 256 + sub * 128 + c0;
                            uint32_t r[32];
                            if (full) tmem_ld32(taddr, r);
                            else {
                                uint32_t r16[16];
                                tmem_ld16(taddr, r16);
#pragma unroll
                                for (int j = 0; j < 16; ++j) { r[j] = r16[j]; r[16 + j] = 0; }
                            }
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 32; ++j) accr[sub][j] = __fadd_rn(accr[sub][j], __uint_as_float(r[j]));
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (kPair) mbar_arrive_leader(&acc_empty[ai]);
                        else mbar_arrive(&acc_empty[ai]);
                    }
                    if (++ai == 2) { ai = 0; aph ^= 1; }
                }
                if (mine) {
                    const int ch_tile = tc.nt * a.n_tile;
                    const float* bias = a.bias + (tc.g * a.n_tiles + tc.nt) * a.n_tile;
                    const int store_ch = a.store_ch[tc.g];
                    float* of32 = a.out_f32[tc.g];
                    const int f32_ch = a.f32_ch[tc.g];
#pragma unroll
                    for (int sub = 0; sub < 2; ++sub) {
                        if (sub >= nsub) break;
                        const int y = tc.y0 + h_in;
                        const int x = tc.x0 + sub * 8 + w_in;
                        const bool valid = tc.valid && (y < a.H) && (x < a.W);
                        const bool writer = a.pool ? (valid && !(lane & 1) && !(lane & 8)) : valid;
                        const bool zero = valid && outside_extent(a, tc.n, y, x);
                        const int yo = a.pool ? y >> 1 : y;
                        const int xo = a.pool ? x >> 1 : x;
                        float v[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float bj = (full || j < 16) ? __ldg(bias + c0 + j) : 0.f;
                            v[j] = accr[sub][j] + bj;
                            if (a.relu) v[j] = fmaxf(v[j], 0.f);
                            if (zero) v[j] = 0.f;
                        }
                        if (a.pool) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 1));
                                v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 8));
                            }
                        }
                        if (writer) {
                            if (a.out != nullptr) {
                                __nv_bfloat16* dst = a.out + (static_cast<size_t>(tc.n * Ho + yo) * Wo + xo) * a.out_cstride +
                                                     a.out_ch_off[tc.g] + ch_tile + c0;
#pragma unroll
                                for (int q8 = 0; q8 < 4; ++q8) {
                                    if (c0 + 8 * q8 < store_ch) {
                                        uint4 u = make_uint4(pack_bf16x2(v[8 * q8], v[8 * q8 + 1]), pack_bf16x2(v[8 * q8 + 2], v[8 * q8 + 3]),
                                                             pack_bf16x2(v[8 * q8 + 4], v[8 * q8 + 5]), pack_bf16x2(v[8 * q8 + 6], v[8 * q8 + 7]));
                                        *reinterpret_cast<uint4*>(dst + 8 * q8) = u;
                                    }
                                }
                                if (a.out_lo != nullptr) {
                                    __nv_bfloat16* dlo = a.out_lo + (dst - a.out);
#pragma unroll
                                    for (int q8 = 0; q8 < 4; ++q8) {
                                        if (c0 + 8 * q8 < store_ch) {
                                            float r8[8];
#pragma unroll
                                            for (int j = 0; j < 8; ++j)
                                                r8[j] = v[8 * q8 + j] - __bfloat162float(__float2bfloat16_rn(v[8 * q8 + j]));
                                            uint4 u = make_uint4(pack_bf16x2(r8[0], r8[1]), pack_bf16x2(r8[2], r8[3]),
                                                                 pack_bf16x2(r8[4], r8[5]), pack_bf16x2(r8[6], r8[7]));
                                            *reinterpret_cast<uint4*>(dlo + 8 * q8) = u;
                                        }
                                    }
                                }
                            }
                            if (of32 != nullptr) {
#pragma unroll
                                for (int j = 0; j < 32; ++j) {
                                    const int c = ch_tile + c0 + j;
                                    if (c < f32_ch)
                                        of32[(static_cast<size_t>(tc.n * f32_ch + c) * Ho + yo) * Wo + xo] = v[j];
                                }
                            }
                        }
                    }
                }
                continue;
            }
            mbar_wait(&acc_full[ai], aph, 6);
            tc_fence_after();
            if (warp == 2 && lane == 0 && t == work0) B2P_TL(6);                // first tile's accumulators complete
            const int ch_tile = tc.nt * a.n_tile;                    // first channel of this n-tile within the group
            const float* bias = a.bias + (tc.g * a.n_tiles + tc.nt) * a.n_tile;
            const int store_ch = a.store_ch[tc.g];
            float* of32 = a.out_f32[tc.g];
            const int f32_ch = a.f32_ch[tc.g];
#pragma unroll 1
            for (int sub = 0; sub < nsub; ++sub) {
                const int y = tc.y0 + h_in;
                const int x = tc.x0 + sub * 8 + w_in;
                const bool valid = tc.valid && (y < a.H) && (x < a.W);
                // pooled: lanes with even (h, w) own the 2x2 window
                const bool writer = a.pool ? (valid && !(lane & 1) && !(lane & 8)) : valid;
                const bool zero = valid && outside_extent(a, tc.n, y, x);
                const int yo = a.pool ? y >> 1 : y;
                const int xo = a.pool ? x >> 1 : x;
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + ai * 256 + sub * 128;
                // 32 accumulator columns per TMEM load (n_tile is a multiple of 16: a 16-column tail handles 48)
#pragma unroll 1
                for (int c0 = half * 32; c0 < a.n_tile; c0 += 64) {
                    const bool full = (c0 + 32 <= a.n_tile);
                    uint32_t r[32];
                    if (full) tmem_ld32(taddr + c0, r);
                    else {
                        uint32_t r16[16];
                        tmem_ld16(taddr + c0, r16);
#pragma unroll
                        for (int j = 0; j < 16; ++j) { r[j] = r16[j]; r[16 + j] = 0; }
                    }
                    float bv[32];
                    {
                        const float4* b4 = reinterpret_cast<const float4*>(bias + c0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 t4 = (full || j < 4) ? __ldg(b4 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                            bv[4 * j] = t4.x; bv[4 * j + 1] = t4.y; bv[4 * j + 2] = t4.z; bv[4 * j + 3] = t4.w;
                        }
                    }
                    tmem_ld_wait();
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        v[j] = __uint_as_float(r[j]) + bv[j];
                        if (a.relu) v[j] = fmaxf(v[j], 0.f);
                        if (zero) v[j] = 0.f;
                    }
                    if (a.pool) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 1));
                            v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 8));
                        }
                    }
                    if (writer) {
                        if (a.out != nullptr) {
                            __nv_bfloat16* dst = a.out + (static_cast<size_t>(tc.n * Ho + yo) * Wo + xo) * a.out_cstride +
                                                 a.out_ch_off[tc.g] + ch_tile + c0;
#pragma unroll
                            for (int q8 = 0; q8 < 4; ++q8) {
                                if (c0 + 8 * q8 < store_ch) {
                                    uint4 u = make_uint4(pack_bf16x2(v[8 * q8], v[8 * q8 + 1]), pack_bf16x2(v[8 * q8 + 2], v[8 * q8 + 3]),
                                                         pack_bf16x2(v[8 * q8 + 4], v[8 * q8 + 5]), pack_bf16x2(v[8 * q8 + 6], v[8 * q8 + 7]));
                                    *reinterpret_cast<uint4*>(dst + 8 * q8) = u;
                                }
                            }
                            if (a.out_lo != nullptr) {      // split mode: residual plane v - bf16(v)
                                __nv_bfloat16* dlo = a.out_lo + (dst - a.out);
#pragma unroll
                                for (int q8 = 0; q8 < 4; ++q8) {
                                    if (c0 + 8 * q8 < store_ch) {
                                        float r8[8];
#pragma unroll
                                        for (int j = 0; j < 8; ++j)
                                            r8[j] = v[8 * q8 + j] - __bfloat162float(__float2bfloat16_rn(v[8 * q8 + j]));
                                        uint4 u = make_uint4(pack_bf16x2(r8[0], r8[1]), pack_bf16x2(r8[2], r8[3]),
                                                             pack_bf16x2(r8[4], r8[5]), pack_bf16x2(r8[6], r8[7]));
                                        *reinterpret_cast<uint4*>(dlo + 8 * q8) = u;
                                    }
                                }
                            }
                        }
                        if (of32 != nullptr) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const int c = ch_tile + c0 + j;
                                if (c < f32_ch)
                                    of32[(static_cast<size_t>(tc.n * f32_ch + c) * Ho + yo) * Wo + xo] = v[j];
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (warp == 2 && lane == 0 && t == work0) B2P_TL(7);                // first tile stored
            if (lane == 0) {
                if (kPair) mbar_arrive_leader(&acc_empty[ai]);     // the leader's MMA warp waits for both CTAs' epilogues
                else mbar_arrive(&acc_empty[ai]);
            }
            if (++ai == 2) { ai = 0; aph ^= 1; }
        }
    }

    tc_fence_before();
    if (threadIdx.x == 0) B2P_TL(8);
    if (kPair) cluster_sync_all();      // both CTAs are done with each other's barriers / the pair's TMEM
    else __syncthreads();
    if (threadIdx.x == 0) B2P_TL(9);
    if (warp == 1) {
        tc_fence_after();
        if (kPair) tmem_dealloc_pair(tmem_base, 512);
        else tmem_dealloc(tmem_base, 512);
    }
}

__global__ void __launch_bounds__(kConvTcThreads, 1) conv_tc_kernel(const __grid_constant__ ConvTcArgs a) {
    conv_tc_body<false, false>(a);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kConvTcThreads, 1)
    conv_tc_pair_kernel(const __grid_constant__ ConvTcArgs a) {
    conv_tc_body<true, false>(a);
}

// K-chunked accumulation (a.chunk; the high-precision split mode): the tensor core sums only one filter row / one channel
// block at a time into TMEM, the epilogue warps add the chunks in fp32 registers with round-to-nearest.
__global__ void __launch_bounds__(kConvTcThreads, 1) conv_tc_chunk_kernel(const __grid_constant__ ConvTcArgs a) {
    conv_tc_body<false, true>(a);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kConvTcThreads, 1)
    conv_tc_pair_chunk_kernel(const __grid_constant__ ConvTcArgs a) {
    conv_tc_body<true, true>(a);
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

}  // namespace

cudaError_t conv_tc_make_maps(ConvTcArgs& a, const __nv_bfloat16* in, int in_cstride, const __nv_bfloat16* w,
                              const __nv_bfloat16* in_lo) {
    PFN_encodeTiled enc = get_encode_fn();
    if (enc == nullptr) return cudaErrorNotSupported;
    if (a.ksize != 1 && a.ksize != 3 && a.ksize != 7) return cudaErrorInvalidValue;
    if (a.n_tile % 16 != 0 || a.n_tile < 16 || a.n_tile > 128) return cudaErrorInvalidValue;
    if (a.groups < 1 || a.groups > 2 || in_cstride % 8 != 0) return cudaErrorInvalidValue;
    if (a.split && in_lo == nullptr) return cudaErrorInvalidValue;
    if (a.pair && (a.n_tile % 32 != 0)) return cudaErrorInvalidValue;     // each CTA of a pair holds n_tile / 2 rows of B
    for (int plane = 0; plane <= (a.split ? 1 : 0); ++plane) {
        cuuint64_t dims[4] = {(cuuint64_t)in_cstride, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)a.n_img};
        cuuint64_t strides[3] = {(cuuint64_t)in_cstride * 2, (cuuint64_t)a.W * in_cstride * 2,
                                 (cuuint64_t)a.H * a.W * in_cstride * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)kPatchPitch, (cuuint32_t)(kTileH + a.ksize - 1), 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        CUresult r = enc(plane ? &a.tm_in_lo : &a.tm_in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                         const_cast<__nv_bfloat16*>(plane ? in_lo : in), dims, strides,
                         box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            fprintf(stderr, "[b200pose] cuTensorMapEncodeTiled(in) failed: %d\n", (int)r);
            return cudaErrorInvalidValue;
        }
    }
    {
        const int cin_pad = a.cin_blocks * 64;
        const int rows = a.groups * a.n_tiles * a.n_tile;
        const int taps = a.ksize * a.ksize;
        // taps per weight stage: as many as leave kMinBStages stages in the ring (small n-tiles: 5 taps of 2 KB per stage for
        // a CTA pair with N = 32; N = 128: one tap per stage as before).  The K-chunked 7x7 mode closes an accumulator set at
        // every filter-row end, which a stage must not straddle.
        const int tap_bytes = (a.pair ? a.n_tile / 2 : a.n_tile) * 128;
        int tps = (kNumBStages * kBStageBytes) / (kMinBStages * tap_bytes);
        if (tps < 1 || (a.chunk && a.ksize == 7)) tps = 1;
        if (tps > taps) tps = taps;
        a.tps = tps;
        cuuint64_t dims[3] = {(cuuint64_t)cin_pad, (cuuint64_t)rows, (cuuint64_t)(2 * taps)};
        cuuint64_t strides[2] = {(cuuint64_t)cin_pad * 2, (cuuint64_t)rows * cin_pad * 2};
        cuuint32_t box[3] = {64, (cuuint32_t)(a.pair ? a.n_tile / 2 : a.n_tile), (cuuint32_t)tps};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&a.tm_w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(w), dims, strides,
                         box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            fprintf(stderr, "[b200pose] cuTensorMapEncodeTiled(w) failed: %d\n", (int)r);
            return cudaErrorInvalidValue;
        }
    }
    return cudaSuccess;
}

namespace {
// Programmatic dependent launch (a.pdl): the next layer's CTAs may start - barrier init, TMEM allocation, descriptor
// prefetch, weight loads - while this layer's last CTAs drain; they wait (griddepcontrol.wait) before touching activations.
// Used by the SMALL-batch plans only, where the ~12 us fixed cost per launch is most of a layer.  At batch 32 it was measured
// and rejected: the isolated network gains ~1 %, the whole step loses ~2 % (3214 vs 3297 frames/s) because the next layer's
// CTAs then win every freed SM against the post-processing kernels of the previous batch.
template <class Kernel>
cudaError_t launch_plain(Kernel kernel, int grid, cudaStream_t stream, const ConvTcArgs& a) {
    if (a.pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kConvTcThreads);
        cfg.dynamicSmemBytes = kConvTcSmemBytes;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, kernel, a);
    }
    kernel<<<grid, kConvTcThreads, kConvTcSmemBytes, stream>>>(a);
    return cudaGetLastError();
}
}  // namespace

cudaError_t conv_tc_launch(const ConvTcArgs& a, int num_sms, cudaStream_t stream) {
    static DynSmemOptIn optin, optin_pair;   // per device: a second net on another GPU of the same process needs its own opt-in
    if (a.pool && ((a.H | a.W) & 1)) return cudaErrorInvalidValue;
    const int tiles_x = (a.W + (a.narrow ? 8 : kTileW) - 1) / (a.narrow ? 8 : kTileW);
    const int tiles_y = (a.H + kTileH - 1) / kTileH;
    static DynSmemOptIn optin_chunk, optin_pair_chunk;
    if (a.chunk && a.n_tile > 64) return cudaErrorInvalidValue;      // one 32-column chunk per epilogue warp
    if (a.tps < 1) return cudaErrorInvalidValue;                     // conv_tc_make_maps has not run
    if (a.pair) {
        const int pairs = ((a.n_img * tiles_y * tiles_x + 1) / 2) * a.groups * a.n_tiles;
        const int clusters = pairs < num_sms / 2 ? pairs : num_sms / 2;
        if (a.chunk) {
            cudaError_t e = optin_pair_chunk.ensure(conv_tc_pair_chunk_kernel, kConvTcSmemBytes);
            if (e != cudaSuccess) return e;
            return launch_plain(conv_tc_pair_chunk_kernel, 2 * clusters, stream, a);
        } else {
            cudaError_t e = optin_pair.ensure(conv_tc_pair_kernel, kConvTcSmemBytes);
            if (e != cudaSuccess) return e;
            return launch_plain(conv_tc_pair_kernel, 2 * clusters, stream, a);   // __cluster_dims__(2,1,1)
        }
    }
    const int total = a.n_img * tiles_y * tiles_x * a.groups * a.n_tiles;
    const int grid = total < num_sms ? total : num_sms;
    if (a.chunk) {
        cudaError_t e = optin_chunk.ensure(conv_tc_chunk_kernel, kConvTcSmemBytes);
        if (e != cudaSuccess) return e;
        return launch_plain(conv_tc_chunk_kernel, grid, stream, a);
    }
    cudaError_t e = optin.ensure(conv_tc_kernel, kConvTcSmemBytes);
    if (e != cudaSuccess) return e;
    return launch_plain(conv_tc_kernel, grid, stream, a);
}

#ifdef B2P_CONV_TIMELINE
cudaError_t conv_tc_read_timeline(unsigned long long* out) {
    cudaError_t e = cudaMemcpyFromSymbol(out, g_conv_timeline, sizeof(g_conv_timeline));
    if (e != cudaSuccess) return e;
    void* p = nullptr;
    e = cudaGetSymbolAddress(&p, g_conv_timeline);
    if (e != cudaSuccess) return e;
    return cudaMemset(p, 0, sizeof(g_conv_timeline));
}
#endif

}  // namespace b2p
