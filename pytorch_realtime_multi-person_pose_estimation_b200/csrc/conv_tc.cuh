// Host-side interface of the tcgen05 "halo-patch" implicit-GEMM convolution (conv_tc.cu).
// Replaces the nn.Conv2d(+ReLU)(+MaxPool2d)(+torch.cat) sequences of
// /root/reference/lib/network/rtpose_vgg.py:23-29,165 for every conv with Cin >= 64.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace b2p {

constexpr int kTileW = 16;        // CTA tile: 16 x 16 output pixels = two 8-wide x 16-high UMMA M=128 sub-tiles
constexpr int kTileH = 16;
constexpr int kPatchPitch = 24;   // patch row pitch in pixels (16 + 6 halo, rounded up to a multiple of 8)
constexpr int kMaxKs = 7;
constexpr int kPatchBytes = kPatchPitch * (kTileH + kMaxKs - 1) * 128;  // 67,584 B per 64-channel block
constexpr int kBStageBytes = 128 * 128;                                 // up to N=128 rows of 64 bf16
#ifndef B2P_CONV_B_STAGES
#define B2P_CONV_B_STAGES 3      // weight (B operand) ring: 48 KB, cut into stages of `tps` taps (conv_tc.cu): three stages of two 8 KB
                                 // half-slices for a CTA pair with N = 128.  The shared memory a conv CTA leaves free decides which
                                 // post-processing kernels of the previous batch can run NEXT to it: at 185 KB the small ones still
                                 // fit; taking everything (four patch stages, 230 KB) cost 9 % of the step; see DESIGN.md 2.4
#endif
constexpr int kNumBStages = B2P_CONV_B_STAGES;
#ifndef B2P_CONV_MIN_B_STAGES
#define B2P_CONV_MIN_B_STAGES 3
#endif
constexpr int kMinBStages = B2P_CONV_MIN_B_STAGES;     // a stage holds as many taps as still leave this many stages in the ring
constexpr int kMaxBStages = 16;       // the ring is cut into stages of the size the layer's n-tile needs (conv_tc.cu)
constexpr int kNumPatchStages = 2;
constexpr int kConvTcThreads = 352;   // warps: 0 patch TMA, 1 MMA, 2-5 and 7-10 epilogue (two per TMEM lane quarter), 6 weight TMA
constexpr int kConvTcSmemBytes = kNumPatchStages * kPatchBytes + kNumBStages * kBStageBytes + 1024 /*align*/ + 512;

struct ConvTcArgs {
    // ---- geometry (stride 1, "same" padding, square kernel)
    int n_img, H, W;
    int ksize;                // 1, 3 or 7
    int cin_blocks;           // 64-channel blocks per group
    int in_ch_base;           // first input channel (in the NHWC buffer) of group 0
    int in_ch_group_stride;   // channel offset between groups in the input buffer (0 = groups share input)
    int groups;               // 1 or 2
    int n_tile;               // UMMA N: multiple of 16, <= 128
    int n_tiles;              // N tiles per group
    // ---- epilogue
    const float* bias;        // [groups * n_tiles * n_tile]
    int relu;
    int pool;                 // fuse MaxPool2d(2,2): output is (H/2, W/2)
    __nv_bfloat16* out;       // NHWC bf16 (may be null)
    int out_cstride;          // channels per pixel of the output buffer
    int out_ch_off[2];        // first output channel per group
    int store_ch[2];          // channels (multiple of 8) stored per group *per n-tile*
    float* out_f32[2];        // optional NCHW fp32 copy per group (heads), may be null
    int f32_ch[2];            // valid channels of the fp32 copy
    int use_base_offset;      // descriptor swizzle-phase field (see DESIGN.md)
    // ---- split-precision ("bf16x3") mode: operands are hi + lo bf16 planes, three MMA terms per K block
    int split;                // 0: plain bf16; 1: A_hi*W_hi + A_hi*W_lo + A_lo*W_hi
    __nv_bfloat16* out_lo;    // residual plane of the output (same geometry as `out`), split mode only
    // ---- CTA-pair mode (tcgen05 cta_group::2): clusters of two CTAs share each weight slice; needs n_tile % 32 == 0
    int pair;
    // ---- K-chunked accumulation (n_tile <= 64): see conv_tc_chunk_kernel
    int chunk;
    // ---- narrow tiles (small batches): the CTA tile is 8 x 16 pixels (one UMMA M=128 sub-tile) instead of 16 x 16
    int narrow;
    // ---- taps per weight stage (set by conv_tc_make_maps together with the weight map's box)
    int tps;
    // ---- programmatic dependent launch of this layer behind the previous one (small-batch plans)
    int pdl;
    // ---- ragged batches: full-resolution (h, w) of every image, the image sitting top-left in its slot of the [H, W]
    //      canvas; output pixels outside (h >> ext_shift, w >> ext_shift) at this layer's input resolution store zeros
    //      (bf16, residual plane and fp32 copy), so that the next layer's halo reads what TMA's zero fill gives the image
    //      alone.  nullptr: every image fills the canvas.
    const int2* ext;
    int ext_shift;
    // ---- tensor maps
    CUtensorMap tm_in;        // 4D (C, W, H, N) bf16, box (64, 24, 16+ks-1, 1), SWIZZLE_128B
    CUtensorMap tm_w;         // 3D (cin_pad, groups*n_tiles*n_tile, 2*taps) bf16 [hi taps | lo taps], box (64, n_tile, tps)
                              // (pair mode: box (64, n_tile / 2, 1) - each CTA of a pair loads its half of the N rows)
    CUtensorMap tm_in_lo;     // residual plane of the input (split mode)
};

// Builds the tensor maps. `in` (and `in_lo` in split mode): NHWC buffers with `in_cstride` channels per pixel.
// `w`: packed weights [2*taps][groups*n_tiles*n_tile][cin_blocks*64]: bf16(w) for the first `taps` slices, the
// residual bf16(w - hi) for the second.
cudaError_t conv_tc_make_maps(ConvTcArgs& a, const __nv_bfloat16* in, int in_cstride, const __nv_bfloat16* w,
                              const __nv_bfloat16* in_lo = nullptr);
cudaError_t conv_tc_launch(const ConvTcArgs& a, int num_sms, cudaStream_t stream);

#ifdef B2P_CONV_TIMELINE
// Debug builds only (tools/conv_timeline.sh): clock64() stamps of the first 64 CTAs at the phase boundaries of conv_tc_body.
constexpr int kTlSlots = 16;
cudaError_t conv_tc_read_timeline(unsigned long long* out /*[64 * kTlSlots]*/);     // copies and clears
#endif

}  // namespace b2p
