// CUDA-core kernels around the tcgen05 conv:
//   conv_first_kernel : conv1_1 (3 -> 64, 3x3, pad 1) + bias + ReLU, fp32 NCHW in -> bf16 NHWC out
//                       (/root/reference/lib/network/rtpose_vgg.py:69).  K = 27 is too thin for UMMA tiles and the
//                       layer is HBM/LSU bound (AI ~ 26 FLOP/B), so it runs on the FP32 pipes.
//   conv_f32_kernel   : generic stride-1 "same" conv, NHWC fp32 in/out, fp32 FMA accumulate - the fp32-parity mode
//                       of every layer (heat/PAF within 1e-3 of the fp32 reference) and the GPU-side cross-check of
//                       the bf16 tensor-core path.
//   maxpool_f32_kernel: MaxPool2d(2,2) NHWC fp32 (parity mode only; the bf16 path fuses pooling in the conv epilogue)
//   nchw_to_nhwc / nhwc_slice_to_nchw : layout glue for the parity path.
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "conv_misc.cuh"
#include "preprocess_core.h"

namespace b2p {

namespace {

// ------------------------------------------------------------------ conv1_1
constexpr int kF_TW = 64, kF_TH = 4;        // output tile per block: 64 x 4 pixels, 2 pixels per thread
constexpr int kF_Threads = 128;

// kIn = 0: `in` is fp32 NCHW (already normalised).  kIn = kPreRtpose / kPreVgg / kPreInception / kPreSsd: `in` is uint8 HWC
// BGR [N,H,W,3] and that normalisation (/root/reference/lib/datasets/preprocessing.py, restated in preprocess_core.h;
// rtpose: x/256 - 0.5, HWC -> CHW) is fused into the tile load.
template <int kIn>
__global__ void __launch_bounds__(kF_Threads) conv_first_kernel(const void* __restrict__ in_v, const float* __restrict__ wgt,
                                                                const float* __restrict__ bias,
                                                                __nv_bfloat16* __restrict__ out,
                                                                __nv_bfloat16* __restrict__ out_lo, int H, int W,
                                                                const int2* __restrict__ ext) {
    constexpr bool kU8 = kIn != 0;
    __shared__ float s_in[3][kF_TH + 2][kF_TW + 2];
    __shared__ __align__(16) float s_w[27][64];
    __shared__ float s_b[64];
    const int n = blockIdx.z, y0 = blockIdx.y * kF_TH, x0 = blockIdx.x * kF_TW;
    // ragged batches: the image's extent in its canvas slot; pixels beyond it are the conv's zero padding
    const int2 e = ext != nullptr ? ext[n] : make_int2(H, W);
    const int tid = threadIdx.x;
    for (int i = tid; i < 27 * 64; i += kF_Threads) {
        // wgt is OIHW [64][3][3][3]; s_w[(c*3+ky)*3+kx][o]
        const int o = i & 63, k = i >> 6;
        s_w[k][o] = wgt[o * 27 + k];
    }
    if (tid < 64) s_b[tid] = bias[tid];
    for (int i = tid; i < 3 * (kF_TH + 2) * (kF_TW + 2); i += kF_Threads) {
        int c, yy, xx;
        if (kU8) {   // channel fastest: consecutive threads read consecutive bytes
            c = i % 3;
            const int r = i / 3;
            yy = r / (kF_TW + 2);
            xx = r - yy * (kF_TW + 2);
        } else {
            c = i / ((kF_TH + 2) * (kF_TW + 2));
            const int r = i - c * (kF_TH + 2) * (kF_TW + 2);
            yy = r / (kF_TW + 2);
            xx = r - yy * (kF_TW + 2);
        }
        const int gy = y0 + yy - 1, gx = x0 + xx - 1;
        float v = 0.f;
        if (gy >= 0 && gy < e.x && gx >= 0 && gx < e.y) {
            if (kU8) {
                const unsigned char u =
                    static_cast<const unsigned char*>(in_v)[(((size_t)n * H + gy) * W + gx) * 3 + pre_src_channel(kIn, c)];
                v = pre_value(kIn, u, c);
            } else {
                v = static_cast<const float*>(in_v)[(((size_t)n * 3 + c) * H + gy) * W + gx];
            }
        }
        s_in[c][yy][xx] = v;
    }
    __syncthreads();
    const int ty = tid >> 5, tx = (tid & 31) * 2;     // 4 rows x 32 pixel pairs
    float v[2][27];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                v[0][(c * 3 + ky) * 3 + kx] = s_in[c][ty + ky][tx + kx];
                v[1][(c * 3 + ky) * 3 + kx] = s_in[c][ty + ky][tx + 1 + kx];
            }
    const int y = y0 + ty, x = x0 + tx;
#pragma unroll 1
    for (int o0 = 0; o0 < 64; o0 += 16) {
        float acc[2][16];
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[0][j] = acc[1][j] = s_b[o0 + j];
#pragma unroll
        for (int k = 0; k < 27; ++k) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
                const float4 w4 = *reinterpret_cast<const float4*>(&s_w[k][o0 + j4 * 4]);
                acc[0][j4 * 4 + 0] = fmaf(v[0][k], w4.x, acc[0][j4 * 4 + 0]);
                acc[0][j4 * 4 + 1] = fmaf(v[0][k], w4.y, acc[0][j4 * 4 + 1]);
                acc[0][j4 * 4 + 2] = fmaf(v[0][k], w4.z, acc[0][j4 * 4 + 2]);
                acc[0][j4 * 4 + 3] = fmaf(v[0][k], w4.w, acc[0][j4 * 4 + 3]);
                acc[1][j4 * 4 + 0] = fmaf(v[1][k], w4.x, acc[1][j4 * 4 + 0]);
                acc[1][j4 * 4 + 1] = fmaf(v[1][k], w4.y, acc[1][j4 * 4 + 1]);
                acc[1][j4 * 4 + 2] = fmaf(v[1][k], w4.z, acc[1][j4 * 4 + 2]);
                acc[1][j4 * 4 + 3] = fmaf(v[1][k], w4.w, acc[1][j4 * 4 + 3]);
            }
        }
        if (y < H) {
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                if (x + p >= W) continue;
                if (y >= e.x || x + p >= e.y) {      // outside the image's extent: +0
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[p][j] = 0.f;
                }
                __nv_bfloat16* dst = out + (((size_t)n * H + y) * W + x + p) * 64 + o0;
                uint32_t pk[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    __nv_bfloat162 b = __floats2bfloat162_rn(fmaxf(acc[p][2 * j], 0.f), fmaxf(acc[p][2 * j + 1], 0.f));
                    pk[j] = *reinterpret_cast<uint32_t*>(&b);
                }
                reinterpret_cast<uint4*>(dst)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                reinterpret_cast<uint4*>(dst)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                if (out_lo != nullptr) {     // split-precision mode: residual plane v - bf16(v)
                    __nv_bfloat16* dlo = out_lo + (dst - out);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float v0 = fmaxf(acc[p][2 * j], 0.f), v1 = fmaxf(acc[p][2 * j + 1], 0.f);
                        __nv_bfloat162 b = __floats2bfloat162_rn(v0 - __bfloat162float(__float2bfloat16_rn(v0)),
                                                                 v1 - __bfloat162float(__float2bfloat16_rn(v1)));
                        pk[j] = *reinterpret_cast<uint32_t*>(&b);
                    }
                    reinterpret_cast<uint4*>(dlo)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    reinterpret_cast<uint4*>(dlo)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                }
            }
        }
    }
}


// ------------------------------------------------------------------ conv1_1 on the tensor cores (bf16 mode)
// conv1_1 is a GEMM with K = 27: far too thin for a tcgen05 tile pipeline (one 128 x 64 x 32 MMA per 128 pixels), and its
// roofline is HBM (0.4 MB in, 17.7 MB out per frame: 0.09 ms per batch of 32 at the measured copy bandwidth) - the fp32
// CUDA-core kernel above needs 0.50 ms for its 7.5 G fused multiply-adds.  Here every warp runs warp-level
// mma.sync.m16n8k16 (bf16 x bf16 -> fp32) on im2col fragments gathered straight from the staged input tile: K is padded
// to 32 with zeros, the 64 output channels are 8 n-tiles, bias is the accumulator's initial value.  The uint8 frames of
// the rtpose normalisation ((x - 128) / 256) are exact in bf16; the weights are rounded to bf16 like every other layer's.
// Output: bf16 NHWC through a swizzled shared-memory tile, 16-byte coalesced stores.
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

template <int kIn>
__global__ void __launch_bounds__(kF_Threads) conv_first_mma_kernel(const void* __restrict__ in_v, const float* __restrict__ wgt,
                                                                    const float* __restrict__ bias,
                                                                    __nv_bfloat16* __restrict__ out, int H, int W,
                                                                    const int2* __restrict__ ext) {
    constexpr bool kU8 = kIn != 0;
    constexpr int kRowF = kF_TW + 2, kPlaneF = (kF_TH + 2) * kRowF;
    __shared__ float s_in[3 * kPlaneF];
    __shared__ __align__(16) uint32_t s_out[kF_TH * kF_TW * 32];      // [pixel][8 chunks of 16 B], chunk index ^ (pixel & 7)
    const int n = blockIdx.z, y0 = blockIdx.y * kF_TH, x0 = blockIdx.x * kF_TW;
    const int2 e = ext != nullptr ? ext[n] : make_int2(H, W);          // ragged batches: the image's extent
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 3 * kPlaneF; i += kF_Threads) {
        int c, yy, xx;
        if (kU8) {   // channel fastest: consecutive threads read consecutive bytes
            c = i % 3;
            const int r = i / 3;
            yy = r / kRowF;
            xx = r - yy * kRowF;
        } else {
            c = i / kPlaneF;
            const int r = i - c * kPlaneF;
            yy = r / kRowF;
            xx = r - yy * kRowF;
        }
        const int gy = y0 + yy - 1, gx = x0 + xx - 1;
        float v = 0.f;
        if (gy >= 0 && gy < e.x && gx >= 0 && gx < e.y) {
            if (kU8) {
                const unsigned char u =
                    static_cast<const unsigned char*>(in_v)[(((size_t)n * H + gy) * W + gx) * 3 + pre_src_channel(kIn, c)];
                v = pre_value(kIn, u, c);
            } else {
                v = static_cast<const float*>(in_v)[(((size_t)n * 3 + c) * H + gy) * W + gx];
            }
        }
        s_in[c * kPlaneF + yy * kRowF + xx] = v;
    }
    // this thread's K indices of the A / B fragments: k-step s, register pair i: kk = 16 s + 8 (i >> 1)... see PTX m16n8k16
    const int q = lane & 3, r0 = lane >> 2;
    int aoff[2][4];                  // [k-step][a-register half: cols 2q, 2q+1, 2q+8, 2q+9] -> s_in offset, or -1 (K padding)
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int kk = 16 * s2 + 2 * q + (j & 1) + 8 * (j >> 1);
            aoff[s2][j] = kk < 27 ? (kk / 9) * kPlaneF + ((kk % 9) / 3) * kRowF + (kk % 3) : -1;
        }
    uint32_t bfrag[8][2][2];         // [n-tile][k-step][b0, b1]: B[k][n] = w[n][k], n = 8 j + r0, k = 16 s + 2 q (+1) (+8)
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int k0 = 16 * s2 + 2 * q + 8 * hh;
                const float w0 = k0 < 27 ? __ldg(wgt + (8 * j + r0) * 27 + k0) : 0.f;
                const float w1 = k0 + 1 < 27 ? __ldg(wgt + (8 * j + r0) * 27 + k0 + 1) : 0.f;
                bfrag[j][s2][hh] = pack_bf16(w0, w1);
            }
    float bs[8][2];
#pragma unroll
    for (int j = 0; j < 8; ++j) { bs[j][0] = __ldg(bias + 8 * j + 2 * q); bs[j][1] = __ldg(bias + 8 * j + 2 * q + 1); }
    __syncthreads();
    const float* srow = s_in + warp * kRowF;             // this warp's output row of the tile (ty = warp)
#pragma unroll 1
    for (int mt = 0; mt < kF_TW / 16; ++mt) {
        uint32_t afrag[2][4];
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
            float v[4][2];                               // [a-register][col 0 / col 1]: rows r0 (a0, a2) and r0 + 8 (a1, a3)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int off = aoff[s2][j];
                v[j][0] = off >= 0 ? srow[off + 16 * mt + r0] : 0.f;
                v[j][1] = off >= 0 ? srow[off + 16 * mt + r0 + 8] : 0.f;
            }
            afrag[s2][0] = pack_bf16(v[0][0], v[1][0]);  // row r0,     k = 2q, 2q+1
            afrag[s2][1] = pack_bf16(v[0][1], v[1][1]);  // row r0 + 8, k = 2q, 2q+1
            afrag[s2][2] = pack_bf16(v[2][0], v[3][0]);  // row r0,     k = 2q+8, 2q+9
            afrag[s2][3] = pack_bf16(v[2][1], v[3][1]);  // row r0 + 8, k = 2q+8, 2q+9
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float d[4] = {bs[j][0], bs[j][1], bs[j][0], bs[j][1]};
            mma_bf16_16816(d, afrag[0], bfrag[j][0][0], bfrag[j][0][1]);
            mma_bf16_16816(d, afrag[1], bfrag[j][1][0], bfrag[j][1][1]);
            // d0, d1: pixel row r0, channels 8j + 2q, +1;  d2, d3: pixel row r0 + 8
            const int p0 = warp * kF_TW + 16 * mt + r0, p1 = p0 + 8;
            s_out[p0 * 32 + ((j ^ (p0 & 7)) << 2) + q] = pack_bf16(fmaxf(d[0], 0.f), fmaxf(d[1], 0.f));
            s_out[p1 * 32 + ((j ^ (p1 & 7)) << 2) + q] = pack_bf16(fmaxf(d[2], 0.f), fmaxf(d[3], 0.f));
        }
    }
    __syncthreads();
    for (int i = tid; i < kF_TH * kF_TW * 8; i += kF_Threads) {
        const int p = i >> 3, ch = i & 7;
        const int y = y0 + p / kF_TW, x = x0 + p % kF_TW;
        if (y < H && x < W)
            reinterpret_cast<uint4*>(out + (((size_t)n * H + y) * W + x) * 64)[ch] =
                (y < e.x && x < e.y) ? reinterpret_cast<const uint4*>(s_out + p * 32)[ch ^ (p & 7)] : make_uint4(0, 0, 0, 0);
    }
}

// ------------------------------------------------------------------ fp32 parity conv
// Block: 64 output pixels (8x8) x 64 output channels, 256 threads, each 4 pixels x 4 channels.
constexpr int kR_Threads = 256;
constexpr int kR_KC = 16;   // input channels per smem chunk

__global__ void __launch_bounds__(kR_Threads) conv_f32_kernel(ConvF32Args a) {
    __shared__ float s_a[kR_KC][64 + 4];     // [cin][pixel]
    __shared__ float s_b[kR_KC][64 + 4];     // [cin][cout]
    const int tiles_x = (a.W + 7) / 8;
    const int tile = blockIdx.x;
    const int n = blockIdx.z;
    const int ty0 = (tile / tiles_x) * 8, tx0 = (tile % tiles_x) * 8;
    const int co0 = blockIdx.y * 64;
    const int tid = threadIdx.x;
    const int pg = tid >> 4, cg = tid & 15;          // pixel group (4 pixels), channel group (4 channels)
    const int pad = a.ks >> 1;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int tap = 0; tap < a.ks * a.ks; ++tap) {
        const int dy = tap / a.ks - pad, dx = tap % a.ks - pad;
        for (int c0 = 0; c0 < a.cin; c0 += kR_KC) {
            // A chunk: 64 pixels x 16 channels
            for (int i = tid; i < 64 * kR_KC; i += kR_Threads) {
                const int p = i / kR_KC, c = i - p * kR_KC;
                const int y = ty0 + (p >> 3) + dy, x = tx0 + (p & 7) + dx;
                float v = 0.f;
                if (y >= 0 && y < a.H && x >= 0 && x < a.W && c0 + c < a.cin)
                    v = a.in[(((size_t)n * a.H + y) * a.W + x) * a.in_cstride + a.in_ch_off + c0 + c];
                s_a[c][p] = v;
            }
            // B chunk: 16 channels x 64 couts ; weights OIHW fp32
            for (int i = tid; i < 64 * kR_KC; i += kR_Threads) {
                const int c = i / 64, o = i - c * 64;
                float v = 0.f;
                if (c0 + c < a.cin && co0 + o < a.cout)
                    v = a.w[(((size_t)(co0 + o) * a.cin + c0 + c) * a.ks + (tap / a.ks)) * a.ks + (tap % a.ks)];
                s_b[c][o] = v;
            }
            __syncthreads();
#pragma unroll
            for (int c = 0; c < kR_KC; ++c) {
                const float4 av = *reinterpret_cast<const float4*>(&s_a[c][pg * 4]);
                const float4 bv = *reinterpret_cast<const float4*>(&s_b[c][cg * 4]);
                const float aa[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int p = pg * 4 + i;
        const int y = ty0 + (p >> 3), x = tx0 + (p & 7);
        if (y >= a.H || x >= a.W) continue;
        const bool zero = a.ext != nullptr && (y >= (a.ext[n].x >> a.ext_shift) || x >= (a.ext[n].y >> a.ext_shift));
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int o = co0 + cg * 4 + j;
            if (o >= a.cout) continue;
            float v = acc[i][j] + a.bias[o];
            if (a.relu) v = fmaxf(v, 0.f);
            if (zero) v = 0.f;          // ragged batches: outside the image's extent
            a.out[(((size_t)n * a.H + y) * a.W + x) * a.out_cstride + a.out_ch_off + o] = v;
            if (a.out_nchw) a.out_nchw[(((size_t)n * a.cout + o) * a.H + y) * a.W + x] = v;
        }
    }
}

__global__ void maxpool_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int H, int W, int C) {
    const int Ho = H / 2, Wo = W / 2;
    const size_t total = (size_t)N * Ho * Wo * C;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = i % C;
        size_t t = i / C;
        const int xo = t % Wo;
        t /= Wo;
        const int yo = t % Ho;
        const int n = t / Ho;
        const float* p = in + (((size_t)n * H + 2 * yo) * W + 2 * xo) * C + c;
        out[i] = fmaxf(fmaxf(p[0], p[C]), fmaxf(p[(size_t)W * C], p[(size_t)W * C + C]));
    }
}

__global__ void nchw_to_nhwc_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int C, int H,
                                        int W, int out_cstride, int out_ch_off) {
    const size_t total = (size_t)N * C * H * W;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int x = i % W;
        size_t t = i / W;
        const int y = t % H;
        t /= H;
        const int c = t % C;
        const int n = t / C;
        out[(((size_t)n * H + y) * W + x) * out_cstride + out_ch_off + c] = in[i];
    }
}

}  // namespace

cudaError_t conv_first_launch(const void* in, int in_is_u8_hwc, const float* w_oihw, const float* bias,
                              __nv_bfloat16* out_nhwc, __nv_bfloat16* out_lo, int N, int H, int W, cudaStream_t s,
                              const int2* ext) {
    dim3 grid((W + kF_TW - 1) / kF_TW, (H + kF_TH - 1) / kF_TH, N);
    if (out_lo == nullptr) {        // bf16 mode: tensor cores
        switch (in_is_u8_hwc) {
            case kPreNone: conv_first_mma_kernel<kPreNone><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, H, W, ext); break;
            case kPreRtpose: conv_first_mma_kernel<kPreRtpose><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, H, W, ext); break;
            case kPreVgg: conv_first_mma_kernel<kPreVgg><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, H, W, ext); break;
            case kPreInception: conv_first_mma_kernel<kPreInception><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, H, W, ext); break;
            case kPreSsd: conv_first_mma_kernel<kPreSsd><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, H, W, ext); break;
            default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
    }
    switch (in_is_u8_hwc) {
        case kPreNone: conv_first_kernel<kPreNone><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, out_lo, H, W, ext); break;
        case kPreRtpose: conv_first_kernel<kPreRtpose><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, out_lo, H, W, ext); break;
        case kPreVgg: conv_first_kernel<kPreVgg><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, out_lo, H, W, ext); break;
        case kPreInception: conv_first_kernel<kPreInception><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, out_lo, H, W, ext); break;
        case kPreSsd: conv_first_kernel<kPreSsd><<<grid, kF_Threads, 0, s>>>(in, w_oihw, bias, out_nhwc, out_lo, H, W, ext); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

namespace {
__global__ void u8hwc_to_f32nchw_kernel(const unsigned char* __restrict__ in, float* __restrict__ out, int N, int H, int W,
                                        int mode, const int2* __restrict__ ext) {
    const size_t total = (size_t)N * 3 * H * W;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int x = i % W;
        size_t t = i / W;
        const int y = t % H;
        t /= H;
        const int c = t % 3;
        const int n = t / 3;
        if (ext != nullptr && (y >= ext[n].x || x >= ext[n].y)) out[i] = 0.f;     // outside a ragged image: conv padding
        else out[i] = pre_value(mode, in[(((size_t)n * H + y) * W + x) * 3 + pre_src_channel(mode, c)], c);
    }
}
}  // namespace

cudaError_t u8hwc_to_f32nchw_launch(const unsigned char* in, float* out, int N, int H, int W, int mode, cudaStream_t s,
                                    const int2* ext) {
    if (mode < kPreRtpose || mode > kPreSsd) return cudaErrorInvalidValue;
    const size_t total = (size_t)N * 3 * H * W;
    const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    u8hwc_to_f32nchw_kernel<<<blocks, 256, 0, s>>>(in, out, N, H, W, mode, ext);
    return cudaGetLastError();
}

cudaError_t conv_f32_launch(const ConvF32Args& a, cudaStream_t s) {
    const int tiles = ((a.W + 7) / 8) * ((a.H + 7) / 8);
    dim3 grid(tiles, (a.cout + 63) / 64, a.n_img);
    conv_f32_kernel<<<grid, kR_Threads, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t maxpool_f32_launch(const float* in, float* out, int N, int H, int W, int C, cudaStream_t s) {
    const size_t total = (size_t)N * (H / 2) * (W / 2) * C;
    const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    maxpool_f32_kernel<<<blocks, 256, 0, s>>>(in, out, N, H, W, C);
    return cudaGetLastError();
}

cudaError_t nchw_to_nhwc_f32_launch(const float* in, float* out, int N, int C, int H, int W, int out_cstride,
                                    int out_ch_off, cudaStream_t s) {
    const size_t total = (size_t)N * C * H * W;
    const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    nchw_to_nhwc_f32_kernel<<<blocks, 256, 0, s>>>(in, out, N, C, H, W, out_cstride, out_ch_off);
    return cudaGetLastError();
}

}  // namespace b2p
