// CUDA-core kernels around the tcgen05 conv (see conv_misc.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace b2p {

struct ConvF32Args {
    const float* in;      // NHWC fp32
    int in_cstride, in_ch_off;
    const float* w;       // OIHW fp32 (the state_dict tensor as is)
    const float* bias;
    float* out;           // NHWC fp32
    int out_cstride, out_ch_off;
    float* out_nchw;      // optional NCHW copy [n][cout][H][W]
    int n_img, H, W, cin, cout, ks, relu;
    const int2* ext;      // ragged batches: full-resolution (h, w) per image; outputs outside (h, w) >> ext_shift are +0
    int ext_shift;        // (nullptr: every image fills the canvas)
};

// in: fp32 NCHW [N,3,H,W] (in_is_u8_hwc = 0), or uint8 HWC BGR [N,H,W,3] with the normalisation `in_is_u8_hwc`
// (preprocess_core.h: 1 rtpose, 2 vgg, 3 inception, 4 ssd) fused into the load.
// ext (ragged batches, device array or null): image i is valid in [0, ext[i].x) x [0, ext[i].y) of its [H, W] slot; input
// pixels beyond it read as 0.0 after normalisation (the conv's zero padding), outputs beyond it are stored as +0.
cudaError_t conv_first_launch(const void* in, int in_is_u8_hwc, const float* w_oihw, const float* bias,
                              __nv_bfloat16* out_nhwc, __nv_bfloat16* out_lo /*residual plane or null*/, int N, int H,
                              int W, cudaStream_t s, const int2* ext = nullptr);
cudaError_t u8hwc_to_f32nchw_launch(const unsigned char* in, float* out, int N, int H, int W, int mode, cudaStream_t s,
                                    const int2* ext = nullptr);
cudaError_t conv_f32_launch(const ConvF32Args& a, cudaStream_t s);
cudaError_t maxpool_f32_launch(const float* in, float* out, int N, int H, int W, int C, cudaStream_t s);
cudaError_t nchw_to_nhwc_f32_launch(const float* in, float* out, int N, int C, int H, int W, int out_cstride,
                                    int out_ch_off, cudaStream_t s);

}  // namespace b2p
