// crop_with_factor kernel: one thread per destination pixel (3 channels), consecutive threads on consecutive pixels
// of a destination row.  Streaming / gather kernel, HBM- and L2-bound: a frame is read at most once (each source row
// pair is shared by the threads of a destination row and stays in L1/L2) and written once; the per-pixel work is two
// double multiplications for the source coordinates and 12 integer MACs.
#include "resize.cuh"

namespace b2p {
namespace {

constexpr int kThreads = 256;

// Destination pixel (y, x) of one frame: its three bytes, zero outside the resized area (the padding).
__device__ __forceinline__ void crop_px3(const unsigned char* src, int src_h, int src_w, const CropGeom& g, int y, int x,
                                         unsigned char* dst) {
    unsigned char v0 = 0, v1 = 0, v2 = 0;
    if (y < g.res_h && x < g.res_w) {
        const long stride = (long)src_w * 3;
        if (g.area2) {
            v0 = rs_area2_px(src, src_h, src_w, stride, 3, 0, x, y);
            v1 = rs_area2_px(src, src_h, src_w, stride, 3, 1, x, y);
            v2 = rs_area2_px(src, src_h, src_w, stride, 3, 2, x, y);
        } else {
            const LinCoef cx = rs_coef_x(x, src_w, g.step), cy = rs_coef_y(y, src_h, g.step);
            v0 = rs_linear_px(src, stride, 3, 0, cx, cy);
            v1 = rs_linear_px(src, stride, 3, 1, cx, cy);
            v2 = rs_linear_px(src, stride, 3, 2, cx, cy);
        }
    }
    dst[0] = v0;
    dst[1] = v1;
    dst[2] = v2;
}

__global__ void __launch_bounds__(kThreads) crop_with_factor_kernel(const unsigned char* __restrict__ in,
                                                                    unsigned char* __restrict__ out, int src_h, int src_w,
                                                                    CropGeom g) {
    const int img = blockIdx.y;
    const long src_bytes = (long)src_h * src_w * 3, dst_px = (long)g.pad_h * g.pad_w;
    const unsigned char* src = in + img * src_bytes;
    unsigned char* dst = out + img * dst_px * 3;
    for (long p = blockIdx.x * (long)kThreads + threadIdx.x; p < dst_px; p += (long)gridDim.x * kThreads) {
        const int y = (int)(p / g.pad_w), x = (int)(p - (long)y * g.pad_w);
        crop_px3(src, src_h, src_w, g, y, x, dst + 3 * p);
    }
}

// Ragged batch: frame i (its own source size and geometry) fills slot i of the [n, canvas_h, canvas_w, 3] canvas from the
// top-left corner; everything beyond its resized area - its padding and the rest of the slot - is zero.
__global__ void __launch_bounds__(kThreads) crop_with_factor_ragged_kernel(const unsigned char* __restrict__ in,
                                                                           unsigned char* __restrict__ out,
                                                                           const RaggedCrop* __restrict__ frames,
                                                                           int canvas_h, int canvas_w) {
    const int img = blockIdx.y;
    const RaggedCrop f = frames[img];
    const long dst_px = (long)canvas_h * canvas_w;
    const unsigned char* src = in + f.src_off;
    unsigned char* dst = out + img * dst_px * 3;
    for (long p = blockIdx.x * (long)kThreads + threadIdx.x; p < dst_px; p += (long)gridDim.x * kThreads) {
        const int y = (int)(p / canvas_w), x = (int)(p - (long)y * canvas_w);
        crop_px3(src, f.src_h, f.src_w, f.g, y, x, dst + 3 * p);
    }
}

// One thread per destination element of the base grid; 16 gathers from the (L1/L2-resident, <= 34 KB) source plane.
__global__ void __launch_bounds__(kThreads) resize_cubic_accum_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                                      long planes, int sh, int sw, int dh, int dw,
                                                                      double step_y, double step_x, int first, float divide_by) {
    const long per = (long)dh * dw, total = planes * per;
    for (long i = blockIdx.x * (long)kThreads + threadIdx.x; i < total; i += (long)gridDim.x * kThreads) {
        const long plane = i / per;
        const int q = (int)(i - plane * per);
        const int y = q / dw, x = q - y * dw;
        const CubCoef cy = rs_cubic_coef(y, sh, step_y), cx = rs_cubic_coef(x, sw, step_x);
        float v = rs_cubic_at(src + plane * (long)sh * sw, sw, 1, cx, cy);
        if (!first) v = __fadd_rn(dst[i], v);
        if (divide_by > 0.f) v = __fdiv_rn(v, divide_by);
        dst[i] = v;
    }
}

}  // namespace

cudaError_t resize_cubic_accum_launch(const float* src, float* dst, long planes, int src_h, int src_w, int dst_h,
                                      int dst_w, int first, float divide_by, cudaStream_t s) {
    if (planes < 1 || src_h < 1 || src_w < 1 || dst_h < 1 || dst_w < 1) return cudaErrorInvalidValue;
    const long total = planes * dst_h * dst_w;
    long b = (total + kThreads - 1) / kThreads;
    if (b > 148L * 8) b = 148L * 8;
    resize_cubic_accum_kernel<<<(unsigned)b, kThreads, 0, s>>>(src, dst, planes, src_h, src_w, dst_h, dst_w,
                                                             rs_step(dst_h, src_h), rs_step(dst_w, src_w), first, divide_by);
    return cudaGetLastError();
}

cudaError_t crop_with_factor_launch(const unsigned char* in, unsigned char* out, int n, int src_h, int src_w,
                                    const CropGeom& g, cudaStream_t s) {
    if (n < 1 || n > 65535) return cudaErrorInvalidValue;
    const long px = (long)g.pad_h * g.pad_w;
    long bx = (px + kThreads - 1) / kThreads;
    const long cap = (148L * 8 + n - 1) / n;      // about one wave of 8 blocks per SM over the whole batch
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    crop_with_factor_kernel<<<dim3((unsigned)bx, (unsigned)n), kThreads, 0, s>>>(in, out, src_h, src_w, g);
    return cudaGetLastError();
}

cudaError_t crop_with_factor_ragged_launch(const unsigned char* in, unsigned char* out, int n, const RaggedCrop* frames,
                                           int canvas_h, int canvas_w, cudaStream_t s) {
    if (n < 1 || n > 65535 || canvas_h < 1 || canvas_w < 1) return cudaErrorInvalidValue;
    const long px = (long)canvas_h * canvas_w;
    long bx = (px + kThreads - 1) / kThreads;
    const long cap = (148L * 8 + n - 1) / n;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    crop_with_factor_ragged_kernel<<<dim3((unsigned)bx, (unsigned)n), kThreads, 0, s>>>(in, out, frames, canvas_h, canvas_w);
    return cudaGetLastError();
}

}  // namespace b2p
