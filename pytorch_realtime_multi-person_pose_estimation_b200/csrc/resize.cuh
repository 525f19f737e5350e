// crop_with_factor on the device (SURVEY.md 8(f) rank 1):  /root/reference/lib/network/im_transform.py:113-134
// uint8 HWC BGR frames of one source size -> bilinear resize (OpenCV INTER_LINEAR arithmetic, resize_core.h) so that
// the short side is dest_size -> zero padding bottom/right to a multiple of `factor`.
#pragma once
#include <cuda_runtime.h>

#include "resize_core.h"

namespace b2p {

// in [n, src_h, src_w, 3] -> out [n, g.pad_h, g.pad_w, 3], both on the device
cudaError_t crop_with_factor_launch(const unsigned char* in, unsigned char* out, int n, int src_h, int src_w,
                                    const CropGeom& g, cudaStream_t s);

// Ragged batch of raw frames of different sizes, packed back to back: frame i starts at byte src_off and has its own
// geometry (crop_geometry of its size).  out [n, canvas_h, canvas_w, 3]: frame i resized and padded exactly as
// crop_with_factor_launch does it, in the top-left corner of slot i, zeros elsewhere.  `frames` is a device array.
struct RaggedCrop {
    CropGeom g;
    long src_off;
    int src_h, src_w;
};
cudaError_t crop_with_factor_ragged_launch(const unsigned char* in, unsigned char* out, int n, const RaggedCrop* frames,
                                           int canvas_h, int canvas_w, cudaStream_t s);

// Bicubic resize of `planes` float32 planes [src_h, src_w] -> [dst_h, dst_w] (resize_core.h: rs_cubic_at), fused with
// the running sum of the multi-scale average: dst = first ? r : dst + r, then dst /= divide_by when divide_by > 0.
cudaError_t resize_cubic_accum_launch(const float* src, float* dst, long planes, int src_h, int src_w, int dst_h,
                                      int dst_w, int first, float divide_by, cudaStream_t s);

}  // namespace b2p
