/* b200pose - C ABI of the B200-native OpenPose (rtpose VGG19) inference path.
 *
 * Plain pointers and sizes only; no torch / numpy types.  Every entry point returns 0 on success and a
 * non-zero code on failure (b200pose_last_error() gives the text) unless stated otherwise.
 *
 * Threading: b200pose_last_error() is per thread; a net / post object and the legacy process_paf surface serialise
 * nothing themselves - use one object per host thread (or your own lock).  All work of a call is enqueued on the
 * cuda_stream argument (plus the post object's private second stream for the person assembly and result copies).
 *
 * Each declaration cites the reference interface it replaces (paths relative to /root/reference).
 * The reference-side bindings (ctypes) are shown in INTEGRATION.md.
 */
#ifndef B200POSE_H
#define B200POSE_H

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------------------
 * 0. Library
 * ---------------------------------------------------------------------------------------------------------- */
const char* b200pose_last_error(void);
int b200pose_version(void);
/* Number of CUDA kernels launched by this library since load (the bench's gpu_launches evidence). */
long b200pose_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * 1. Network: replaces rtpose_model.forward                       lib/network/rtpose_vgg.py:158-198
 *    (get_model / make_vgg19_block / make_stages                  lib/network/rtpose_vgg.py:13-56, 60-225)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200pose_net b200pose_net;

#define B200POSE_NUM_TENSORS 184   /* state_dict entries, reference order (model0, model{1..6}_1, model{1..6}_2) */
#define B200POSE_MODE_BF16 0       /* tcgen05 tensor cores, bf16 operands, fp32 accumulate                       */
#define B200POSE_MODE_FP32 1       /* fp32-parity mode: fp32 FMA everywhere (1e-3 bar of BASELINE.json)          */
#define B200POSE_MODE_BF16X3 2     /* high-precision tensor-core mode: value + residual bf16 planes for activations and
                                      weights, 3 MMA terms per K block (A_hi*W_hi + A_hi*W_lo + A_lo*W_hi); measured
                                      1.4e-3 max-abs @368x368 (bf16: 7e-2, fp32 mode: 3e-5) - the tensor core's own fp32
                                      accumulation is the floor, see DESIGN.md 2.3                                   */

int b200pose_net_create(b200pose_net** out, int cuda_device);
void b200pose_net_destroy(b200pose_net* net);
/* Shape of state_dict tensor `index` (weights: 4 dims OIHW, biases: 1 dim); returns number of dims. */
int b200pose_net_tensor_shape(int index, long dims[4]);
/* Copy one fp32 tensor (host memory, OIHW / [O]) into the net.  Replaces load_state_dict(), demo/picture_demo.py:46. */
int b200pose_net_set_tensor(b200pose_net* net, int index, const float* host_data, long count);
/* Pack weights for the device (bf16 K-major slices, padded heads, concat-permuted 7x7 inputs). */
int b200pose_net_finalize(b200pose_net* net);
/* forward: input fp32 NCHW [n,3,H,W] (H, W multiples of 8); outputs[12] fp32 NCHW in saved_for_loss order
 * [paf1, heat1, ..., paf6, heat6] (paf [n,38,H/8,W/8], heat [n,19,H/8,W/8]); entries may be NULL to skip the
 * copy-out.  *_on_device: 0 = host pointers (copies are issued on `cuda_stream` and synchronised before return),
 * 1 = device pointers (asynchronous on `cuda_stream`).  cuda_stream: a cudaStream_t cast to void* (NULL = default).
 * On a real stream (not the legacy default stream, not one that is being captured) the 52 launches of a SMALL-batch
 * (launch-bound: up to 4 frames of 368x368) bf16 / bf16x3 forward pass are captured at the SECOND use of a (shape, mode, input pointer) into a CUDA graph and replayed afterwards
 * (a caller that passes a fresh pointer every time never pays a capture); the input buffer's
 * CONTENTS may change between calls, results are those of plain launches (tests/test_gpu.py:
 * test_graph_replay_equals_plain_launches).  B200POSE_GRAPH=0 disables the capture. */
int b200pose_net_forward(b200pose_net* net, const float* input, int input_on_device, int n, int H, int W, int mode,
                         float* const* outputs, int outputs_on_device, void* cuda_stream);
/* Same, but the input is uint8 HWC BGR frames [n,H,W,3] (what cv2.imread / crop_with_factor produce) and
 * rtpose_preprocess (x/256 - 0.5, HWC -> CHW; lib/datasets/preprocessing.py:16-21, evaluate/coco_eval.py:93-94) is fused
 * into the first convolution's load: 4x less H2D traffic, no fp32 staging. */
int b200pose_net_forward_u8(b200pose_net* net, const unsigned char* images, int input_on_device, int n, int H, int W,
                            int mode, float* const* outputs, int outputs_on_device, void* cuda_stream);
/* Normalisation the uint8 entry points (b200pose_net_forward_u8, b200pose_infer_u8*, b200pose_infer_raw_u8*) fuse into
 * the first convolution: get_outputs' `preprocess` argument (evaluate/coco_eval.py:92-100; functions in
 * lib/datasets/preprocessing.py:16-86).  Default B200POSE_PRE_RTPOSE.  Bit-identical to the numpy functions. */
#define B200POSE_PRE_RTPOSE 1      /* x/256 - 0.5                                   */
#define B200POSE_PRE_VGG 2         /* BGR -> RGB, /255, (x - mean) / std            */
#define B200POSE_PRE_INCEPTION 3   /* BGR -> RGB, x/128 - 1                         */
#define B200POSE_PRE_SSD 4         /* x - (123, 117, 104) on (B, G, R)              */
int b200pose_net_set_preprocess(b200pose_net* net, int preprocess);
/* Ragged batch: n already-cropped uint8 BGR frames of DIFFERENT sizes in one [n,H,W,3] canvas, frame i valid in
 * [0,ext_h[i]) x [0,ext_w[i]) of its slot (top-left corner).  ext_h / ext_w: host arrays of n extents, each a multiple
 * of 8 in [8, H] / [8, W] (H, W: multiples of 8, normally the largest extents).  Canvas bytes outside an extent are not
 * read.  outputs[12] as for b200pose_net_forward_u8, canvas-shaped ([n,C,H/8,W/8]); inside (ext_h[i]/8, ext_w[i]/8)
 * every value is bit-identical to b200pose_net_forward_u8 of frame i alone (same mode), outside it is exactly +0.
 * Every layer still computes the whole canvas: the cost is that of n frames of H x W.  Ragged calls always launch
 * directly (no CUDA graph).  Errors (no fault): null extent arrays, an extent that is not a multiple of 8 or exceeds
 * the canvas, n outside [1, 4096]. */
int b200pose_net_forward_u8_ragged(b200pose_net* net, const unsigned char* canvas, int input_on_device, int n, int H,
                                   int W, const int* ext_h, const int* ext_w, int mode, float* const* outputs,
                                   int outputs_on_device, void* cuda_stream);
/* Measurement hook: re-runs the launch list of the last bf16 forward (conv1_1 + 51 tensor-core launches) with a CUDA
 * event pair around every launch; fills per-launch milliseconds and ALGORITHMIC FLOPs (2 x MACs of the unpadded
 * convolution).  Returns the number of launches, < 0 on error. */
int b200pose_net_profile(b200pose_net* net, float* ms, double* flops, int cap, void* cuda_stream);
/* Device pointers of the last forward's stage-6 maps (NCHW fp32), valid until the next forward. */
int b200pose_net_last_maps(b200pose_net* net, const float** paf, const float** heat, int* n, int* h, int* w);

/* ------------------------------------------------------------------------------------------------------------
 * 2. Post-processing: replaces NMS + paf_to_pose_cpp + pafprocess  lib/utils/paf_to_pose.py:67-145, 372-406
 *                                                                  lib/pafprocess/pafprocess.cpp:22-218
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200pose_post b200pose_post;

#define B200POSE_HUMAN_FLOATS 73   /* score, then 18 x (x, y, peak score, peak id or -1); x, y in input pixels */
/* status bits */
#define B200POSE_ST_PEAK_OVERFLOW 1
#define B200POSE_ST_CAND_OVERFLOW 2
#define B200POSE_ST_ROW_OVERFLOW 4
#define B200POSE_ST_HUMAN_OVERFLOW 8

int b200pose_post_create(b200pose_post** out, int cuda_device, int batch_cap, int peak_cap_per_part, int human_cap);
void b200pose_post_destroy(b200pose_post* post);
/* heat [n,19,h,w], paf [n,38,h,w] (layout 0 = NCHW) or heat [n,h,w,19], paf [n,h,w,38] (layout 1 = NHWC, what
 * get_outputs returns per image, evaluate/coco_eval.py:111-112); fp32, low resolution (stride 8).
 * thresh = cfg.TEST.THRESH_HEATMAP.  Results stay on the device until fetched. */
int b200pose_post_run(b200pose_post* post, const float* heat, const float* paf, int on_device, int layout, int n, int h,
                      int w, float thresh, void* cuda_stream);
/* Every run copies its results (person rows, counts, status) to pinned host memory by itself, on a second stream right
 * after the person assembly, into one of two slots (run parity) - so a caller may submit run i+1 before reading run i
 * (at most two runs in flight).  The getters below read the selected slot.
 *   b200pose_post_last_ticket : ticket (0-based index) of the most recently submitted run, -1 if none
 *   b200pose_post_select      : block until run `ticket` is on the host and make the getters read it
 *   b200pose_post_sync        : select(last ticket) */
long b200pose_post_last_ticket(b200pose_post* post);
int b200pose_post_select(b200pose_post* post, long ticket);
int b200pose_post_sync(b200pose_post* post);
/* Diagnostics: out[0..2] = max SM cycles of the limbs kernel phases (scoring, exact sort, greedy) over all blocks since
 * the last reset, out[3] = max candidates of a limb, out[4] = total candidates. */
int b200pose_post_debug(b200pose_post* post, unsigned long long* out, int n, int reset);
/* Test hook: sorts n 64-bit candidate keys (high word = ~score bits, low word = pair index) on the device with the
 * product's sorting kernels - libstdc++'s std::sort order (pafprocess.cpp:97), ties included.  Host pointers. */
int b200pose_post_debug_sort(b200pose_post* post, const unsigned long long* keys, int n, unsigned long long* out);
/* OR of the status words of every image of every run since the last reset (sticky accumulator kept on the device):
 * with runs in flight a caller reads only some results back; this proves that no run at all overflowed a capacity
 * (the reference's std::vectors grow without bound, pafprocess.cpp:24-44, so an overflow is a divergence).  < 0 on error. */
int b200pose_post_status_accum(b200pose_post* post, int reset);
int b200pose_post_num_humans(b200pose_post* post, int img);             /* < 0 on error */
int b200pose_post_status(b200pose_post* post, int img);                 /* status bits of the last run */
int b200pose_post_get_humans(b200pose_post* post, int img, float* out, int max_humans);   /* returns count */
/* joint list rows (x, y, score, id, part), the array paf_to_pose.py:376-378 builds; returns count */
int b200pose_post_get_peaks(b200pose_post* post, int img, float* out, int max_peaks);

/* ------------------------------------------------------------------------------------------------------------
 * 3. Fused path: net forward + post-processing without leaving the device (the batched entry point of
 *    SURVEY.md 8b).  input: fp32 NCHW [n,3,H,W].
 * ---------------------------------------------------------------------------------------------------------- */
int b200pose_infer(b200pose_net* net, b200pose_post* post, const float* input, int input_on_device, int n, int H, int W,
                   int mode, float thresh, void* cuda_stream);

int b200pose_infer_u8(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device, int n,
                      int H, int W, int mode, float thresh, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------------------
 * 3b. Flip test-time averaging: replaces handle_paf_and_heat        evaluate/coco_eval.py:197-242
 *     out = (normal + mirror_W(flipped)[left/right-swapped channels, PAF x components negated]) / 2, bit-identical to
 *     the reference's float32 arithmetic.  Unlike the reference it does not modify flipped_paf in place.
 *     All six pointers are host (on_device = 0; copies on `cuda_stream`, synchronised before return) or device (1,
 *     asynchronous); layout 0 = [n,C,h,w], 1 = [n,h,w,C] (what get_outputs returns per image), C = 19 / 38.
 *     `post` provides the device and the staging buffers.
 * ---------------------------------------------------------------------------------------------------------- */
int b200pose_flip_merge(b200pose_post* post, const float* normal_heat, const float* flipped_heat,
                        const float* normal_paf, const float* flipped_paf, int on_device, int layout, int n, int h, int w,
                        float* out_heat, float* out_paf, void* cuda_stream);
/* Fused flip-TTA inference: the n frames and their W-mirrored copies (made on the device) run through the network as
 * one 2n batch, the two map sets are merged as above and the fused post-processing runs on the averaged maps; nothing
 * leaves the device but the person rows.  Equivalent to get_outputs(img) + get_outputs(img[:, ::-1]) +
 * handle_paf_and_heat + paf_to_pose_cpp for frames that need no padding in W (a padded frame must be mirrored before
 * crop_with_factor pads it: use b200pose_net_forward on both orientations + b200pose_flip_merge instead).
 * Results are fetched exactly like b200pose_infer's. */
int b200pose_infer_flip(b200pose_net* net, b200pose_post* post, const float* input, int input_on_device, int n, int H,
                        int W, int mode, float thresh, void* cuda_stream);
int b200pose_infer_u8_flip(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device,
                           int n, int H, int W, int mode, float thresh, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------------------
 * 3c. Device-side crop_with_factor: replaces crop_with_factor / _factor_closest   lib/network/im_transform.py:113-134
 *     (called by get_outputs, evaluate/coco_eval.py:87-91, with dest_size = cfg.DATASET.IMAGE_SIZE, factor =
 *     cfg.MODEL.DOWNSAMPLE, is_ceil = True).  uint8 HWC BGR frames of ONE source size (a video stream, or one shape
 *     bucket of a data set) -> cv2.resize(fx = fy = dest_size / min(h, w)) with OpenCV's 8-bit INTER_LINEAR arithmetic,
 *     bit for bit (csrc/resize_core.h) -> zero padding bottom/right to a multiple of `factor` (a multiple of 8).
 *   b200pose_crop_geometry         : host only; the values crop_with_factor returns / implies
 *   b200pose_net_crop_with_factor  : images [n,src_h,src_w,3] -> out [n,pad_h,pad_w,3]; host or device pointers
 *   b200pose_infer_raw_u8          : raw frames -> resize/pad -> network -> fused post-processing, all on the device;
 *                                    flip != 0 adds left/right flip test-time averaging: the RAW frame is mirrored
 *                                    before it is resized and padded, exactly like get_outputs(img[:, ::-1]) would see
 *                                    it, then the maps are merged as handle_paf_and_heat does.
 *     Person coordinates are in pixels of the padded frame (pad_h x pad_w), like the reference's.
 * ---------------------------------------------------------------------------------------------------------- */
int b200pose_crop_geometry(int src_h, int src_w, int dest_size, int factor, double* im_scale, int* res_h, int* res_w,
                           int* pad_h, int* pad_w);
int b200pose_net_crop_with_factor(b200pose_net* net, const unsigned char* images, int images_on_device, int n, int src_h,
                                  int src_w, int dest_size, int factor, unsigned char* out, int out_on_device,
                                  void* cuda_stream);
int b200pose_infer_raw_u8(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device, int n,
                          int src_h, int src_w, int dest_size, int factor, int mode, float thresh, int flip,
                          void* cuda_stream);
/* Ragged batch of raw frames of different sizes: frame i is [src_h[i],src_w[i],3] uint8 BGR, the frames packed back to
 * back in `frames` (frame i starts at byte sum_{j<i} 3 src_h[j] src_w[j]; host or device).  Each frame gets its own
 * crop_with_factor(dest_size, factor) as in b200pose_infer_raw_u8, all n then run through the network and the fused
 * post-processing as ONE batch on a canvas of the largest padded height x the largest padded width.  Person rows of
 * frame i equal those of b200pose_infer_raw_u8 on frame i alone, in pixels of frame i's own padded frame.  Results are
 * fetched like b200pose_infer's (tickets, two runs in flight); a host input stays alive until then.  No flip.
 * Errors (no fault): null pointers, n < 1 or n > the post's batch_cap, a frame size crop_with_factor rejects. */
int b200pose_infer_raw_u8_ragged(b200pose_net* net, b200pose_post* post, const unsigned char* frames,
                                 int input_on_device, int n, const int* src_h, const int* src_w, int dest_size,
                                 int factor, int mode, float thresh, void* cuda_stream);
/* Host only: the layout b200pose_infer_raw_u8_ragged gives n raw frames - per frame its byte offset in the packed input
 * (src_off[n]) and its padded size (pad_h[n], pad_w[n], as b200pose_crop_geometry reports for it alone), and the canvas
 * (largest pad_h x largest pad_w).  Errors: null pointers, n < 1, a frame size crop_with_factor rejects. */
int b200pose_ragged_layout(int n, const int* src_h, const int* src_w, int dest_size, int factor, long* src_off,
                           int* pad_h, int* pad_w, int* canvas_h, int* canvas_w);

/* Multi-scale (+ flip) test-time averaging, BASELINE.json configs[4].  The reference at this commit has no multi-scale
 * loop (get_outputs is single-scale, evaluate/coco_eval.py:87-91); the protocol is composed from its own functions:
 * for every scale s: crop_with_factor(img, int(base_size * s), factor) -> network (-> handle_paf_and_heat with the
 * mirrored RAW frame when flip != 0) -> bicubic resize of the 57 maps to the grid of base_size (OpenCV INTER_CUBIC
 * formula, csrc/resize_core.h) -> running float32 sum; average = sum / n_scales; fused post-processing on the average.
 * oracle/glue_port.py::multi_scale_maps restates exactly this composition. */
int b200pose_infer_raw_u8_multiscale(b200pose_net* net, b200pose_post* post, const unsigned char* images,
                                     int input_on_device, int n, int src_h, int src_w, int base_size, int factor,
                                     const double* scales, int n_scales, int mode, float thresh, int flip,
                                     void* cuda_stream);

/* ------------------------------------------------------------------------------------------------------------
 * 4. Legacy SWIG surface of lib/pafprocess (pafprocess.h:53-59, pafprocess.i:14): same names, same argument
 *    meaning; state is kept in a process-global context exactly like the reference's file-scope globals
 *    (pafprocess.cpp:12-13).  peaks [p1,p2,5] rows (x, y, score, id, part) sorted by part as paf_to_pose_cpp
 *    builds them; heatmap is not dereferenced (only h1 is used, pafprocess.cpp:83); pafmap [f1,f2,f3] is the
 *    x8 nearest-upsampled HWC array.  process_paf returns 0 like the reference, or a non-zero code if the
 *    device path failed (the reference has no failure mode).
 * ---------------------------------------------------------------------------------------------------------- */
int process_paf(int p1, int p2, int p3, float* peaks, int h1, int h2, int h3, float* heatmap, int f1, int f2, int f3,
                float* pafmap);
int get_num_humans(void);
int get_part_cid(int human_id, int part_id);
float get_score(int human_id);
int get_part_x(int cid);
int get_part_y(int cid);
float get_part_score(int cid);

#ifdef __cplusplus
}
#endif
#endif
