/*
 * vsr_b200.h -- C ABI of libvsr_b200.so, the B200 (sm_100a) implementation of the
 * per-frame warp-and-fuse hot path of PlanNoa/video_super_resolution.
 *
 * This header is the drop-in boundary.  Every entry point
 *   - takes raw DEVICE pointers, plain sizes and an explicit CUDA stream (passed as void*,
 *     i.e. a cudaStream_t / CUstream); no ATen / torch types cross it;
 *   - never allocates, frees or synchronises: outputs and workspaces are caller-allocated
 *     (the reference convention, resample2d.py:17-19, channelnorm.py:12);
 *   - returns 0 on success, VSR_ERR_* (<1000) for argument errors and 1000+cudaError_t
 *     for CUDA failures (the reference returns a constant 1 and drops CUDA errors,
 *     resample2d_cuda.cc:12,23 -- see INTEGRATION.md for the binding a maintainer adds).
 *
 * "ref:" comments cite the interface of /root/reference that each function replaces.
 * Layout names: NCHW = reference layout (resample2d.py:10-11), NHWC = channels-last pixels
 * as produced by the reference's video loader (utils/video_utils.py:23).
 */
#ifndef VSR_B200_H_
#define VSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSR_OK 0
#define VSR_ERR_INVALID_ARG 1   /* null pointer, non-positive size, unsupported option   */
#define VSR_ERR_UNSUPPORTED 2   /* shape/geometry outside what the kernels implement      */
#define VSR_ERR_WORKSPACE 3     /* caller workspace too small                             */
#define VSR_ERR_STATE 4         /* plan used before weights were loaded, etc.             */
#define VSR_ERR_CUDA_BASE 1000  /* 1000 + cudaError_t                                      */

typedef void* vsr_stream_t; /* cudaStream_t */

/* Library identification / launch accounting (bench.py's gpu_launches). */
const char* vsr_version(void);
/* number of kernels this library launched in the calling process since load/reset */
uint64_t vsr_launch_count(void);
void vsr_launch_count_reset(void);
/* human readable text for a VSR error code (static storage) */
const char* vsr_error_string(int code);

/* ------------------------------------------------------------------------------------------
 * a3 / a4: the pinned warp.  ref: resample2d_cuda.cc:6-13 `resample2d_cuda_forward(input1,
 * input2, output, kernel_size, bilinear)` -> resample2d_kernel.cu:15-72,200-242.
 * input1 (B,C,H,W) f32, flow (B,2,H,W) f32 (channel 0 horizontal), output (B,C,H,W) f32, all
 * NCHW contiguous.  Arithmetic is the reference's, bit for bit: fp32 coordinates, border-clamped
 * taps, tap weights formed in double, per-tap products rounded to fp32 and summed TL,TR,BL,BR.
 * kernel_size 1 is the only value the reference uses (resample2d.py:44); 2..16 follow resample2d_kernel.cu:54-61: the
 * four taps are summed again at every offset of a kernel_size x kernel_size window, un-normalised, with the
 * reference's un-clamped NCHW address arithmetic (an offset past a row / plane end reads the next row / plane);
 * addresses past the end of the tensor, where the reference reads out of bounds, are pinned to its last element.
 * ---------------------------------------------------------------------------------------- */
int vsr_resample2d_forward(const float* input1, const float* flow, float* output,
                           int B, int C, int H, int W, int kernel_size, int bilinear,
                           vsr_stream_t stream);

/* Channels-last variant used by the pipeline (frames C=3, features C=32).  src/dst (B,H,W,C)
 * f32, flow (B,H,W,2) f32.  If norm_out != NULL it additionally receives, per pixel,
 * sqrt(sum_c (ref[b,y,x,c] - dst[b,y,x,c])^2) with fp32 accumulation, i.e. the reference's
 * `channelnorm(img - resampled)` (models.py:86-88) fused into the warp; `ref` may be NULL iff
 * norm_out is NULL.  `bilinear`: 0 = nearest, 1 = the reference's arithmetic bit for bit (as
 * vsr_resample2d_forward), 2 = fast: same taps / border rule with fp32 FMA weights (differs from
 * mode 1 by a few fp32 ulps, <= 1e-4 on 0..255 data; no fp64 conversions, the pipeline default). */
int vsr_warp_nhwc_f32(const float* src, const float* flow, float* dst,
                      const float* ref, float* norm_out,
                      int B, int H, int W, int C, int bilinear, vsr_stream_t stream);

/* The neighbour warp of `windows` independent frame windows in a single launch (1..65535; one window is windows = 1),
 * without a gathered copy of the frames: frames (windows,T,H,W,3) f32 NHWC; flows (windows,T-1,H,W,2) f32, one field
 * per NEIGHBOUR in frame order with the centre frame left out, each mapping centre coordinates to that neighbour;
 * warped (windows,T-1,H,W,3); resid (windows,T-1,H,W) or NULL = per-pixel L2 norm of (frames[centre] - warped[n])
 * (models.py:86-88 fused).  Window b is warped to its own centre frame, bit-identical to a call on it alone.
 * Arithmetic and `bilinear` modes as vsr_warp_nhwc_f32. */
int vsr_warp_windows_nhwc3(const float* frames, const float* flows, float* warped, float* resid, int windows,
                           int T, int centre, int H, int W, int bilinear, vsr_stream_t stream);

/* Flow composition out(p) = g(p) + f(p + g(p)) with f sampled bilinearly (the warp's taps and border rule,
 * fp32 blend): if g maps image A to B and f maps B to C, out maps A to C.  Used to chain adjacent-pair flows into
 * centre -> neighbour flows for windows longer than 3 frames.  One link of the chains of `windows` frame windows in one
 * launch (1..65535): window b composes the (H,W,2) f32 fields at g + b*stride and f + b*stride into out + b*stride
 * (stride in floats, even; it may be 0 when windows = 1).  The centre -> neighbour fields of a (windows,T-1,H,W,2)
 * array are (T-1)*H*W*2 floats apart.  g == NULL is the identity field: out = f (the first link of a chain). */
int vsr_compose_flow_windows(const float* g, const float* f, float* out, int windows, int64_t stride, int H, int W,
                             vsr_stream_t stream);

/* Nearest-neighbour label/mask warp on u8 (north star "VOSProjection: mask/label warping"),
 * ref arithmetic: resample2d_kernel.cu:65-70 (floor(xf + 0.5) in double, border clamp).
 * labels/dst (B,H,W) u8, flow (B,H,W,2) f32.  Bit-exact. */
int vsr_warp_labels_u8(const uint8_t* labels, const float* flow, uint8_t* dst,
                       int B, int H, int W, vsr_stream_t stream);
/* `windows` label images (windows,H,W) -> dst (windows,H,W) in one launch (1..65535); window b is warped along the
 * (H,W,2) field at flow + b*flow_stride (floats, even; it may be 0 when windows = 1). */
int vsr_warp_labels_u8_windows(const uint8_t* labels, const float* flow, uint8_t* dst, int windows,
                               int64_t flow_stride, int H, int W, vsr_stream_t stream);

/* ref: channelnorm_cuda.cc `channelnorm_cuda_forward(input1, output, norm_deg)` ->
 * channelnorm_kernel.cu:19-60.  input (B,C,H,W) f32 NCHW, output (B,1,H,W).  norm_deg is accepted
 * and ignored exactly as the reference does (channelnorm_kernel.cu:53-59). */
int vsr_channelnorm_forward(const float* input, float* output, int B, int C, int H, int W,
                            int norm_deg, vsr_stream_t stream);

/* The other two dtypes of the reference's AT_DISPATCH_FLOATING_TYPES_AND_HALF (channelnorm_kernel.cu:111,152): fp16 and
 * fp64 tensors, forward and backward, with the reference's arithmetic (square in the tensor's type, fp32 sum and sqrt,
 * result cast back).  dtype: VSR_DTYPE_*; VSR_DTYPE_F32 forwards to the fp32 entry points. */
#define VSR_DTYPE_F32 0
#define VSR_DTYPE_F16 1
#define VSR_DTYPE_F64 2
int vsr_channelnorm_forward_typed(const void* input, void* output, int B, int C, int H, int W, int norm_deg, int dtype,
                                  vsr_stream_t stream);
int vsr_channelnorm_backward_typed(const void* input, const void* output, const void* grad_output, void* grad_input,
                                   int B, int C, int H, int W, int norm_deg, int dtype, vsr_stream_t stream);

/* Backward passes of the two autograd Functions (SURVEY.md 8f rank 2).
 * ref: resample2d_cuda.cc:14-26 `resample2d_cuda_backward(input1, input2, gradOutput, gradInput1,
 * gradInput2, kernel_size, bilinear)` -> resample2d_kernel.cu:75-198,244-323; channelnorm_cuda.cc
 * `channelnorm_cuda_backward(input1, output, gradOutput, gradInput1, norm_deg)` ->
 * channelnorm_kernel.cu:64-96.  All tensors NCHW f32 contiguous.  grad_input1 must be ZERO on entry
 * (the reference's caller allocates it with .zero_(), resample2d.py:32): the 4-tap scatter adds into
 * it with atomics, so it is deterministic only up to fp32 summation order; grad_input2 and the
 * channel-norm gradient are bit-identical to the reference binary. */
int vsr_resample2d_backward(const float* input1, const float* flow, const float* grad_output,
                            float* grad_input1, float* grad_input2,
                            int B, int C, int H, int W, int kernel_size, int bilinear, vsr_stream_t stream);
int vsr_channelnorm_backward(const float* input, const float* output, const float* grad_output,
                             float* grad_input, int B, int C, int H, int W, int norm_deg, vsr_stream_t stream);
/* Deterministic variant of vsr_resample2d_backward: grad_input1 is bit-identical to oracle/oracle.c
 * or_resample2d_backward (fp32 sums of w*g in row-major source order, taps TL, TR, BL, BR), so it is the same on
 * every run; grad_input2 comes from the same kernel as above.  Every element of grad_input1 is written (any contents on
 * entry).  workspace: vsr_resample2d_backward_deterministic_workspace_bytes(B,H,W) bytes of device memory (any
 * contents, 16-byte aligned).  kernel_size must be 1 (VSR_ERR_UNSUPPORTED otherwise, and for B*H*W >= 2^32).  The
 * scatter is turned into a gather (stable radix sort of the sources by their top-left tap, then one thread per
 * target): a target that many sources reach -- every out-of-image sample is clamped to a border pixel -- sums them
 * in sequence on one thread. */
size_t vsr_resample2d_backward_deterministic_workspace_bytes(int B, int H, int W);
int vsr_resample2d_backward_deterministic(const float* input1, const float* flow, const float* grad_output,
                                          float* grad_input1, float* grad_input2, int B, int C, int H, int W,
                                          int kernel_size, int bilinear, void* workspace, size_t workspace_bytes,
                                          vsr_stream_t stream);

/* FlowNetC cost volume (SURVEY.md 8f rank 1; outside the warp-and-fuse hot path).
 * ref: correlation_cuda.cc:10-86 `correlation_forward_cuda(input1, input2, rInput1, rInput2, output,
 * pad_size, kernel_size, max_displacement, stride1, stride2, corr_type_multiply)` ->
 * correlation_cuda_kernel.cu:46-147.  input1/input2 (B,C,H,W) f32 NCHW; output (B, D*D, outH, outW)
 * f32 with D = 2*(max_displacement/stride2)+1 and outH/outW from vsr_correlation_output_shape (the
 * reference resizes `output` itself; here the caller allocates, as everywhere in this ABI).  No
 * padded NHWC copies (`rInput1/2`) are needed.  fp32 results agree with the reference to fp32
 * summation order (tested <= 1e-5 relative).  Positions outside the image are zeros for any pad_size;
 * the reference is only defined for pad_size >= max_displacement + (kernel_size-1)/2 (with less it
 * indexes outside its padded copies). */
int vsr_correlation_output_shape(int C, int H, int W, int pad_size, int kernel_size, int max_displacement,
                                 int stride1, int stride2, int* out_channels, int* out_h, int* out_w);
int vsr_correlation_forward(const float* input1, const float* input2, float* output, int B, int C, int H, int W,
                            int pad_size, int kernel_size, int max_displacement, int stride1, int stride2,
                            int corr_multiply, vsr_stream_t stream);
/* Backward of the cost volume (completes CorrelationFunction, correlation.py:32-47): replaces
 * correlation_cuda.backward = correlation_backward_cuda(input1, input2, rInput1, rInput2, gradOutput, gradInput1,
 * gradInput2, ...) correlation_cuda.cc:89-166 -> correlation_cuda_kernel.cu:148-333.  grad_output (B, D*D, outH, outW),
 * grad_input1/2 (B,C,H,W), all f32; every element of the gradients is written (no pre-zeroing needed).  stride1 must
 * be 1 (VSR_ERR_UNSUPPORTED otherwise: the reference's kernels write out of bounds for stride1 > 1). */
int vsr_correlation_backward(const float* input1, const float* input2, const float* grad_output,
                             float* grad_input1, float* grad_input2, int B, int C, int H, int W, int pad_size,
                             int kernel_size, int max_displacement, int stride1, int stride2, int corr_multiply,
                             vsr_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a1 / a2: flow projection (forward splat + count + normalise + hole fill), SURVEY.md App. B.
 * ref surface: FlowProjectionModule.forward (FlowProjectionModule.py:18-33) and
 * DepthProjectionModule.forward (DepthProjectionModule.py:12-18); the splat body itself has no
 * reference implementation (parity unpinned, oracle/oracle.c is the contract).
 * flow (B,h,w,2) f32; inv_depth (B,h,w) f32 > 0 or NULL (NULL = unweighted FlowProjection);
 * outputs: proj (B,h,w,2) f32, wsum (B,h,w) f32 or NULL, count (B,h,w) i32, hole (B,h,w) u8.
 * workspace: vsr_flow_projection_workspace_bytes(B,h,w) bytes of device memory (any contents).
 * count / hole are bit-exact; proj / wsum are fp32 sums in nondeterministic order.
 * A target counts as a hole when nothing hit it OR when its hits carry no positive weight (sum of inverse
 * depths <= 0 or NaN): it is then filled from its neighbours like any other hole instead of dividing by zero.
 * This entry point makes no assumption about the flow (config C3's +-64 px): atomic scatter into an L2-resident
 * cell array, the stages of successive images pipelined inside one cooperative persistent kernel.
 *
 * vsr_flow_projection_forward_bounded: the caller additionally PROMISES |fx|, |fy| <= max_disp for every pixel
 * (the smooth fields of configs C2/C4/C5: 8 px).  For 0 <= max_disp <= 8 (and an even w) the batch runs through
 * shared-memory tiles (target tile + halo, owner-computes accumulation without atomics, one coalesced pass out).  A
 * broken promise (a component beyond 8 px) is detected on the device and the batch is redone by the general path: the
 * result never depends on the promise, only the speed does.  Any other max_disp (negative, NaN, > 8) selects the
 * general path directly.
 * ---------------------------------------------------------------------------------------- */
size_t vsr_flow_projection_workspace_bytes(int B, int h, int w);
int vsr_flow_projection_forward(const float* flow, const float* inv_depth,
                                float* proj, float* wsum, int32_t* count, uint8_t* hole,
                                void* workspace, size_t workspace_bytes,
                                int B, int h, int w, vsr_stream_t stream);
int vsr_flow_projection_forward_bounded(const float* flow, const float* inv_depth,
                                        float* proj, float* wsum, int32_t* count, uint8_t* hole,
                                        void* workspace, size_t workspace_bytes,
                                        int B, int h, int w, float max_disp, vsr_stream_t stream);
/* Deterministic projection: proj, wsum, count and hole are bit-identical to oracle/oracle.c or_flow_projection --
 * for every target the fp32 contributions of its sources are added in fp64 in row-major source order, then rounded
 * and divided in fp32 -- so they are the same on every run, whatever the flow.  Same arguments as
 * vsr_flow_projection_forward; workspace: vsr_flow_projection_deterministic_workspace_bytes(B,h,w) bytes (any contents,
 * 16-byte aligned; the images are processed one after another and share it).  Slower than the default paths: a stable
 * radix sort of the sources by cell, then one thread per target merging its four cells' lists. */
size_t vsr_flow_projection_deterministic_workspace_bytes(int B, int h, int w);
int vsr_flow_projection_forward_deterministic(const float* flow, const float* inv_depth,
                                              float* proj, float* wsum, int32_t* count, uint8_t* hole,
                                              void* workspace, size_t workspace_bytes,
                                              int B, int h, int w, vsr_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a5: VOS mask arithmetic.  ref: VOSProjectionModule.py:22-25 (sigmoid(a)+sigmoid(b) > 0.7),
 * utils/tools.py:76-77 (maskprocess) and network/video_super_resolution.py:58-60
 * (MaskedArray(img, mask, fill_value=0).filled()).
 * vsr_vos_threshold_windows: `windows` logit pairs in one launch (one window is windows = 1):
 * logits_a/logits_b (windows,h,w) f32 -> mask (windows,h,w) u8 in {0,1}.
 * vsr_mask_fill: image (C,h,w) f32 -> masked (C,h,w) f32 = image where mask==0 else 0.
 * ---------------------------------------------------------------------------------------- */
int vsr_vos_threshold_windows(const float* logits_a, const float* logits_b, uint8_t* mask,
                              int windows, int h, int w, vsr_stream_t stream);
int vsr_mask_fill(const float* image, const uint8_t* mask, float* masked,
                  int C, int h, int w, vsr_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a7: assembly of the (M,3,h,w) map stack, M = 3T-1.  ref: network/video_super_resolution.py:33-40
 * (transpose1323 + interpolate + torch.cat) and :43-44,:57-62 (nearest downsize of the first-pass
 * output, MaskedArray fill with the VOS mask, second cat).  Stack order along dim 0
 * (video_super_resolution.py:40 generalised to T frames): T frames (warped neighbours, the centre
 * frame at centre_idx), T-1 flow maps (projected fx, projected fy, warp-residual norm), T-1 depth
 * maps tiled x3 (utils/tools.py:76-77), 1 estimate.
 * Both entry points take `windows` frame windows in one launch (1..65535; one window is windows = 1), window b
 * bit-identical to a call on it alone.
 * vsr_assemble_stack_windows: warped (windows,T-1,h,w,3) NHWC, proj (windows,T-1,h,w,2), resid / depth
 * (windows,T-1,h,w), estimate (windows,3,h,w) NCHW or NULL, stack (windows,M,3,h,w).  The centre frame and the
 * fallback frame of window b are the (h,w,3) NHWC images at centre + b*frame_stride and fallback + b*frame_stride
 * (floats; it may be 0 when windows = 1).  For frames (windows,T,h,w,3), frame_stride = T*h*w*3, and centre / fallback
 * point at frame centre_idx / 0 of window 0.  Without an estimate the slot receives the fallback frame: LR frame 0 of
 * the window (video_super_resolution.py:37-38 `else data_clone[0:1]`).
 * vsr_estimate_slot_windows: slot (3,h,w) = mask ? 0 : hr[:, y*scale, x*scale] for hr (windows,3,h*scale,w*scale) and
 * mask (windows,h,w) u8 or NULL.  The slot of window b is the (3,h,w) image at slot + b*slot_stride (floats; it may be
 * 0 when windows = 1).  For the estimate slots of a (windows,M,3,h,w) stack, slot = map M-1 of window 0 and
 * slot_stride = M*3*h*w.
 * ---------------------------------------------------------------------------------------- */
int vsr_assemble_stack_windows(const float* warped, const float* centre, const float* proj, const float* resid,
                               const float* depth, const float* estimate, const float* fallback, float* stack,
                               int windows, int64_t frame_stride, int T, int centre_idx, int h, int w,
                               vsr_stream_t stream);
int vsr_estimate_slot_windows(const float* hr, const uint8_t* mask, float* slot, int windows, int64_t slot_stride,
                              int h, int w, int scale, vsr_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md 8f rank 3: flow colour coding + resize glue on the device.
 * ref: utils/flow_utils.py:4-24 (flow2img), :27-61, :64-112; FlowProjectionModule.py:31-32 (the reference
 * colour-codes on the host: .cpu().numpy() -> flow2img -> torch.tensor(...).cuda());
 * network/video_super_resolution.py:35,52 (transpose1323 + F.interpolate, default nearest).
 * flow (h,w,2) f32 -> img_u8 (h,w,3) u8 Middlebury colour code (NULL to skip) and/or
 * planes (3,out_h,out_w) f32 = the same image transposed to CHW and nearest-resized (NULL to skip).
 * The normalisation is a global max of the flow magnitude (flow_utils.py:14-15), so it is one flow
 * map per call.  workspace: >= 8 bytes of device memory, 4-byte aligned.  NumPy >= 2 promotion rules
 * (fp32 up to the normalising division, float64 after `+ eps`), see tests/golden/flow2img.npz.
 * ---------------------------------------------------------------------------------------- */
int vsr_flow_to_image(const float* flow, int h, int w, uint8_t* img_u8, float* planes, int out_h,
                      int out_w, void* workspace, vsr_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a6 / a7: the fusion / upsampling convolutions (SRFBN + per-pixel fc over the map axis).
 * ref: SRProjectionModule.forward (SRProjectionModule.py:133-147), FeedbackBlock (:7-93),
 * blocks.py:7-74, with the INTENDED dense-concat dataflow (SURVEY.md Appendix C).
 *
 * A plan owns nothing on the device: weights live in a caller buffer that
 * vsr_srfbn_pack_weights fills, activations in a caller workspace.
 * Geometry: x4 (k=8,s=4,p=2, the reference's only one, SRProjectionModule.py:101-103) or x2
 * (k=6,s=2,p=2, SRFBN's x2 geometry -- BASELINE config C4; the reference has no x2 code, SURVEY.md 8 a6);
 * num_features=32, num_groups=6, num_steps>=1, M stacked maps (reference: 8).
 * ---------------------------------------------------------------------------------------- */
typedef struct vsr_srfbn_plan vsr_srfbn_plan;

typedef struct vsr_srfbn_config {
  int32_t num_maps;      /* M: maps stacked along dim 0 (video_super_resolution.py:40), fc in-features */
  int32_t h, w;          /* LR size; output is (upscale*h, upscale*w)                            */
  int32_t num_steps;     /* SRProjectionModule num_steps (default 3)                             */
  int32_t num_groups;    /* must be 6                                                            */
  int32_t num_features;  /* must be 32                                                           */
  int32_t upscale;       /* 4 or 2                                                               */
} vsr_srfbn_config;

/* Host-side weights in the reference's state-dict layout (SURVEY.md Appendix C), fp32, host
 * memory.  Arrays indexed by group.  PReLU slopes are single floats (blocks.py:70-71). */
typedef struct vsr_srfbn_weights {
  const float* sub_mean_bias;      /* (3)   MeanShift bias, weight is identity (blocks.py:46-55)  */
  const float* add_mean_bias;      /* (3)                                                         */
  const float* conv_in_w;          /* (128,3,3,3)  */
  const float* conv_in_b;          /* (128)        */
  float conv_in_slope;
  const float* feat_in_w;          /* (32,128,1,1) */
  const float* feat_in_b;
  float feat_in_slope;
  const float* compress_in_w;      /* (32,64,1,1)  */
  const float* compress_in_b;
  float compress_in_slope;
  const float* up_w[6];            /* ConvTranspose (32 in,32 out,8,8); x2: (32,32,6,6) */
  const float* up_b[6];
  float up_slope[6];
  const float* down_w[6];          /* Conv (32 out,32 in,8,8); x2: (32,32,6,6) */
  const float* down_b[6];
  float down_slope[6];
  const float* uptran_w[5];        /* (32,32*(i+2),1,1), i=0..4 */
  const float* uptran_b[5];
  float uptran_slope[5];
  const float* downtran_w[5];
  const float* downtran_b[5];
  float downtran_slope[5];
  const float* compress_out_w;     /* (32,192,1,1) */
  const float* compress_out_b;
  float compress_out_slope;
  const float* out_w;              /* ConvTranspose (32,32,8,8); x2: (32,32,6,6) */
  const float* out_b;
  float out_slope;
  const float* conv_out_w;         /* (3,32,3,3), no activation */
  const float* conv_out_b;
  const float* fc0_w;              /* (32,M) */
  const float* fc0_b;              /* (32)   */
  const float* fc2_w;              /* (1,32) */
  const float* fc2_b;              /* (1)    */
} vsr_srfbn_weights;

int vsr_srfbn_plan_create(const vsr_srfbn_config* cfg, vsr_srfbn_plan** out_plan);
void vsr_srfbn_plan_destroy(vsr_srfbn_plan* plan);
/* Optional, before vsr_srfbn_bind: cap the activation workspace.  The M stacked maps are independent until the per-pixel
 * fc fuse, so the plan then sweeps its layers over chunks of `vsr_srfbn_chunk_maps` maps (the largest divisor of M whose
 * workspace fits under the cap); results are bit-identical to the unchunked plan.  cap_bytes == 0 removes the cap.
 * VSR_ERR_WORKSPACE if not even one map at a time fits (the chunk and workspace are then unchanged, but the cap stays
 * set and holds for the setters after it); VSR_ERR_STATE after bind.  (Config C4 unchunked: 89 GB.) */
int vsr_srfbn_plan_set_workspace_cap(vsr_srfbn_plan* plan, size_t cap_bytes);
int vsr_srfbn_chunk_maps(const vsr_srfbn_plan* plan);
/* Optional, before vsr_srfbn_bind: the number of frame windows W (1..65535, default 1) one forward fuses.  x is then
 * (W*M,3,h,w), window-major; y (W,3,s*h,s*w), y_u8 (W,s*h,s*w,3), vsr_srfbn_debug_premix (W*M,3,s*h,s*w).  The layers
 * sweep all W*M maps (chunk_maps is a divisor of W*M under a workspace cap, W*M without one) and the fc fuse writes
 * frame b from the maps [b*M, (b+1)*M), bit-identical to a one-window forward of window b.  M (num_maps) stays the fc
 * in-features.  The refresh entry points refresh the maps [first_map, M) of every window, one sweep per window.
 * Workspace and profile counts scale with W.  VSR_ERR_INVALID_ARG for W outside 1..65535; VSR_ERR_STATE after bind;
 * VSR_ERR_WORKSPACE if a workspace cap is set and not even one map fits (the plan is then unchanged). */
int vsr_srfbn_plan_set_windows(vsr_srfbn_plan* plan, int windows);
/* bytes of device memory the caller must provide */
size_t vsr_srfbn_weight_bytes(const vsr_srfbn_plan* plan);
size_t vsr_srfbn_workspace_bytes(const vsr_srfbn_plan* plan);
/* Converts the fp32 state-dict weights to the packed BF16 GEMM operands in host memory
 * (`host_packed`, vsr_srfbn_weight_bytes bytes); the caller copies them to the device. */
int vsr_srfbn_pack_weights(const vsr_srfbn_plan* plan, const vsr_srfbn_weights* w, void* host_packed);
/* Binds device buffers (packed weights + workspace) and builds the TMA descriptors. */
int vsr_srfbn_bind(vsr_srfbn_plan* plan, const void* dev_weights, void* dev_workspace,
                   size_t workspace_bytes);
/* x: (M,3,h,w) f32 NCHW, 0..255 (video_super_resolution.py:40,62); y: (1,3,s*h,s*w) f32.
 * With vsr_srfbn_plan_set_windows(W): x (W*M,3,h,w), y (W,3,s*h,s*w), y_u8 (W,s*h,s*w,3). */
int vsr_srfbn_forward(vsr_srfbn_plan* plan, const float* x, float* y, vsr_stream_t stream);
/* Same, with the fused frame also (or only) as u8 pixels: y_u8 (s*h,s*w,3) NHWC = clamp(y,0,255) rounded half to
 * even, the format the reference's loader holds frames in (utils/video_utils.py:23) -- what a frame writer or the
 * final gather consumes.  Either of y / y_u8 may be NULL, not both. */
int vsr_srfbn_forward_u8(vsr_srfbn_plan* plan, const float* x, float* y, uint8_t* y_u8, vsr_stream_t stream);
/* The fuse pass of a frame (video_super_resolution.py:62) feeds `data` -- the frames -- unchanged and replaces the
 * other maps: the M maps are independent until the per-pixel fc, so a second call whose stack differs from the previous
 * forward's only in the maps [first_map, M) sweeps the layers over those maps alone and reuses the per-map images of
 * the others, which are still in the workspace.  Bit-identical to vsr_srfbn_forward_u8 on the same stack.
 * vsr_srfbn_prepare_refresh (after bind, once per first_map; not with a workspace cap) builds the second layer list;
 * vsr_srfbn_forward_refresh_u8 needs a preceding full forward of the same plan on the same stream (VSR_ERR_STATE). */
int vsr_srfbn_prepare_refresh(vsr_srfbn_plan* plan, int first_map);
int vsr_srfbn_forward_refresh_u8(vsr_srfbn_plan* plan, const float* x, float* y, uint8_t* y_u8, int first_map,
                                 vsr_stream_t stream);
/* Map-parallel forward: one frame over G GPUs, bit-identical to vsr_srfbn_forward_u8 on one (DESIGN.md 11).  The maps go
 * through the conv stack independently until the per-pixel fc, and the fc needs all M maps of a pixel but nothing of
 * any other pixel, so rank r sweeps the maps [m_r, m_{r+1}), the ranks exchange row bands of the per-map images, and
 * each rank fuses the rows of its band with the same kernel and the same additions as the one-GPU forward.
 * vsr_srfbn_plan_set_map_range (before bind, like set_windows / set_workspace_cap): the plan sweeps the stack maps
 *   [m0, m1) only and lays out the per-map images of m1-m0 maps; x stays the full (M,3,h,w) stack and the fc in-features
 *   stay M.  A workspace cap chunks inside the range (chunk_maps divides m1-m0).  VSR_ERR_UNSUPPORTED with windows > 1
 *   (either order); VSR_ERR_WORKSPACE as set_workspace_cap (the plan is then unchanged).  vsr_srfbn_forward[_u8] and
 *   vsr_srfbn_forward_refresh_u8 return VSR_ERR_UNSUPPORTED on a plan whose range is not all maps.
 * vsr_srfbn_forward_maps: sweeps the range of x; the per-map images stay in the workspace (no fc).
 * vsr_srfbn_forward_maps_refresh: after vsr_srfbn_prepare_refresh(plan, first_map) and a forward_maps of the same plan,
 *   re-sweeps only [max(first_map, m0), m1) -- nothing when that is empty -- for a stack that changed only in the maps
 *   [first_map, M) (the fuse pass).  windows must be 1.
 * vsr_srfbn_pack_bands: lr_bounds (host, bands+1 ints) 0 = l_0 < l_1 < ... < l_bands = h, bands 1..64; band p is the HR
 *   rows [s*l_p, s*l_{p+1}).  Copies the range's per-map images into send (bands, m1-m0, 3, rows_p, s*w) f32, band-major
 *   and back to back (band p starts (m1-m0)*3*s*l_p*s*w floats in), the send buffer of one all_to_all with split sizes
 *   (m1-m0)*3*rows_p*s*w.  Maps partitioned contiguously in rank order make each rank's receive buffer (M,3,rows,s*w).
 * vsr_srfbn_fuse_band: maps (M,3,rows,s*w) f32 (16-byte aligned) -> y_band (3,rows,s*w) f32 (16-byte aligned) and / or
 *   y_u8_band (rows,s*w,3) u8 -- for band p, the frame's (H,W,3) u8 buffer + s*l_p*W*3 bytes.  rows a multiple of s.
 *   The fc_fuse kernel of vsr_srfbn_forward_u8 with the band as the frame: every output is bit-identical.
 * vsr_unpack_bands: the reorder after a gather of bands.  src: `bands` bands band_stride elements apart (0: back to back
 *   as above), band p holding `planes` planes of bounds[p+1]-bounds[p] rows of `row` elements; dst (planes,
 *   bounds[bands], row) receives band p's rows at [bounds[p], bounds[p+1]) of every plane.  elem_bytes 1 or 4 (4-byte
 *   aligned pointers).  E.g. the fp32 frame from (G,3,rows_max,W) padded bands, the (H,W,3) u8 frame (planes 1, row
 *   W*3 bytes), the (3,h,w) LR estimate slot. */
int vsr_srfbn_plan_set_map_range(vsr_srfbn_plan* plan, int m0, int m1);
int vsr_srfbn_forward_maps(vsr_srfbn_plan* plan, const float* x, vsr_stream_t stream);
int vsr_srfbn_forward_maps_refresh(vsr_srfbn_plan* plan, const float* x, int first_map, vsr_stream_t stream);
int vsr_srfbn_pack_bands(const vsr_srfbn_plan* plan, const int* lr_bounds, int bands, float* send, vsr_stream_t stream);
int vsr_srfbn_fuse_band(vsr_srfbn_plan* plan, const float* maps, int rows, float* y_band, uint8_t* y_u8_band,
                        vsr_stream_t stream);
int vsr_unpack_bands(const void* src, void* dst, int elem_bytes, int64_t planes, int64_t row, const int* bounds,
                     int bands, int64_t band_stride, vsr_stream_t stream);
/* Per-launch accounting for bench.py: with profiling enabled, vsr_srfbn_forward brackets every
 * kernel launch with CUDA events on the caller's stream; vsr_srfbn_profile_read waits for the last
 * forward and returns, per kernel class, the summed device time (ms), the number of launches, and
 * the layers' specified 2*MAC FLOPs and compulsory bytes (inputs + outputs of each launch, once).
 * Arrays have VSR_SRFBN_KERNEL_CLASSES entries, in the order of vsr_srfbn_kernel_class_name(). */
#define VSR_SRFBN_KERNEL_CLASSES 10
const char* vsr_srfbn_kernel_class_name(int k);
int vsr_srfbn_profile_enable(vsr_srfbn_plan* plan, int enable);
int vsr_srfbn_profile_read(vsr_srfbn_plan* plan, double* ms, int32_t* launches, double* flops, double* bytes);
/* per-launch device time of the last profiled forward, in launch order; returns the number of
 * launches (<0 on error) and fills at most `capacity` entries */
int vsr_srfbn_profile_launches(vsr_srfbn_plan* plan, float* ms, int32_t* kclass, int32_t capacity);

/* Test hook: per-map network output before the fc fuse, (M,3,s*h,s*w) f32 (SRProjectionModule.py:143);
 * valid after vsr_srfbn_forward on the same stream. */
int vsr_srfbn_debug_premix(const vsr_srfbn_plan* plan, float* out_maps, vsr_stream_t stream);
/* Test hook: runs the layers [first, first + count) of a bound plan's layer list (count >= 1) over the plan's first chunk
 * of maps of x, exactly as a forward's sweep launches them: the im2col of those maps first when first == 0, and the last
 * layer (conv_out) reads x for its skip and writes the chunk's premix slot.  The layer list is the one a profiled forward
 * of an unchunked plan reports through vsr_srfbn_profile_launches, without its first (im2col) and last (fc) launch.
 * VSR_ERR_INVALID_ARG for a null plan or x or a range outside the list, VSR_ERR_STATE for an unbound plan; no CUDA call
 * before these checks. */
int vsr_srfbn_debug_run_layers(vsr_srfbn_plan* plan, const float* x, int first, int count, vsr_stream_t stream);
/* Test hook (host only, valid once the plan is created, bound or not): byte offset and size of one activation buffer in
 * the plan's workspace layout.  LR takes index 0..6 and HR 0..5, every other id index 0.  Sizes for chunk_maps maps
 * (P = chunk_maps*h*w LR pixels): A0, XFEAT, HIDDEN, LR, U P*64 (BF16 (P,32)); C128 P*256; HR x4 chunk_maps*(h+1)*(w+1)*
 * 16*64 (HR block layout), x2 4P*64 (NHWC); HB s*s*P*64; HT (x2) 4P*64; ACC (x4) P*512 (fp32 partial slots); PREMIX the
 * per-map images of every swept map.  VSR_ERR_UNSUPPORTED for a buffer the plan does not have (x4: HR index 5, kept on
 * chip by the merged kernel, and HT; x2: ACC); VSR_ERR_INVALID_ARG for a null pointer or an id / index out of range. */
#define VSR_SRFBN_BUF_A0 0
#define VSR_SRFBN_BUF_C128 1
#define VSR_SRFBN_BUF_XFEAT 2
#define VSR_SRFBN_BUF_HIDDEN 3
#define VSR_SRFBN_BUF_LR 4
#define VSR_SRFBN_BUF_U 5
#define VSR_SRFBN_BUF_HR 6
#define VSR_SRFBN_BUF_HB 7
#define VSR_SRFBN_BUF_HT 8
#define VSR_SRFBN_BUF_ACC 9
#define VSR_SRFBN_BUF_PREMIX 10
#define VSR_SRFBN_BUFFERS 11
int vsr_srfbn_debug_buffer(const vsr_srfbn_plan* plan, int id, int index, size_t* offset, size_t* bytes);

/* Single-layer test hooks: run ONE layer of the stack through the same tcgen05 kernels the plan
 * uses, on BF16 channels-last operands, so tests can compare layer by layer with torch.nn fp32
 * (SURVEY.md Appendix C).  All pointers device.  `act`: 1 = PReLU(slope), 0 = none.
 *   pointwise: y[r, 0:32] = act(sum_k x[r, k] * w[n, k] + b[n]),  x (rows, K) bf16, K%32==0, K<=224
 *   deconv   : ConvTranspose2d(32,32,8,4,2): x (B,h,w,32) bf16 -> y (B,4h,4w,32) bf16 (block_layout=0)
 *              or the HR block layout (B,8,h+1,w+1,64) (block_layout=1, DESIGN.md 2)
 * w/b in the reference (torch) layouts, fp32, HOST memory. */
int vsr_test_pointwise(const void* x_bf16, int64_t rows, int K, const float* w_host,
                       const float* b_host, float slope, int act, void* y_bf16,
                       void* workspace, size_t workspace_bytes, vsr_stream_t stream);
int vsr_test_deconv(const void* x_bf16, int B, int h, int w, const float* w_host,
                    const float* b_host, float slope, int block_layout, void* y_bf16,
                    void* workspace, size_t workspace_bytes, vsr_stream_t stream);
/*   x2_layer : one layer of the x2 geometry (SRFBN's k6 s2 p2; SURVEY.md 8 a6 / config C4; the reference
 *              hard-wires x4, SRProjectionModule.py:101-103) + PReLU:
 *              up=1 ConvTranspose2d(32,32,6,2,2): x (B,h,w,32) -> y (B,2h,2w,32), w (32 in,32 out,6,6);
 *              up=0 Conv2d(32,32,6,2,2): x (B,2h,2w,32) -> y (B,h,w,32), w (32 out,32 in,6,6). */
int vsr_test_x2_layer(const void* x_bf16, int up, int B, int h, int w, const float* w_host,
                      const float* b_host, float slope, void* y_bf16, void* workspace,
                      size_t workspace_bytes, vsr_stream_t stream);
size_t vsr_test_workspace_bytes(int B, int h, int w);
/*   fused_down: the kernel the plan uses for the HR half of a feedback group
 *              (SRProjectionModule.py:70-80): PReLU(Conv1x1 over nsrc concatenated HR maps) ->
 *              Conv2d(32,32,8,4,2) -> PReLU.  hr: (nsrc,B,8,h+1,w+1,64) bf16 block layout; nsrc==1
 *              skips the 1x1 (group 0: the strided conv alone).  wt (32,32*nsrc), wd (32,32,8,8) fp32
 *              host.  y (B,h,w,32) bf16.
 *              workspace: vsr_test_workspace_bytes + B*h*w*512 bytes. */
int vsr_test_fused_down(const void* hr_bf16, int nsrc, int B, int h, int w, const float* wt_host,
                        const float* bt_host, float slope_t, const float* wd_host, const float* bd_host,
                        float slope_d, void* y_bf16, void* workspace, size_t workspace_bytes,
                        vsr_stream_t stream);
/*   fused_updown: the kernel the plan uses for feedback groups 3-5 of the x4 stack, with the group's
 *              transposed conv inside: U = PReLU(ConvTranspose2d(32,32,8,4,2)(lr)) is source nsrc-1
 *              of the fused_down computation above.  lr (B,h,w,32) bf16;
 *              hr: (nsrc,B,8,h+1,w+1,64) bf16 block layout, slots 0..nsrc-2 read, slot nsrc-1 receives U
 *              (zero ring included) iff store, untouched otherwise; nsrc 2..6.  wu (32 in,32 out,8,8),
 *              wt (32,32*nsrc), wd (32,32,8,8) fp32 host.  y (B,h,w,32) bf16.
 *              workspace: vsr_test_workspace_bytes + B*h*w*512 bytes, any contents. */
int vsr_test_fused_updown(const void* lr_bf16, void* hr_bf16, int nsrc, int store, int B, int h, int w,
                          const float* wu_host, const float* bu_host, float slope_u, const float* wt_host,
                          const float* bt_host, float slope_t, const float* wd_host, const float* bd_host,
                          float slope_d, void* y_bf16, void* workspace, size_t workspace_bytes,
                          vsr_stream_t stream);
/*   conv_in  : the stack's first layer as the plan runs it: sub_mean (sub_bias), Conv2d(3,128,3,p1) zero-padding the
 *              SHIFTED image, + PReLU.  x (B,3,h,w) f32 -> y (B,h,w,128) bf16; w (128,3,3,3), b (128), sub_bias (3)
 *              fp32 host.  workspace: vsr_test_workspace_bytes + B*h*w*64 bytes (the im2col operand). */
int vsr_test_conv_in(const float* x, int B, int h, int w, const float* w_host, const float* b_host, float slope,
                     const float* sub_bias_host, void* y_bf16, void* workspace, size_t workspace_bytes,
                     vsr_stream_t stream);
/*   conv_out : the stack's last layer as the plan runs it: Conv2d(32,3,3,p1) of hb (B,s*h,s*w,32) bf16 + bilinear
 *              upsampling (align_corners=False) of x (B,3,h,w) f32 + sub_bias, + add_bias -> y (B,3,s*h,s*w) f32;
 *              scale s 2 or 4.  w (3,32,3,3), b (3), sub_bias (3), add_bias (3) fp32 host.
 *              workspace: vsr_test_workspace_bytes bytes. */
int vsr_test_conv_out(const void* hb_bf16, const float* x, int scale, int B, int h, int w, const float* w_host,
                      const float* b_host, const float* sub_bias_host, const float* add_bias_host, float* y,
                      void* workspace, size_t workspace_bytes, vsr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VSR_B200_H_ */
