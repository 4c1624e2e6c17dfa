/* vid2vid-b200 -- C ABI of the sm_100a frame-synthesis engine (libv2v_b200.so).
 *
 * Plain pointers and sizes only: no torch / ATen types cross this boundary.  Every function returns
 * 0 on success and a non-zero code on failure (cudaError_t value, or V2V_ERR_* below);
 * v2v_last_error() returns a human-readable message for the calling thread.  Nothing here allocates
 * caller-visible memory: callers own all input / output tensors (the reference's Python Functions
 * allocate outputs the same way: resample2d.py:17, channelnorm.py:11, correlation.py:22-24).  All work
 * is enqueued on the cudaStream_t the caller passes (the reference enqueues on
 * at::cuda::getCurrentCUDAStream(), correlation_cuda.cc:76) and is re-entrant across plans.
 *
 * Two groups of entry points:
 *  (1) stand-alone operators -- one per native op of the reference's pybind11 extensions (b1 in
 *      SURVEY.md 8b) and per HBM-bound helper of the model layer;
 *  (2) the plan runtime -- the nn.Module surface (b2): Python describes a generator / discriminator
 *      once as a graph of logical values and convolution units; the runtime lowers it to halo-padded
 *      NHWC bf16 buffers, TMA tensor maps, packed weights and a kernel sequence captured in a CUDA
 *      graph, and runs it per frame against caller-owned fp32 NCHW tensors.
 */
#ifndef V2V_B200_H
#define V2V_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* v2v_stream_t; /* == cudaStream_t */
typedef struct v2v_plan v2v_plan;

#define V2V_ERR_INVALID 10001
#define V2V_ERR_STATE 10002
#define V2V_ERR_UNSUPPORTED 10003

enum { V2V_PAD_NONE = 0, V2V_PAD_ZERO = 1, V2V_PAD_REFLECT = 2 };
enum { V2V_ACT_NONE = 0, V2V_ACT_RELU = 1, V2V_ACT_LRELU = 2, V2V_ACT_TANH = 3, V2V_ACT_SIGMOID = 4 };
enum { V2V_NORM_NONE = 0, V2V_NORM_BATCH = 1, V2V_NORM_INSTANCE = 2 };
enum { V2V_IMPL_UMMA = 0, V2V_IMPL_SIMT = 1 };
/* Arithmetic of the convolution stack (accumulation is fp32 in both):
 *   V2V_PREC_BF16    operands rounded to bf16, one tcgen05.mma per K block ("fast"; ~2^-9 relative operand error)
 *   V2V_PREC_BF16X3  fp32-class: every operand x is carried as hi = bf16(x), lo = bf16(x - hi) and the kernel accumulates
 *                    A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (three MMAs per K block, ~2^-17 relative); raw conv outputs and
 *                    norm statistics stay fp32.  This is the mode whose results are compared with the fp32 reference
 *                    (nn.Conv2d in fp32, models/networks.py:132-183) at a stated fp32-class tolerance. */
enum { V2V_PREC_BF16 = 0, V2V_PREC_BF16X3 = 1 };

int v2v_version(void);
const char* v2v_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * (1) Stand-alone operators.  All tensors fp32, contiguous NCHW, on the current device.
 * ---------------------------------------------------------------------------------------------- */

/* correlation_cuda.forward (correlation_cuda.cc:10-87; kernel correlation_cuda_kernel.cu:73-147).
 * in1,in2 (N,C,H,W) -> out (N, D*D, outH, outW), D = 2*(max_disp/stride2)+1; shapes via
 * v2v_correlation_out_shape.  kernel_size must be 1 (the only value FlowNetC uses, FlowNetC.py:31).
 * The reference's rbot1/rbot2 scratch tensors are not needed. */
int v2v_correlation_out_shape(int H, int W, int pad_size, int kernel_size, int max_displacement, int stride1,
                              int stride2, int* outC, int* outH, int* outW);
int v2v_correlation_forward(const float* in1, const float* in2, float* out, int N, int C, int H, int W, int pad_size,
                            int kernel_size, int max_displacement, int stride1, int stride2, int corr_type_multiply,
                            v2v_stream_t stream);

/* resample2d_cuda.forward (resample2d_cuda.cc:6-13; kernel resample2d_kernel.cu:15-64).
 * in1 (N,C,inH,inW), flow (N,2,H,W) -> out (N,C,H,W); kernel_size must be 1. */
int v2v_resample2d_forward(const float* in1, const float* flow, float* out, int N, int C, int H, int W, int inH,
                           int inW, int kernel_size, v2v_stream_t stream);

/* channelnorm_cuda.forward (channelnorm_cuda.cc:6-13; kernel channelnorm_kernel.cu:18-60).
 * in (N,C,H,W) -> out (N,1,H,W) = sqrt(sum_c in^2); norm_deg must be 2. */
int v2v_channelnorm_forward(const float* in, float* out, int N, int C, int H, int W, int norm_deg,
                            v2v_stream_t stream);

/* BaseNetwork.resample / BaseModel.resample (models/networks.py:102-115, models/base_model.py:183-196):
 * grid_sample(image, linspace grid + flow/((dim-1)/2), bilinear, border).  image (N,C,H,W),
 * flow (N,2,H,W) in pixels.  align_corners: 0 = installed-PyTorch default, 1 = PyTorch-0.4 semantics. */
int v2v_resample_forward(const float* image, const float* flow, float* out, int N, int C, int H, int W,
                         int align_corners, v2v_stream_t stream);

/* Vid2VidModelG.encode_input + BaseModel.get_edges (models/vid2vid_model_G.py:86-112,
 * models/base_model.py:146-152).  labels, inst: (F,H,W) float ids (F = batch*frames; inst may be NULL
 * when use_instance == 0) -> out (F, label_nc + use_instance, H, W). */
int v2v_onehot_edges(const float* labels, const float* inst, float* out, int F, int label_nc, int use_instance, int H,
                     int W, v2v_stream_t stream);

/* AvgPool2d(3, stride=2, padding=1, count_include_pad=False) on P planes (BaseModel.build_pyr,
 * models/base_model.py:122-134): in (P,H,W) -> out (P,(H-1)/2+1,(W-1)/2+1). */
int v2v_avgpool3s2(const float* in, float* out, int P, int H, int W, v2v_stream_t stream);

/* Vid2VidModelG.compute_mask (models/vid2vid_model_G.py:322-330): real_A (B,T,C,H,W), frame t ->
 * mask (B,1,H,W) = clamp(sum over fg_labels of real_A[:, t, label], 0, 1).  n_labels <= 16. */
int v2v_fg_mask(const float* real_A, float* mask, int B, int T, int C, int H, int W, int t, const int* fg_labels,
                int n_labels, v2v_stream_t stream);

/* Streaming clip input (test.py:31-41 feeds a tG-frame window of label ids per generated frame, of which only the newest
 * frame is new): window (T,H,W) float ids, oldest first, is shifted by one frame in place and `frame` (H,W; dtype 0 uint8,
 * 1 int32, 2 float) appended.  Keeps the window resident so a step uploads one uint8 frame instead of T float ones. */
int v2v_ids_window_push(float* window, const void* frame, int dtype, int T, int H, int W, v2v_stream_t stream);
/* util.tensor2im (util/util.py:48-71) on the device: image (C,H,W) float in [-1,1] -> out (H,W,C) uint8
 * = uint8(clip((image + 1) / 2 * 255, 0, 255)). */
int v2v_tensor2im_u8(const float* image, uint8_t* out, int C, int H, int W, v2v_stream_t stream);

/* Losses of the training step (models/vid2vid_model_D.py:117-140,199-213; criteria models/networks.py:731-812) and the
 * backward of the helpers they differentiate through.  `out` / `grad_out` are 1-element device tensors (no host sync);
 * sum_ws: one double of scratch.
 *   l1_loss: out = mean |a*m - b*m| over N*C*H*W; mask (N,1,H,W) broadcast over channels or NULL (plain L1); b may be NULL (= 0).
 *   mse_const: out = mean (x - target)^2   (GANLoss, LSGAN). */
int v2v_l1_loss_forward(const float* a, const float* b, const float* mask, int N, int C, int H, int W, double* sum_ws, float* out,
                        v2v_stream_t stream);
int v2v_l1_loss_backward(const float* a, const float* b, const float* mask, int N, int C, int H, int W, const float* grad_out,
                         float* grad_a, float* grad_b, v2v_stream_t stream);
int v2v_mse_const_forward(const float* x, int64_t numel, float target, double* sum_ws, float* out, v2v_stream_t stream);
int v2v_mse_const_backward(const float* x, int64_t numel, float target, const float* grad_out, float* grad_x, v2v_stream_t stream);
/* Backward of v2v_avgpool3s2 (grad_in written) and of v2v_resample_forward (grad_image accumulated with atomics into a
 * caller-zeroed tensor, grad_flow written; either may be NULL). */
int v2v_avgpool3s2_backward(const float* grad_out, float* grad_in, int P, int H, int W, v2v_stream_t stream);
int v2v_resample_backward(const float* image, const float* flow, const float* grad_out, float* grad_image, float* grad_flow, int N,
                          int C, int H, int W, int align_corners, v2v_stream_t stream);

/* Face discriminator of the pose training step (--add_face_disc, models/vid2vid_model_D.py:148-158,215-230).
 * face_window: bounding box, over all N images of real_A (N,C,H,W), of the face pixels -- channel 2 > 0.9 (predicate 0) or, with
 *   --openpose_only (predicate 1), 0.19 < c0 < 0.21 && c1 < -0.99 && -0.61 < c2 < -0.59, compared in fp32 -- turned into the
 *   reference's fixed window: centre clamped to [half, dim - 1 - half], window [centre - half, centre + half) per axis.
 *   win: 10 int32 of device memory, zeroed by the caller before the first call and reusable afterwards (one launch per call,
 *   no memset): win[0..4] = {found, ys, ye, xs, xe} (all 0 when no face pixel exists), win[5..9] scratch left zeroed.
 * crop_concat_forward: out (N, Ca+Cb, Ly, Lx) = cat(a[:, :, ys:ys+Ly, xs:xs+Lx], b[...same window...], dim=1), a (N,Ca,H,W),
 *   b (N,Cb,H,W), the window origin read from win[1] / win[3] on the device.
 * crop_backward: grad_b (N,Cb,H,W) = channels [c_off, c_off+Cb) of grad_out (N, c_off+Cb, Ly, Lx) inside the window, 0 outside. */
int v2v_face_window(const float* real_A, int N, int C, int H, int W, int predicate, int half_y, int half_x, int32_t* win,
                    v2v_stream_t stream);
int v2v_crop_concat_forward(const float* a, int Ca, const float* b, int Cb, int N, int H, int W, const int32_t* win, int Ly, int Lx,
                            float* out, v2v_stream_t stream);
int v2v_crop_backward(const float* grad_out, int c_off, int Cb, int N, int H, int W, const int32_t* win, int Ly, int Lx, float* grad_b,
                      v2v_stream_t stream);

/* FlowNet2 glue (models/flownet2_pytorch/models.py:97-160, models/flownet.py:43-58), fp32 NCHW.
 * flownet_prep: the image pair -> x (B,6,H,W) = (pair - mean over both frames and all pixels, per sample and colour) / rgb_max,
 *   frame 0 in channels 0-2, frame 1 in 3-5 (models.py:97-103); x1 (may be NULL) = the frame-1 half as its own contiguous
 *   (B,3,H,W) tensor; mean_ws: B*3 floats of scratch.  Plane (frame f, sample b, colour c) = frame{f} + b*batch_stride +
 *   c*channel_stride floats: the reference's stacked (B,3,2,H,W) `inputs` is frame1 = frame0 + H*W, strides 6*H*W / 2*H*W;
 *   two separate (B,3,H,W) images (models/flownet.py:51) are strides 3*H*W / H*W. */
int v2v_flownet_prep(const float* frame0, const float* frame1, int64_t batch_stride, int64_t channel_stride, float* x, float* x1,
                     float* mean_ws, int B, int H, int W, float rgb_max, v2v_stream_t stream);
/* F.interpolate on `planes` planes (h,w) -> (H,W): mode 0 bilinear (align_corners=False), 1 nearest; values are multiplied by
 * `mul` first (`* div_flow`, models.py:106,118,130) -- or divided by pre_div when pre_div != 1 (FlowNetSD, models.py:142-143);
 * out_div (may be NULL) additionally receives out / div (`/ div_flow` of the next evidence stack).  use_scale_factor: 1 when the reference passes scale_factor= (nn.Upsample, models.py:49-60),
 * 0 when it passes size= (models/flownet.py:49-50,55-57). */
int v2v_resize(const float* in, float* out, float* out_div, int planes, int h, int w, int H, int W, int mode, int use_scale_factor,
               float mul, float pre_div, float div, v2v_stream_t stream);
/* out (N,C,H,W) = a[:, c_off:c_off+C] - b   (brightness error x[:, :3] - resampled_img1, models.py:113-116) */
int v2v_sub_channels(const float* a, const float* b, float* out, int N, int Ca, int c_off, int C, int H, int W, v2v_stream_t stream);
/* conf (N,1,H,W) = (sum_c (im1 - warped)^2 < threshold) as 0/1 floats (models/flownet.py:52-54, threshold 0.02) */
int v2v_flow_conf(const float* im1, const float* warped, float* conf, int N, int C, int H, int W, float threshold,
                  v2v_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (2) Plan runtime.
 *
 * A plan is built once per (module, input shape): create -> describe (g_* calls, in execution order)
 * -> finalize -> run per frame.  "values" are logical NHWC activations identified by small ints;
 * "raws" are un-normalised convolution outputs.  Caller tensors are addressed by IO slot: the
 * pointers are supplied at run time (v2v_plan_run), so PyTorch may hand over new tensors each call.
 * Parameter pointers (weights, biases, norm affine / running stats) are device pointers to the
 * caller's fp32 tensors in PyTorch layout; they are read when weights are (re)packed
 * (finalize / v2v_plan_repack) and, for norm parameters, at run time.
 * ---------------------------------------------------------------------------------------------- */

typedef struct v2v_conv_desc {
  int Cin, Cout, kh, kw;
  int stride;          /* 1 or 2 */
  int pad;             /* padding of the convolution (the ReflectionPad2d amount when pad_mode is reflect) */
  int pad_mode;        /* V2V_PAD_ZERO / V2V_PAD_REFLECT */
  int transposed;      /* 1: nn.ConvTranspose2d(stride 2) with `pad` and `output_padding` */
  int output_padding;
  const float* weight; /* conv: [Cout][Cin][kh][kw]; transposed: [Cin][Cout][kh][kw] */
  const float* bias;   /* [Cout] or NULL */
  /* Optional second parameter set stacked along Cout (heads only): output channels [Cout - Cout2, Cout) come from
   * weight2 [Cout2][Cin][kh][kw] / bias2.  Lets two reference convs that read the same input (model_final_flow and
   * model_final_w, models/networks.py:182-183) run as one convolution.  Cout2 == 0: unused. */
  int Cout2;
  const float* weight2;
  const float* bias2;
} v2v_conv_desc;

typedef struct v2v_norm_desc {
  int kind;                      /* V2V_NORM_* ; statistics are always those of the current tensor (train mode) */
  const float* gamma;            /* [C] or NULL */
  const float* beta;             /* [C] or NULL */
  float* running_mean;           /* [C] or NULL: updated as nn.BatchNorm2d does in train mode */
  float* running_var;
  int64_t* num_batches_tracked;  /* or NULL */
  float momentum, eps;
} v2v_norm_desc;

typedef struct v2v_head_channel {
  int slot;        /* IO slot of the destination fp32 NCHW tensor */
  int channel;     /* destination channel index */
  int dst_C;       /* channel count of the destination tensor */
  int act;         /* V2V_ACT_* applied after bias */
  float scale;     /* multiplied after the activation (flow head: 20 * 2^scale) */
} v2v_head_channel;

int v2v_plan_create(int device, int conv_impl /* V2V_IMPL_* */, v2v_plan** out);
int v2v_plan_destroy(v2v_plan* plan);
/* Select V2V_PREC_* (default V2V_PREC_BF16); must precede the first v2v_g_* call. */
int v2v_plan_set_precision(v2v_plan* plan, int precision);

/* Channels [c_off, c_off + C) of the fp32 NCHW tensor (N, C_src, H, W) bound to IO slot `slot`. */
int v2v_g_input(v2v_plan* plan, int slot, int N, int C_src, int c_off, int C, int H, int W, int* value_out);
/* As v2v_g_input with flags.  V2V_INPUT_EXACT_BF16: the caller promises that every element of the window is exactly
 * representable in bf16 (one-hot label maps, 0/1 edge maps -- what encode_input produces at full resolution,
 * models/vid2vid_model_G.py:93-105): precise plans then skip the all-zero lo half of that operand (2 MMAs per K block, no
 * change in results). */
#define V2V_INPUT_EXACT_BF16 1
int v2v_g_input_ex(v2v_plan* plan, int slot, int N, int C_src, int c_off, int C, int H, int W, int flags, int* value_out);
/* Convolution of a value; result is a raw (pre-norm) tensor. */
int v2v_g_conv(v2v_plan* plan, int value_in, const v2v_conv_desc* conv, int* raw_out);
/* value = act(norm(raw)) + add0 + add1   (add ids may be -1).  Conv bias is folded into running_mean only.
 * With V2V_NORM_NONE and a biased conv the pass computes act(raw + bias) (FlowNet2's norm-less units). */
int v2v_g_norm_act(v2v_plan* plan, int raw_in, const v2v_norm_desc* norm, int act, float slope, int add0, int add1,
                   int* value_out);
/* Same, on output channels [c_off, c_off + C) of the raw tensor (c_off % 8 == 0): lets convolutions that share their
 * input and geometry run as one conv with stacked weights (v2v_conv_desc.weight2) and still feed separate norm layers
 * (model_down_seg.1 / indv_down.1, models/networks.py:132,153).  The slice starting at Cout - Cout2 uses bias2. */
int v2v_g_norm_act_slice(v2v_plan* plan, int raw_in, int c_off, int C, const v2v_norm_desc* norm, int act, float slope,
                         int add0, int add1, int* value_out);
/* value = act(conv(value_in) + bias)   (layers without normalisation) */
int v2v_g_conv_act(v2v_plan* plan, int value_in, const v2v_conv_desc* conv, int act, float slope, int* value_out);
/* Small-Cout head (Cout <= 16): per channel bias + activation + scale -> fp32 NCHW planes of caller tensors. */
int v2v_g_head(v2v_plan* plan, int value_in, const v2v_conv_desc* conv, const v2v_head_channel* channels);
/* value = torch.cat(values, dim=1) (FlowNet2's skip / evidence stacks, FlowNetC.py:105-126, models.py:117,144). */
int v2v_g_concat(v2v_plan* plan, const int* values, int n, int* value_out);
/* value = act(correlation_cuda.forward(a, b)) with the FlowNetC parameters (FlowNetC.py:30-31,79-84); runs the stand-alone
 * correlation kernel on plan-internal scratch.  kernel_size 1, stride1 1, pad_size == max_displacement only. */
int v2v_g_correlation(v2v_plan* plan, int value_a, int value_b, int pad_size, int kernel_size, int max_displacement, int stride1,
                      int stride2, int act, float slope, int* value_out);
/* Export a value as fp32 NCHW into the caller tensor bound to `slot`. */
int v2v_g_export(v2v_plan* plan, int value, int slot);
/* Fused warp / blend / fg composite on caller tensors (slots; -1 = absent).  s_raw is read (head output)
 * and, with a fg model, overwritten with the composited raw image; s_final is written. */
int v2v_g_composite(v2v_plan* plan, int s_raw, int s_flow, int s_weight, int s_prev, int prev_C, int s_fg, int s_mask,
                    int s_final, int N, int H, int W, int use_warp, int align_corners);

/* As v2v_g_composite, with the composited raw image written to IO slot s_raw_out (>= 0) instead of over s_raw: training
 * plans need the head output intact for the backward. */
int v2v_g_composite_ex(v2v_plan* plan, int s_raw, int s_flow, int s_weight, int s_prev, int prev_C, int s_fg, int s_mask,
                       int s_final, int s_raw_out, int N, int H, int W, int use_warp, int align_corners);

/* Training plans (before finalize): keep the batch statistics and allocate dense fp32 gradient buffers. */
int v2v_plan_set_training(v2v_plan* plan, int on);
/* Backward of the LAST v2v_plan_run of this plan (whose intermediate buffers the plan still holds): autograd of
 * netG.forward / netD.forward as train.py:50-93 drives it.  io_ptrs: the forward tensors, as passed to v2v_plan_run.
 * grad_io_ptrs[slot]: for output slots the incoming gradient (fp32 NCHW, NULL = none); for input slots the destination of
 * the input gradient (accumulated into; NULL = not wanted).  params / param_grads: n_params pairs (parameter device pointer as
 * given in the conv / norm descriptors, gradient tensor of the same layout, accumulated into). */
int v2v_plan_backward(v2v_plan* plan, void* const* io_ptrs, void* const* grad_io_ptrs, int n_io, const void* const* params,
                      void* const* param_grads, int n_params, v2v_stream_t stream);

/* Lower the graph, pack the weights, build the TMA descriptors and the kernel list.  v2v_plan_finalize allocates the plan's
 * arena (activation buffers, raw conv outputs, packed weights, statistics rows) itself; v2v_plan_finalize_ws places it in
 * caller-owned device memory instead: `workspace` must be 1024-byte aligned and hold v2v_plan_workspace_bytes(plan) bytes
 * (valid to ask BEFORE finalize: the layout is computed on the host), stays owned by the caller and must outlive the plan.
 * (Training plans additionally allocate their gradient buffers and backward sub-plans themselves.) */
int v2v_plan_finalize(v2v_plan* plan, v2v_stream_t stream);
int v2v_plan_finalize_ws(v2v_plan* plan, void* workspace, int64_t workspace_bytes, v2v_stream_t stream);
/* Re-read all weight pointers and repack (after an optimiser step / load_state_dict). */
int v2v_plan_repack(v2v_plan* plan, v2v_stream_t stream);
/* Run once.  io_ptrs[slot] = device pointer of the caller tensor bound to that slot.  use_graph: 0 eager, 1 replay the
 * captured CUDA graph, 2 eager without the running-statistics side effect (recomputation before a backward). */
int v2v_plan_run(v2v_plan* plan, void* const* io_ptrs, int n_io, int use_graph, v2v_stream_t stream);

/* Runs the plan once eagerly with a CUDA event after every kernel: kinds[i] (0 import, 1 conv, 2 raw-stats,
 * 3 stats-finalize, 4 norm-apply, 5 export, 6 composite), ms[i] device time, macs[i] algorithmic conv MACs. */
int v2v_plan_profile(v2v_plan* plan, void* const* io_ptrs, int n_io, v2v_stream_t stream, int max_ops, int* kinds,
                     float* ms, double* macs, int* n_ops);

/* Introspection (host logic tests, bench accounting). */
int v2v_plan_num_kernels(const v2v_plan* plan);             /* kernels launched per run */
double v2v_plan_conv_macs(const v2v_plan* plan);            /* algorithmic conv MACs per run (dense, unpadded) */
int64_t v2v_plan_workspace_bytes(const v2v_plan* plan);       /* arena bytes; may be called before finalize (host only) */
/* Writes a JSON description of the lowered plan (buffers, tiles, tap groups) into buf; returns needed size. */
int64_t v2v_plan_describe(const v2v_plan* plan, char* buf, int64_t cap);

/* Host-only: the tap-group table the kernel would use for a convolution (pure function; no GPU).
 * Each group g: plane[g], dy[g], dx[g], tap0[g]; R[0] taps per group, tap r reading the group's patch shifted by
 * (r / R[1]) rows and (r % R[1]) columns (R must hold 2 entries); phase p covers groups
 * [phase_begin[p], phase_begin[p+1]); per-phase output offsets oy_add/ox_add; buffer padding pads[4] =
 * {top, left, bottom, right}; parity; grid_h/grid_w; out_h/out_w.  Arrays must hold 64 / 5 / 4 entries. */
int v2v_conv_tap_table(const v2v_conv_desc* conv, int H, int W, int allow_reuse, int* n_groups, int* R, int* plane,
                       int* dy, int* dx, int* tap0, int* n_phases, int* phase_begin, int* oy_add, int* ox_add,
                       int* pads, int* parity, int* grid_hw, int* out_hw, int* mul);

#ifdef __cplusplus
}
#endif
#endif /* V2V_B200_H */
