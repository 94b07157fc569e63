/*
 * dmv3d.h -- C ABI of libdmv3d.so: hand-written sm_100a CUDA kernels for the
 * appearance-flow training hot path of aclike/dynamic_multiview_3d.
 *
 * The reference has no FFI of its own (it is pure Python on TensorFlow 1.3); each entry
 * point below replaces one TensorFlow library op that the reference's op helpers
 * (dyn_mult_view/mv3d/utils/tf_utils.py) or its optimizer call dispatch to.  The
 * "replaces" notes give the reference call site (paths relative to the reference root).
 *
 * Conventions (SURVEY.md 8(b)(iii)):
 *   - every function returns int: 0 = DMV_OK, negative = DMV_E_*; dmv_last_error() has the
 *     message of the calling thread's last failure; nothing throws or aborts;
 *   - all tensor pointers are DEVICE pointers, NHWC contiguous; the caller owns every
 *     buffer (including workspaces, sized by the matching *_workspace_size call);
 *   - every launch is asynchronous on the cudaStream_t passed as `stream` (void*);
 *     no host synchronisation, no persistent allocation, no global mutable state
 *     besides a diagnostic launch counter;
 *   - "bf16" buffers hold __nv_bfloat16 (uint16_t storage).
 */
#ifndef DMV3D_H_
#define DMV3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMV_OK 0
#define DMV_E_INVALID_ARG (-1)
#define DMV_E_ALIGN (-2)
#define DMV_E_UNSUPPORTED_SHAPE (-3)
#define DMV_E_CUDA (-4)
#define DMV_E_WORKSPACE (-5)

/* sampler flags */
#define DMV_SAMPLER_ADD_GRID 1u /* input is a flow field; warp = flow + grid is formed in-kernel
                                   (replaces warp_pts_layer + coords, tf_utils.py:35-52)        */
#define DMV_SAMPLER_GRID_XY 2u  /* grid channel 0 = column, channel 1 = row.  Default (flag clear)
                                   is the reference's (Y,X) order: channel 0 = ROW index,
                                   tf_utils.py:48-51 -- zero flow then yields the transpose      */

/* activations fused into epilogues (tf_utils.py:25-33; tanh heads main_model.py:79) */
#define DMV_ACT_NONE 0
#define DMV_ACT_LRELU 1 /* 0.6x + 0.4|x| */
#define DMV_ACT_RELU 2  /* 0.5x + 0.5|x| */
#define DMV_ACT_TANH 3

/* loss modes */
#define DMV_LOSS_L2 0 /* euclidean_loss, tf_utils.py:18-19 */
#define DMV_LOSS_L1 1 /* l1_loss,        tf_utils.py:22-23 */

/* element types of activation tensors at the conv/linear boundary */
#define DMV_DT_BF16 0
#define DMV_DT_F32 1
#define DMV_DT_S2D 2 /* the pointer is the space-to-depth bf16 tensor written by dmv_thin_s2d_prep (thin stride-2
                        layers only: e0's image, the flow head's gradient); shapes still describe the ORIGINAL tensor */

/* implementation selector for conv/deconv/linear entry points */
#define DMV_ALGO_AUTO 0    /* tcgen05/TMEM/TMA implicit GEMM where the shape allows, else SIMT */
#define DMV_ALGO_SIMT 1    /* straightforward CUDA-core kernels (bring-up + on-GPU cross-check)  */
#define DMV_ALGO_TCGEN05 2 /* force the tensor-core path; DMV_E_UNSUPPORTED_SHAPE if it cannot  */
/* Weight packing split from the layer call (OR-ed into `algo` of dmv_conv2d_fwd / dmv_conv2d_dgrad / dmv_deconv2d_fwd /
 * dmv_deconv2d_dgrad).  Some tensor-core forms read the bf16 weights in a packed layout that the call writes into the head
 * of `workspace` first.  PACK_ONLY: do just that (same shape arguments, same workspace; x / y / dx may be any non-null
 * pointers) and return -- a no-op for forms that need no packing.  PREPACKED: the workspace already holds this layer's
 * packed weights (a PACK_ONLY call with identical arguments ran after the last weight update): skip the packing kernel.
 * The train step packs every layer once per step on a side stream, off the forward / input-gradient chain. */
#define DMV_ALGO_PACK_ONLY 0x100
#define DMV_ALGO_PREPACKED 0x200

/* ---- library info ------------------------------------------------------------------- */
int dmv_version(void);                      /* MAJOR*10000 + MINOR*100 + PATCH */
const char* dmv_arch(void);                 /* "sm_100a" */
int dmv_last_error(char* buf, size_t n);    /* copies the thread's last error text */
long long dmv_launch_count(void);           /* kernels launched by this library so far */
long long dmv_tc_launch_count(void);        /* of which tcgen05 tensor-core kernels */
/* successful launches so far whose label (the text of the library's launch check, e.g. "halo_tc", "igemm_tc (split-K)")
 * equals `what`: tells which kernel form a call took.  Thread-safe; 0 for an unknown label or NULL. */
long long dmv_launch_count_named(const char* what);

/* ---- bilinear sampler --------------------------------------------------------------- *
 * replaces tf.contrib.resampler.resampler -- tf_utils.py:40-42 (resample_layer) and
 * multi_view_model/tests/test_resampler.py:44; with DMV_SAMPLER_ADD_GRID also
 * warp_pts_layer/coords (tf_utils.py:35-52).
 *   data  [B,H,W,C] f32      wf [B,Hout,Wout,2] f32 (warp points, or flow with ADD_GRID)
 *   out   [B,Hout,Wout,C] f32
 *   dbg_idx  optional int32 [B,Hout,Wout,4] = (fx,fy,cx,cy), 0 for invalid samples
 *   dbg_mask optional uint8 [B,Hout,Wout]: bit0 sample valid, bits1..4 taps
 *            (fx,fy),(cx,cy),(fx,cy),(cx,fy) in range
 * wf channel 0 is x (column of `data`), channel 1 is y (row).                          */
int dmv_sampler_fwd(const float* data, const float* wf, float* out, int32_t* dbg_idx,
                    uint8_t* dbg_mask, int B, int H, int W, int C, int Hout, int Wout,
                    unsigned flags, void* stream);

/* dmv_sampler_fwd with a source shared by `group` consecutive output samples (rendering one source image from many
 * viewpoints without copying it):
 *   data [B_src,H,W,C] f32      wf [B_src*group,Hout,Wout,2] f32      out [B_src*group,Hout,Wout,C] f32
 * out sample n (0 <= n < B_src*group) samples data[n / group]; every value has the bits dmv_sampler_fwd gives on the
 * source repeated `group` times along the batch.  No debug outputs; no backward (inference only).
 * DMV_E_INVALID_ARG / DMV_E_UNSUPPORTED_SHAPE / DMV_E_ALIGN as dmv_sampler_fwd; a refused call launches nothing. */
int dmv_sampler_fwd_shared_src(const float* data, int B_src, int group, const float* wf, float* out,
                               int H, int W, int C, int Hout, int Wout, unsigned flags, void* stream);

/* ---- several targets of one source (multi-target training) ---- *
 * Output sample n (0 <= n < B_src*group) warps data[n / group]: data [B_src,H,W,C] f32, wf / grad_wf [B_src*group,Hout,Wout,2],
 * gen_out / target / grad_out [B_src*group,Hout,Wout,C].  No gradient wrt the source (it is a network input).  Every value
 * has the bits of the plain call on the source repeated `group` times along the batch.  Refusals: DMV_E_INVALID_ARG for a
 * null pointer or non-positive B_src / group, DMV_E_UNSUPPORTED_SHAPE when B_src*group overflows and as the plain call,
 * DMV_E_ALIGN as the plain call; a refused call launches nothing.
 *   dmv_sampler_loss_fused_shared_src: dmv_sampler_loss_fused; workspace dmv_sampler_loss_workspace_size(B_src*group, Hout, Wout).
 *   dmv_sampler_grad_flow_shared_src:  the grad_wf half of dmv_sampler_bwd (grad_out = d loss / d out).                        */
int dmv_sampler_loss_fused_shared_src(const float* data, int B_src, int group, const float* wf, const float* target,
                                      const float* chan_weight, int mode, float inv_count, float* gen_out, float* grad_wf,
                                      float* loss_out, int H, int W, int C, int Hout, int Wout, unsigned flags,
                                      void* workspace, size_t workspace_bytes, void* stream);
int dmv_sampler_grad_flow_shared_src(const float* data, int B_src, int group, const float* wf, const float* grad_out,
                                     float* grad_wf, int H, int W, int C, int Hout, int Wout, unsigned flags, void* stream);

/* replaces the registered gradient "ResamplerGrad" (implicit via
 * tf.train.AdamOptimizer.minimize, appearance_flow_model.py:77).
 *   grad_data [B,H,W,C] f32 or NULL (skip: the source is a network input)
 *   grad_wf   [B,Hout,Wout,2] f32 (gradient wrt warp == wrt flow)
 * grad_data is produced by a deterministic owner-computes scatter (no atomics): same
 * inputs -> same bits.  workspace (only read / written when grad_data != NULL):
 * dmv_sampler_bwd_workspace_size bytes, 16-byte aligned -- a pre-pass fills it with the tap
 * bounding box of every 1024-pixel output tile and of each of its 32 warp chunks
 * (33 int4 per tile); it needs no initialisation and may be shared by calls on one stream. */
size_t dmv_sampler_bwd_workspace_size(int B, int H, int W, int C, int Hout, int Wout);
int dmv_sampler_bwd(const float* data, const float* wf, const float* grad_out,
                    float* grad_data, float* grad_wf, int B, int H, int W, int C, int Hout,
                    int Wout, unsigned flags, void* workspace, size_t workspace_bytes,
                    void* stream);

/* Training-step fusion of the three calls above: resample_layer(src, warp_pts_layer(flow)) (tf_utils.py:35-42,
 * appearance_flow_model.py:126-127), euclidean_loss / l1_loss against the target (tf_utils.py:18-23,
 * appearance_flow_model.py:73) and the gradient wrt the flow (ResamplerGrad through the loss gradient) in ONE kernel:
 *   gen_out [B,Hout,Wout,C] = the warped image (as dmv_sampler_fwd, same bits)
 *   loss_out = inv_count * sum_pixels sum_c w_c * ((gen - target)^2 | |gen - target|)
 *   grad_wf [B,Hout,Wout,2] = d loss / d flow                     (as dmv_loss_fused_fwd_bwd + dmv_sampler_bwd)
 * Needs C in {1,3,4}, W*C and Wout*C multiples of 4, 16-byte aligned buffers; otherwise DMV_E_UNSUPPORTED_SHAPE
 * (use the three separate calls).  workspace: dmv_sampler_loss_workspace_size bytes, zeroed ONCE by the caller and
 * not shared with other calls (it holds a self-resetting counter).                                                */
size_t dmv_sampler_loss_workspace_size(int B, int Hout, int Wout);
int dmv_sampler_loss_fused(const float* data, const float* wf, const float* target, const float* chan_weight,
                           int mode, float inv_count, float* gen_out, float* grad_wf, float* loss_out, int B, int H,
                           int W, int C, int Hout, int Wout, unsigned flags, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Several source views per target (Zhou et al.'s multi-view appearance flow) in ONE kernel: each view's warp, the
 * confidence-weighted fusion, the loss and the gradient wrt the 3-channel head.  View v of target b is row v*B + b:
 *   data   [views*B,H,W,C] f32      head [views*B,Hout,Wout,3] f32: channels 0-1 the flow (grid added per flags, as
 *                                   dmv_sampler_fwd), channel 2 the confidence logit; read in place
 *   target [B,Hout,Wout,C] f32, or NULL: forward only (fused_out required, grad_head and loss_out NULL)
 *   fused_out [B,Hout,Wout,C] = sum_v softmax_v(logit) * warp(src_v, flow_v), or NULL
 *   grad_head [views*B,Hout,Wout,3] = (dL/dflow, dL/dlogit), written whole (channel 2 is 0 for views == 1), or NULL
 *             (a validation pass: loss only)
 *   loss_out  device float[1] as dmv_loss_fused_fwd_bwd (no mask)
 * fused_out and grad_head have the bits of dmv_sampler_fwd per view, dmv_loss_fused_fwd_bwd (V = views, the logits) and
 * the grad_wf half of dmv_sampler_bwd on its grad_gen.  The loss is a deterministic per-CTA sum (same inputs -> same
 * bits; within 1e-6 relative of the composition's, which sums in another order).  1 <= views <= 8, C in {1,3,4}, W*C and
 * Wout*C multiples of 4, Hout > 1, 16-byte aligned buffers.  workspace (training only):
 * dmv_sampler_loss_workspace_size(B, Hout, Wout) bytes, zeroed once, not shared between concurrent calls.
 * Refusals launch nothing: DMV_E_INVALID_ARG for a null data / head, a NULL combination the mode does not allow, or an
 * unknown loss mode; DMV_E_UNSUPPORTED_SHAPE for views, C or the shape; DMV_E_ALIGN; DMV_E_WORKSPACE.                */
int dmv_sampler_fuse_views_loss(const float* data, int views, const float* head, const float* target,
                                const float* chan_weight, int mode, float inv_count, float* fused_out, float* grad_head,
                                float* loss_out, int B, int H, int W, int C, int Hout, int Wout, unsigned flags,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ---- fused loss (+ multi-view confidence fusion) forward and backward ----------------- *
 * replaces euclidean_loss / l1_loss (tf_utils.py:18-23) and the weighted sums of
 * main_model.py:144-154, multiobject_appflow.py:223-283, plus their gradients.
 *   gen     [V,B,H,W,C] f32 (V = 1: plain loss)       target [B,H,W,C] f32
 *   logits  [V,B,H,W] f32 confidence logits, NULL when V == 1
 *           fused = sum_v softmax_v(logits)_v * gen_v   (SURVEY 8(f)-3; not in the reference)
 *   mask    optional [B,H,W,1] f32: diff = (fused - target) * mask (masked_image_loss)
 *   chan_weight host float[C]: per-channel loss weights (e.g. 1,1,1,0.1 for RGB-D)
 *   inv_count  1 / (global B*H*W): the mean's divisor (global batch under data parallelism)
 *   loss_out   device float[1]: sum_c w_c * L(diff_c) * inv_count   (overwritten)
 *   grad_gen   [V,B,H,W,C] f32 or NULL; grad_logits [V,B,H,W] f32 or NULL
 *   fused_out  optional [B,H,W,C] f32 (V > 1)
 *   workspace  dmv_loss_workspace_size(B*H*W) bytes                                      */
size_t dmv_loss_workspace_size(long long pixels);
int dmv_loss_fused_fwd_bwd(const float* gen, const float* logits, int V, const float* target,
                           const float* mask, const float* chan_weight, int mode,
                           float inv_count, float* loss_out, float* grad_gen,
                           float* grad_logits, float* fused_out, long long pixels, int C,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---- SSIM + L1 photometric loss (Monodepth / SfMLearner-style) ----------------------------------------------- *
 * Per image and channel, with x = gen and y = target reflection-padded by one pixel (row -1 reads row 1, row H reads
 * row H-2, the same for columns) and the 3x3 window centred on every pixel p:
 *   SSIM_p = ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),  C1 = 0.01^2, C2 = 0.03^2,
 *   s_xx = mean(x^2) - mu_x^2, s_xy = mean(xy) - mu_x mu_y   (Monodepth2's SSIM without its final clamp)
 *   loss_out = inv_count * sum_{n,p} sum_c w_c * (alpha * (1 - SSIM_p,c) / 2 + (1 - alpha) * |x - y|)
 * alpha = 0 is the L1 loss; d|d|/dd = 0 at d = 0.  The loss is a deterministic per-CTA sum (same inputs -> same bits).
 *   gen, target, grad_gen [B,H,W,C] f32; grad_gen = d loss / d gen, or NULL (loss only: a validation pass)
 *   chan_weight host float[C]; workspace dmv_loss_workspace_size(B*H*W) bytes, 8-byte aligned, zeroed once and not
 *   shared between concurrent calls.  Launches one kernel (label "loss_fused").
 * Refusals launch nothing: DMV_E_INVALID_ARG for a null pointer or alpha outside [0, 1] or NaN; DMV_E_UNSUPPORTED_SHAPE
 * for C not in {1,3,4}, B < 1 or H, W < 2; DMV_E_WORKSPACE; DMV_E_ALIGN for an unaligned workspace.
 * There is no fused warp + SSIM form: warp with dmv_sampler_fwd, take this loss, and the flow gradient with the grad_wf
 * half of dmv_sampler_bwd (a fused kernel measured no faster than these three calls; DESIGN.md §4).               */
int dmv_ssim_loss_fwd_bwd(const float* gen, const float* target, const float* chan_weight, float alpha, float inv_count,
                          float* loss_out, float* grad_gen, int B, int H, int W, int C, void* workspace,
                          size_t workspace_bytes, void* stream);

/* x[i] *= *scalar (device scalar): chains an upstream loss gradient without a host sync */
int dmv_scale_by_device_scalar(float* x, const float* scalar, long long n, void* stream);

/* ---- conv / deconv / linear ----------------------------------------------------------- *
 * TF-SAME padding is computed inside (out = ceil(in/s), extra padding bottom/right).
 * Weights are bf16 copies of the fp32 masters in the REFERENCE layouts:
 *   conv   w[kh,kw,Cin,Cout]   (tf_utils.py:75-77)      deconv w[kh,kw,Cout,Cin] (tf_utils.py:93-95)
 *   linear Matrix[K,N]         (tf_utils.py:62-64)
 * x_dtype / y_dtype are DMV_DT_*; accumulation is fp32.  bias may be NULL.
 * `act` is fused into the forward epilogue; backward entry points take the gradient wrt
 * the PRE-activation (dmv_act_bwd produces it from the post-activation output).          */

/* Scratch sizes.  Geometry is always that of the SAME conv the layer is (or is the gradient
 * of): BIG side [B,H,W,Cbig] (conv input / deconv output), small side ceil(H/stride) with
 * Csmall channels (conv output / deconv input).
 *   dmv_conv_workspace_size : forward and dgrad entry points (weight repacking; the patch
 *                             matrix of layers with < 8 big-side channels); NULL allowed
 *                             with DMV_ALGO_SIMT
 *   dmv_wgrad_workspace_size: wgrad entry points (deterministic split-K partials)
 * For linear layers use B = M, H = W = 1, kh = kw = stride = 1, Cbig = K, Csmall = N.      */
size_t dmv_conv_workspace_size(int B, int H, int W, int Cbig, int Csmall, int kh, int kw, int stride);
/* replaces tf.nn.conv2d(...,'SAME') + b  -- conv2d_msra, tf_utils.py:70-84 */
int dmv_conv2d_fwd(const void* x, int x_dtype, const void* w_bf16, const float* bias, void* y,
                   int y_dtype, int B, int H, int W, int Cin, int Cout, int kh, int kw,
                   int stride, int act, void* workspace, size_t workspace_bytes, int algo,
                   void* stream);
/* replaces Conv2DBackpropInput (implicit, appearance_flow_model.py:77).
 * Input-gradient entry points (conv, deconv, linear) take `y_in` / `act_in`: when `y_in` (bf16, the layer's own INPUT
 * as stored, i.e. the output of the producing layer's activation) is non-NULL and act_in != DMV_ACT_NONE they write
 *     dx * act_in'(y_in)      -- the gradient w.r.t. the producer's PRE-activation (TF: the LeakyRelu/Relu grad node) --
 * instead of dx.  Library builds with -DDMV_DACT_EPILOGUE=1 apply the factor to the fp32 accumulator in the tensor-core
 * epilogue (one rounding); the default build runs the elementwise pass (dmv_act_bwd, in place) behind the kernel --
 * measured faster with the present kernels, profiles/r02_dact_fusion.txt.  Results agree to one bf16 ulp.            */
int dmv_conv2d_dgrad(const void* dy_bf16, const void* w_bf16, void* dx_bf16, const void* y_in,
                     int act_in, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                     void* workspace, size_t workspace_bytes, int algo, void* stream);
/* replaces Conv2DBackpropFilter + BiasAddGrad.  dw f32 [kh,kw,Cin,Cout], db f32 [Cout] or NULL.
 * Deterministic split-K (fixed-order second pass).  workspace: dmv_wgrad_workspace_size.   */
size_t dmv_wgrad_workspace_size(int B, int H, int W, int Cbig, int Csmall, int kh, int kw, int stride);
int dmv_conv2d_wgrad(const void* x, int x_dtype, const void* dy_bf16, float* dw, float* db, int B,
                     int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                     void* workspace, size_t workspace_bytes, int algo, void* stream);

/* replaces tf.nn.conv2d_transpose(x, w, output_shape, strides) -- deconv2d_msra,
 * tf_utils.py:87-98 (no bias).  x [B,Hin,Win,Cin] -> y [B,Hout,Wout,Cout], where
 * Hin == ceil(Hout/stride).                                                               */
int dmv_deconv2d_fwd(const void* x_bf16, const void* w_bf16, void* y, int y_dtype, int B, int Hout,
                     int Wout, int Cin, int Cout, int kh, int kw, int stride, int act,
                     void* workspace, size_t workspace_bytes, int algo, void* stream);
int dmv_deconv2d_dgrad(const void* dy, int dy_dtype, const void* w_bf16, void* dx_bf16,
                       const void* y_in, int act_in, int B, int Hout, int Wout, int Cin, int Cout,
                       int kh, int kw, int stride, void* workspace, size_t workspace_bytes, int algo,
                       void* stream);
int dmv_deconv2d_wgrad(const void* x_bf16, const void* dy, int dy_dtype, float* dw, int B, int Hout,
                       int Wout, int Cin, int Cout, int kh, int kw, int stride, void* workspace,
                       size_t workspace_bytes, int algo, void* stream);

/* replaces tf.matmul(x, Matrix) + b -- linear_msra, tf_utils.py:54-67, and its gradients */
int dmv_linear_fwd(const void* x_bf16, const void* w_bf16, const float* bias, void* y_bf16, int M,
                   int K, int N, int act, void* workspace, size_t workspace_bytes, int algo,
                   void* stream);
int dmv_linear_dgrad(const void* dy_bf16, const void* w_bf16, void* dx_bf16, const void* y_in,
                     int act_in, int M, int K, int N, void* workspace, size_t workspace_bytes,
                     int algo, void* stream);
int dmv_linear_wgrad(const void* x_bf16, const void* dy_bf16, float* dw, float* db, int M, int K,
                     int N, void* workspace, size_t workspace_bytes, int algo, void* stream);

/* ---- elementwise ---------------------------------------------------------------------- *
 * replaces relu / lrelu (tf_utils.py:25-33), tf.nn.tanh and their gradients.
 * dmv_act_bwd: dpre = dy * act'(y) computed from the POST-activation output y
 * (lrelu/relu: slope by sign(y), TF's value at 0; tanh: 1 - y^2).                          */
int dmv_act_fwd(const void* x, void* y, int dtype, long long n, int act, void* stream);
int dmv_act_bwd(const void* dy, const void* y, void* dpre, int dtype, long long n, int act,
                void* stream);
/* dmv_act_bwd fused with the bias gradient (BiasAddGrad): db[c] = sum_rows dpre[row][c], bf16 [rows][C],
 * C % 8 == 0; deterministic.  The wgrad entry points may then be called with db = NULL.          */
size_t dmv_act_bwd_bias_workspace_size(long long rows, int C);
int dmv_act_bwd_bias(const void* dy_bf16, const void* y_bf16, void* dpre_bf16, float* db, long long rows,
                     int C, int act, void* workspace, size_t workspace_bytes, void* stream);
/* dmv_act_bwd_bias of a layer whose output [rows][C] was consumed `group` times (dy has rows * group rows, row r*group+t
 * for use t; row pitch ld_dy >= C elements, ld_dy % 8 == 0, so dy may be a column slice of a wider gradient):
 *   dpre[r][c] = bf16_rn((sum_{t = 0 .. group-1, in order, fp32} dy[r*group+t][c]) * act'(y[r][c])),  db = column sums of dpre.
 * workspace: dmv_act_bwd_bias_workspace_size(rows, C).  At group = 1, ld_dy = C the bits of dmv_act_bwd_bias. */
int dmv_act_bwd_bias_grouped(const void* dy_bf16, long long ld_dy, int group, const void* y_bf16, void* dpre_bf16,
                             float* db, long long rows, int C, int act, void* workspace, size_t workspace_bytes,
                             void* stream);
/* Thin stride-2 layers (image side of e0, appearance_flow_model.py:88; 2-channel side of the flow head, :125) run on
 * X2[n][H/2][W/2][32] = the 2x2 pixel block as channels (ph, pw, c), zero padded, bf16.  The conv / deconv entry
 * points build X2 themselves from a DMV_DT_F32 / DMV_DT_BF16 tensor; a caller that keeps X2 between the forward
 * and the weight-gradient call (or between dgrad and wgrad of the flow head) passes it with DMV_DT_S2D instead.
 * dmv_thin_s2d_size returns the bytes of X2, or 0 when the layer shape does not take this path.                    */
size_t dmv_thin_s2d_size(int N, int H, int W, int C_thin, int C_wide, int kh, int kw, int stride);
int dmv_thin_s2d_prep(const void* thin, int thin_dtype, void* x2, int N, int H, int W, int C_thin, void* stream);
/* uint8 pixels -> float32, dst = src / divisor in IEEE division (tf.cast(image, tf.float32) / 255.0,
 * utils/read_tf_records.py:111): lets the input pipeline ship the reference's uint8 pixel format over PCIe. */
int dmv_u8_to_f32(const unsigned char* src, float* dst, long long n, float divisor, void* stream);
/* The reader's whole image preparation (utils/read_tf_records.py:100-111) in one kernel: uint8 [B,H0,W0,C] as stored ->
 * central crop to min(H0,W0) (tf.image.resize_image_with_crop_or_pad) -> tf.image.resize_bicubic to [S,S] (TF-1.3 rule:
 * legacy coordinates in = out * crop / S, Keys A = -0.75 from a 1024-entry table, clamped taps, horizontal then vertical,
 * float32) -> / divisor.  With H0 = W0 = S (the reference's 128) it equals dmv_u8_to_f32 bit for bit.  C in {1,3,4}. */
int dmv_u8_crop_resize_bicubic(const unsigned char* src, float* dst, int B, int H0, int W0, int C, int S, float divisor,
                               void* stream);
int dmv_cast_f32_to_bf16(const float* src, void* dst_bf16, long long n, void* stream);
int dmv_cast_bf16_to_f32(const void* src_bf16, float* dst, long long n, void* stream);

/* ---- optimizer ------------------------------------------------------------------------ *
 * replaces tf.train.AdamOptimizer(lr).minimize -- appearance_flow_model.py:77 (ApplyAdam):
 *   m += (g - m)(1-b1);  v += (g*g - v)(1-b2);  theta -= (m * lr_t) / (sqrt(v) + eps)
 * with lr_t = lr * sqrt(1 - b2^t) / (1 - b1^t) (eps NOT bias-corrected).
 * dmv_adam_tick advances the device-resident state {b1^t, b2^t, lr_t, t} by one step so a
 * captured CUDA graph needs no host-side scalar updates: state is float[4], initialise to
 * {1, 1, 0, 0}.  dmv_adam_multi updates `count` tensors (host arrays of device pointers),
 * optionally writing a bf16 copy of the new parameters; grad_scale multiplies the gradient
 * first (e.g. 1/world_size).                                                               */
int dmv_adam_tick(float* state4, float lr, float beta1, float beta2, void* stream);
int dmv_adam_multi(float* const* params, const float* const* grads, float* const* m,
                   float* const* v, void* const* bf16_copy, const long long* n, int count,
                   const float* state4, float beta1, float beta2, float eps, float grad_scale,
                   void* stream);

/* dmv_adam_multi that does nothing unless *gate != 0 (device int): an update whose launch is scheduled before it is
 * known whether a gradient is pending -- the optimizer update of the late FC matrices is applied at the START of the next
 * step, next to the encoder's forward pass, inside a captured CUDA graph (data_parallel.py).  dmv_set_flag writes the
 * gate from the stream. */
int dmv_adam_multi_gated(float* const* params, const float* const* grads, float* const* m,
                         float* const* v, void* const* bf16_copy, const long long* n, int count,
                         const float* state4, float beta1, float beta2, float eps, float grad_scale,
                         const int* gate, void* stream);
int dmv_set_flag(int* flag, int value, void* stream);

/* dmv_linear_wgrad + dmv_adam_multi on one FC matrix in ONE pass (single-process training; the data-parallel exchange
 * needs the gradient in memory and keeps the two calls): the tile of dW = x^T dy (tf.matmul's weight gradient,
 * tf_utils.py:54-67) is formed in registers and consumed by ApplyAdam (appearance_flow_model.py:77) -- theta, m, v
 * fp32 [K,N] and the bf16 compute copy are updated, the gradient is never written (26 instead of 34 B/parameter).
 * dw_out (optional, fp32 [K,N]) also receives the gradient (tests).  K, N multiples of 8, 16-byte aligned pointers;
 * state4 as advanced by dmv_adam_tick for this step.  The caller orders it after the layer's dgrad (it rewrites the
 * bf16 weights that dgrad reads). */
int dmv_linear_wgrad_adam(const void* x_bf16, const void* dy_bf16, float* theta, float* m, float* v,
                          void* bf16_copy, float* dw_out, int M, int K, int N, const float* state4,
                          float beta1, float beta2, float eps, float grad_scale, void* stream);

/* ---- data-parallel exchange (new work: the reference is single-GPU, SURVEY 8(e)) -------------------- *
 * One chunk of the per-step exchange as ONE kernel over peer-mapped (symmetric) memory on the NVSwitch domain:
 *   reduce-scatter of the gradients  ->  TF-Adam on the slice this rank owns  ->  all-gather of the bf16 compute copy.
 * The chunk is elements [start, start + world * n_slice) of the flat buffers (variables.py); rank r owns
 * [start + r * n_slice, start + (r+1) * n_slice).  The owner reads the summed gradient of its slice straight from its
 * peers' gradient buffers -- `grad_peers[r]` (device pointers to every rank's flat fp32 gradient buffer; fixed summation
 * order r = 0..world-1, so the result is deterministic and the same on whichever rank computes it) or, when `grad_mc`
 * is non-NULL, one `multimem.ld_reduce.add.f32` per 16 bytes on the multicast mapping (in-switch reduction) --, updates
 * theta / m / v in its LOCAL fp32 buffers, and writes the refreshed bf16 copy into every rank's bf16 buffer
 * (`half_peers[r]`, or one `multimem.st` on `half_mc`).  No gradient is written back, nothing is read twice, no
 * library collective runs.
 * Cross-rank ordering: `signal_peers[r]` points at rank r's signal words (uint32, dmv_dp_signal_words() of them, zeroed
 * once, symmetric); slot `slot` holds a "gradients ready" and an "update written" word per rank.  Each launch takes the
 * next epoch from `local_state` (uint32[2 * slots], zeroed once: epoch, ticket), releases its ready word to every
 * peer, acquires all of theirs, works, releases its done word, and the last CTA waits for every peer's done word -- so
 * when the kernel has completed on a rank, that rank's bf16 chunk is complete and none of its peers still reads its
 * gradients.  All ranks must launch the same slots in the same order (they do: the order gradients become ready).
 * `replicated` != 0: no slicing -- every rank sums the whole range [start, start + n_slice) and updates all of it
 * locally (the bias tail, whose fp32 masters every rank keeps); nothing is written to peers.
 * world <= 8; n_slice % 8 == 0; start * 4 and the buffers 16-byte aligned; `ctas` CTAs of 256 threads (0 = default). */
int dmv_dp_signal_words(int slots);
int dmv_dp_exchange_chunk(const void* const* grad_peers, void* const* half_peers, void* const* signal_peers,
                          const void* grad_mc, void* half_mc, float* master, float* m, float* v,
                          void* local_state, long long start, long long n_slice, int rank, int world, int slot,
                          int replicated, const float* state4, float beta1, float beta2, float eps,
                          float grad_scale, int ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DMV3D_H_ */
