/*
 * b200sr.h -- C ABI of libb200sr.so: the RRDBNet generator (forward + backward) of MiNeves00/SR-GAN-FD as
 * hand-written sm_100a CUDA kernels.
 *
 * What this boundary replaces in the reference (pure PyTorch, no FFI of its own -- the "binding" is the
 * nn.Module.forward / autograd boundary):
 *   - ESRGAN/model.py:211-232   RRDBNet._forward_impl      (= BSRGAN/model.py:366-381, Real_ESRGAN/model.py:246-263,
 *                                                             A-ESRGAN/model.py:534-549)
 *   - ESRGAN/model.py:49-60     _ResidualDenseBlock.forward
 *   - ESRGAN/model.py:77-86     _ResidualResidualDenseBlock.forward
 *   - the autograd backward of all of the above (triggered at ESRGAN/train_rrdbnet.py:261, BSRGAN/train_bsrgan.py:463)
 * The reference-side stub that binds these entry points (ctypes, inside one torch.autograd.Function) is shown in
 * INTEGRATION.md and shipped as sr_gan_fd_b200/function.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch tensors); the library never frees or keeps one
 *     past the call, except that a plan caches TMA descriptors keyed on the workspace / packed / grads addresses;
 *   - all work is enqueued on the given stream, no hidden synchronisation (plan creation and the first call per
 *     workspace address do host-side descriptor encoding only);
 *   - return 0 on success, a negative b200sr_status otherwise; b200sr_last_error() gives a thread-local message;
 *   - plain C types only (no torch / C++ types).
 */
#ifndef B200SR_H_
#define B200SR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200sr_plan b200sr_plan;
typedef void* b200sr_stream; /* cudaStream_t */

enum b200sr_status {
  B200SR_OK = 0,
  B200SR_ERR_INVALID = -1,     /* bad argument / unsupported configuration */
  B200SR_ERR_CUDA = -2,        /* a CUDA runtime / driver call failed       */
  B200SR_ERR_UNSUPPORTED = -3  /* device is not sm_100                      */
};

enum b200sr_dtype { B200SR_F32 = 0, B200SR_F16 = 1, B200SR_BF16 = 2 };

/* Network + problem geometry.  Mirrors the reference constructor arguments (ESRGAN/model.py:145-153):
 * channels must be 64 and growth 32 (the only values the reference configs use; the tiles are built on them). */
typedef struct b200sr_net_desc {
  int32_t in_channels;  /* conv1 input channels (after Real-ESRGAN's pixel-unshuffle), 1..64 */
  int32_t out_channels; /* conv4 output channels, 1..16 */
  int32_t channels;     /* 64 */
  int32_t growth;       /* 32 */
  int32_t num_blocks;   /* RRDB count (23) */
  int32_t n_up;         /* nearest-x2 + conv stages: 0 (x1) .. 3 (x8) */
  int32_t batch, height, width; /* LR input geometry */
  int32_t training;     /* 1: keep activations for backward, build the backward schedule */
  int32_t grad_bucket_rrdbs; /* gradient buckets announced through b200sr_bucket_cb: RRDBs per bucket (0 = 1; the tail convs and
                              * conv1 are buckets of their own, the last trunk bucket holds at most two RRDBs so that little
                              * communication is left exposed after the last kernel) */
  int32_t deterministic; /* 1: bit-reproducible backward (see "Deterministic plans" below); 0: the default, atomic reductions */
} b200sr_net_desc;

/* Trunk plans (b200sr_trunk_plan_create): the stack of num_blocks RRDBs without conv1, the long skip and the tail -- what
 * nn.Sequential(*RRDBs) computes, for generators that keep the RRDB trunk and change everything around it.  The descriptor is the
 * generator's; a trunk plan requires n_up == 0 and in_channels == out_channels == channels == 64.  Every other entry point of a
 * generator plan works on it, with these shapes:
 *   x      [batch, 64, height, width], f32 / f16 / bf16, element strides x_strides[4] (NCHW or channels_last);
 *   y      [batch, 64, height, width] fp32 contiguous, NOT clamped;
 *   dy, dx [batch, 64, height, width] fp32 contiguous (dx: the gradient w.r.t. the trunk input);
 *   params 2 x 5 x 3 x num_blocks pointers, the convs in the Sequential's state_dict order (0.rdb1.conv1.weight, 0.rdb1.conv1.bias, ...);
 *   conv_wanted_or_null  5 x 3 x num_blocks bytes, same order.
 * The trunk kernels are the generator's: for the same input, a trunk plan's y is bit for bit the generator's trunk output. */

/* Unclamped plans (b200sr_unclamped_plan_create): the whole generator for models whose output is conv4's, not clamped -- BasicSR /
 * Real-ESRGAN RRDBNet, A-ESRGAN's Generator_RRDB.  It accepts exactly the descriptors b200sr_plan_create accepts, and every
 * generator entry point works on it unchanged (packing, forward, backward, b200sr_backward_select, launch counts, buckets,
 * deterministic mode, b200sr_debug_buffer).  What differs:
 *   y   [batch, out_channels, s*height, s*width] fp32: conv4's output, NOT clamped to [0, 1];
 *   dy  the gradient w.r.t. that unclamped y: it enters the backward as it is, with no clamp pass-through mask;
 *   the training workspace holds no "CMASK", so it is smaller by that buffer (batch x out_channels x s*height x s*width bytes,
 *   rounded up to 1024).
 * Launch list, parameter order, flat-gradient layout and b200sr_pack_layout_id are those of the clamped plan of the same descriptor,
 * so the packed buffer can be shared; for the same input, clamp(y_unclamped, 0, 1) is bit for bit the clamped plan's y. */

/* Deterministic plans (the `deterministic` member of the net, VGG and discriminator descriptors; torch.use_deterministic_algorithms).
 * A default plan sums weight and bias gradients (and the VGG loss value) with atomics, so their order -- and the last bits --
 * depend on CTA scheduling.  A deterministic plan gives bit-identical outputs for bit-identical inputs, for one GPU model,
 * one library build and one plan geometry: its reductions store per-split / per-block partials into a workspace area that
 * only deterministic plans have, and one ordered-sum launch behind each weight- or bias-gradient launch adds them in index
 * order (b200sr_num_launches / b200sr_backward_launches count those launches).  The split counts are fixed when the plan is
 * built.  Packing does not depend on the flag: b200sr_pack_layout_id is equal for the two modes, and one packed buffer serves both.
 * The single-layer b200sr_conv3x3_wgrad keeps its atomic flush. */

/* Called from inside b200sr_backward (on the calling host thread) each time every kernel that contributes to a
 * contiguous range [offset, offset+count) of the flat gradient buffer has been ENQUEUED on the stream: the callee
 * may record an event and start the NCCL all-reduce of that bucket on another stream. */
typedef void (*b200sr_bucket_cb)(void* user, int64_t offset, int64_t count);

int b200sr_plan_create(const b200sr_net_desc* desc, b200sr_plan** out);
int b200sr_trunk_plan_create(const b200sr_net_desc* desc, b200sr_plan** out); /* see "Trunk plans" above */
int b200sr_unclamped_plan_create(const b200sr_net_desc* desc, b200sr_plan** out); /* see "Unclamped plans" above */
void b200sr_plan_destroy(b200sr_plan* plan);

/* sizes (bytes) of the caller-allocated buffers */
size_t b200sr_workspace_bytes(const b200sr_plan* plan);
size_t b200sr_packed_bytes(const b200sr_plan* plan);
/* identifies the layout of the packed-weight buffer: plans of one network may pack differently (the dense-block schedule
 * depends on the geometry); a packed buffer may be shared between plans only if their ids are equal */
uint64_t b200sr_pack_layout_id(const b200sr_plan* plan);
/* number of parameter tensors (2 per conv: weight, bias) and total fp32 elements, in state_dict order */
int32_t b200sr_num_params(const b200sr_plan* plan);
int64_t b200sr_param_numel(const b200sr_plan* plan);
/* algorithmic FLOPs (2 x MACs of the reference graph) of one forward / one backward at the plan's geometry */
double b200sr_flops(const b200sr_plan* plan, int backward);
/* number of kernel launches one forward (backward = 0) / backward enqueues; backward = 1: no gradient-bucket callback
 * (one merged gradient unpack), backward = 2: with a callback (one unpack launch per bucket) */
int32_t b200sr_num_launches(const b200sr_plan* plan, int backward);

/* params: host array of b200sr_num_params() device pointers, fp32, state_dict order (conv1.weight, conv1.bias,
 * trunk.0.rdb1.conv1.weight, ...; weights OIHW).  Re-packs them into the bf16 tiles the kernels consume. */
int b200sr_pack_weights(b200sr_plan* plan, const float* const* params, void* packed, b200sr_stream stream);

/* x: [batch, in_channels, height, width] with element strides x_strides[4] (NCHW or channels_last), dtype per
 * b200sr_dtype.  y: [batch, out_channels, s*height, s*width] fp32 contiguous, clamped to [0,1] (unclamped plans: not clamped). */
int b200sr_forward(b200sr_plan* plan, const void* x, int x_dtype, const int64_t* x_strides, const void* packed,
                   void* workspace, float* y, b200sr_stream stream);

/* dy: gradient w.r.t. y, fp32 contiguous.  workspace/packed must be the ones used by the matching forward.
 * flat_grads: b200sr_param_numel() floats, OVERWRITTEN with the parameter gradients (state_dict order).
 * dx_or_null: NULL, or [batch, in_channels, height, width] fp32 contiguous, OVERWRITTEN with the gradient w.r.t. x
 * (what autograd produces in the reference when x.requires_grad). */
int b200sr_backward(b200sr_plan* plan, const float* dy, const void* packed, void* workspace, float* flat_grads,
                    float* dx_or_null, b200sr_bucket_cb cb, void* user, b200sr_stream stream);

/* As b200sr_backward, restricted to what the caller wants (frozen and partially frozen generators).
 * conv_wanted_or_null: host array of b200sr_num_params()/2 bytes in state_dict conv order (conv1, trunk.0.rdb1.conv1 ...
 * conv2, upsampling*, conv3, conv4); 1 = this conv's weight and/or bias gradient is wanted.  NULL = all wanted.
 * flat_grads_or_null: NULL = no parameter gradient at all (frozen generator); then conv_wanted must be NULL or all zero.
 * Entries of flat_grads belonging to unwanted convs are zero.  Buckets (cb) are announced only for ranges that
 * contain a wanted conv.
 * The data-gradient walk reaches conv1 only when dx is wanted or conv1 is; otherwise it ends after the lowest dense block that
 * holds a wanted conv (or after the HR tail, or is skipped).  A weight- or bias-gradient launch runs when one of the convs it
 * writes is wanted: a dense block's five convs share one launch.  With nothing wanted (no dx, no wanted conv) the call only
 * zeroes flat_grads_or_null.  b200sr_backward(...) is b200sr_backward_select(..., NULL, ...). */
int b200sr_backward_select(b200sr_plan* plan, const float* dy, const void* packed, void* workspace,
                           float* flat_grads_or_null, float* dx_or_null, const uint8_t* conv_wanted_or_null,
                           b200sr_bucket_cb cb, void* user, b200sr_stream stream);
/* kernel launches b200sr_backward_select enqueues for a mask (NULL = all wanted), counted as b200sr_num_launches counts them
 * (memsets are not launches): with_dx = the input gradient is wanted, with_cb = a bucket callback is installed (one unpack
 * launch per announced bucket instead of one merged unpack).  (plan, NULL, 0, 0) == b200sr_num_launches(plan, 1) and
 * (plan, NULL, 0, 1) == b200sr_num_launches(plan, 2).  0 for plans without a generator backward. */
int32_t b200sr_backward_launches(const b200sr_plan* plan, const uint8_t* conv_wanted_or_null, int with_dx, int with_cb);

/* ---- single-layer entry points (used by the parity tests) ------------------------------------------------------
 * x: NHWC bf16 [n*h*w][x_stride], the conv reads channels [0, cin).  w: fp32 OIHW [cout][cin][3][3], bias [cout] or
 * NULL.  y: NHWC bf16 [n*h*w][y_stride], written at channel y_coff.  act = 1 applies LeakyReLU(0.2).
 * scratch: >= b200sr_conv3x3_scratch_bytes(cin, cout) bytes. */
size_t b200sr_conv3x3_scratch_bytes(int cin, int cout);
int b200sr_conv3x3_fwd(const void* x, int n, int h, int w_, int cin, int x_stride, const float* w, const float* bias,
                       int cout, int act, void* y, int y_stride, int y_coff, void* scratch, b200sr_stream stream);
/* dx[n*h*w][dx_stride] (bf16, channels [dx_coff, dx_coff+cin)) = conv_transpose of dy (bf16, channels [0, cout)) */
int b200sr_conv3x3_dgrad(const void* dy, int n, int h, int w_, int cout, int dy_stride, const float* w, int cin,
                         void* dx, int dx_stride, int dx_coff, void* scratch, b200sr_stream stream);
/* dw[cout][cin][3][3] fp32 = sum_pixels x (bf16, channels [0, cin)) * dy (bf16, channels [0, cout)); cin <= 128,
 * cout <= 160, cout % 16 == 0.  dw is overwritten.  scratch: >= b200sr_conv3x3_wgrad_scratch_bytes(cin, cout). */
size_t b200sr_conv3x3_wgrad_scratch_bytes(int cin, int cout);
int b200sr_conv3x3_wgrad(const void* x, int n, int h, int w_, int cin, int x_stride, const void* dy, int cout,
                         int dy_stride, float* dw, void* scratch, b200sr_stream stream);

/* ---- next to the path (SURVEY.md section 8f): fused GradScaler-unscale + Adam + EMA over a list of fp32 tensors --------------
 * Replaces optimizer.step() + AveragedModel.update_parameters() of ESRGAN/train_rrdbnet.py:263-267 (torch.optim.Adam
 * semantics with L2 weight decay; EMA rule ema <- (1-d)*ema + d*p of train_rrdbnet.py:182, first update copies).
 * tensor_table: DEVICE array of n_tensors records {float* p; const float* g; float* m; float* v; float* ema (or NULL);
 * int64 numel; int64 block0} where block0 = running sum of ceil(numel/1024); total_blocks = that sum over all tensors;
 * block_tensor: DEVICE int32[total_blocks], block -> tensor index.  step: DEVICE float scalar, Adam steps taken so far
 * (advanced by the call unless skipped).  grad_scale / found_inf: device scalars or NULL (GradScaler protocol: gradients
 * are divided by *grad_scale; when *found_inf > 0 the Adam update is skipped -- the EMA still updates, as the reference
 * calls update_parameters unconditionally).  A NULL g marks a frozen parameter: no Adam update (p, m, v keep their values, as
 * torch.optim.Adam skips a parameter without a gradient), the EMA still averages it. */
int b200sr_fused_adam_ema(const void* tensor_table, const int32_t* block_tensor, int n_tensors, int64_t total_blocks, float lr,
                          float beta1, float beta2, float eps, float weight_decay, float* step, float ema_decay, int ema_copy,
                          const float* grad_scale, const float* found_inf, b200sr_stream stream);

/* ---- next to the path (SURVEY.md section 8f rank 4): the evaluation epilogue of validate() / test_*.py / inference.py -------
 * PSNR / SSIM on the Y channel as ESRGAN/image_quality_assessment.py:361-541 computes them (crop_border, rgb_to_ycbcr_torch with
 * only_use_y_channel, fp64, 11x11 gaussian window = outer product of window11, valid convolution), one pass per metric.
 * raw, dst: [n, 3, h, w] fp32 RGB in [0, 1].  Outputs are per-image SUMS (device doubles, either may be NULL):
 * psnr_sqerr_sum[i] = sum over the cropped frame of (255 Y_raw - 255 Y_dst)^2   -> PSNR = 10 log10(255^2 / (sum / count + 1e-8))
 * ssim_map_sum[i]   = sum of the SSIM map over its (h - 2 crop - 10) x (w - 2 crop - 10) positions -> SSIM = sum / count */
int b200sr_iqa_psnr_ssim_y(const float* raw, const float* dst, int n, int h, int w, int crop_border, const double* window11,
                           double* psnr_sqerr_sum, double* ssim_map_sum, b200sr_stream stream);
/* The same sums, bit-reproducible: per-block partials go to scratch (device, >= b200sr_iqa_det_scratch_bytes(n, h, w) bytes for
 * an n x h x w batch; a crop never needs more) and are added in block order. */
size_t b200sr_iqa_det_scratch_bytes(int n, int h, int w);
int b200sr_iqa_psnr_ssim_y_det(const float* raw, const float* dst, int n, int h, int w, int crop_border, const double* window11,
                               double* psnr_sqerr_sum, double* ssim_map_sum, double* scratch, b200sr_stream stream);
/* ESRGAN/imgproc.py:160-183 tensor_to_image: x [c, h, w] fp32 -> out_hwc [h, w, c] uint8 = trunc(clamp(255 x, 0, 255));
 * range_norm: x <- (x + 1) / 2 first; half: round to fp16 and multiply in fp16 as the reference does with half=True */
int b200sr_tensor_to_image_u8(const float* x, int c, int h, int w, int range_norm, int half, uint8_t* out_hwc, b200sr_stream stream);

/* ---- next to the path (SURVEY.md section 8f rank 3): VGG19 perceptual features / content loss -----------------------------------
 * The sixteen 3x3 convs of torchvision vgg19().features (up to conv5_4, index `last_conv` 0..15) on the chain kernel, input
 * normalisation, ReLU, 2x2 max-pools, the L1 feature loss of ESRGAN/model.py:246-292 / BSRGAN/model.py:501-554 and (optionally) its
 * gradient w.r.t. the first `grad_images` images.  The batch holds the sr images followed by the gt images (batch = 2 x pairs).
 * Plans share b200sr_workspace_bytes / b200sr_packed_bytes / b200sr_pack_weights (params: conv l weight at 2l, bias at 2l+1, fp32
 * OIHW) / b200sr_plan_destroy with the generator plans. */
typedef struct b200sr_vgg_desc {
  int32_t batch, height, width; /* images (sr then gt), input geometry */
  int32_t last_conv;            /* last conv to evaluate (0..15; 15 = conv5_4 = torchvision features.34) */
  int32_t feat_mask;            /* bit l set: keep conv l's output as fp32 (a feature node): BEFORE the ReLU for l == last_conv, AFTER it
                                 * for l < last_conv -- what torchvision's create_feature_extractor hands the reference, whose
                                 * in-place ReLUs overwrite every extracted conv output except the one that ends the graph */
  int32_t grad_conv;            /* -1, or the conv whose L1 feature loss is differentiated w.r.t. the input images */
  int32_t grad_images;          /* images (from 0) that receive a gradient: the sr half */
  float mean[3], std[3];        /* transforms.Normalize of the input */
  int32_t deterministic;        /* 1: b200sr_vgg_feature_l1 sums per-block partials in block order (bit-reproducible) */
} b200sr_vgg_desc;
int b200sr_vgg_plan_create(const b200sr_vgg_desc* desc, b200sr_plan** out);
/* x: [batch, 3, height, width] fp32 in [0, 1] with element strides x_strides[4] */
int b200sr_vgg_forward(b200sr_plan* plan, const float* x, const int64_t* x_strides, const void* packed, void* workspace,
                       b200sr_stream stream);
/* *out_sum (device double) = sum |f_sr - f_gt| over conv_index's feature map (mean = sum / (pairs * H_l * W_l * C_l)) */
int b200sr_vgg_feature_l1(b200sr_plan* plan, const void* workspace, int conv_index, int pairs, double* out_sum, b200sr_stream stream);
/* dx: [grad_images, 3, height, width] fp32, gradient of upstream[0] * mean|f_sr - f_gt| (grad_conv's features) w.r.t. the NORMALISED
 * input images (divide by std for the raw images); upstream: device float */
int b200sr_vgg_backward(b200sr_plan* plan, const float* upstream, const void* packed, void* workspace, float* dx, b200sr_stream stream);

/* ---- next to the path (SURVEY.md section 8f rank 2): the U-Net discriminator with spectral-norm convs --------------------------------
 * Replaces DiscriminatorUNet._forward_impl (BSRGAN/model.py:143-167 = Real_ESRGAN/model.py:81-105) and its autograd backward
 * (triggered at BSRGAN/train_bsrgan.py:420,430,463): conv1 3x3 -> three 4x4 stride-2 convs + LeakyReLU(0.2) -> three times
 * [bilinear x2, 3x3 conv + LeakyReLU, + skip] -> two 3x3 convs + LeakyReLU -> 3x3 conv to the logit map.  The spectral
 * normalisation itself (power iteration, W / sigma) stays with the caller: `params` holds the EFFECTIVE weights, and the returned
 * gradients are w.r.t. those.  Plans share b200sr_workspace_bytes / b200sr_packed_bytes / b200sr_pack_weights / b200sr_num_params /
 * b200sr_param_numel / b200sr_flops / b200sr_plan_destroy with the generator plans.
 * params (b200sr_pack_weights): 20 device pointers, weight then bias of conv1, down1, down2, down3, up1, up2, up3, conv2, conv3,
 * conv4 in that order; the bias entries of the eight bias-free convs are ignored (pass NULL).  Weights fp32 OIHW. */
typedef struct b200sr_disc_desc {
  int32_t in_channels;  /* 1..16 (3) */
  int32_t out_channels; /* 1..16 (1) */
  int32_t channels;     /* 64 */
  int32_t batch, height, width; /* height and width multiples of 8 (the reference's skip additions need that, too) */
  int32_t training;     /* 1: build the backward schedule */
  int32_t fp16;         /* 16-bit format of the activations / packed weights / gradients: 1 = fp16 (what the reference's autocast runs
                         * this network in; needs in_channels == 3, other widths fall back to bf16), 0 = bf16 (wider range) */
  int32_t deterministic; /* 1: bit-reproducible weight and bias gradients (see "Deterministic plans" above) */
} b200sr_disc_desc;
int b200sr_disc_plan_create(const b200sr_disc_desc* desc, b200sr_plan** out);
/* x: [batch, in_channels, height, width], element strides x_strides[4], dtype per b200sr_dtype;
 * y: [batch, out_channels, height, width] fp32 contiguous (the logit map) */
int b200sr_disc_forward(b200sr_plan* plan, const void* x, int x_dtype, const int64_t* x_strides, const void* packed, void* workspace,
                        float* y, b200sr_stream stream);
/* dy: gradient w.r.t. y, fp32 contiguous.  flat_grads_or_null: b200sr_param_numel() floats, OVERWRITTEN with the gradients of the
 * effective weights in `params` order (absent biases take no room) -- NULL skips every weight-gradient kernel (the generator
 * update, where the discriminator is frozen).  dx_or_null: [batch, in_channels, height, width] fp32, OVERWRITTEN with the gradient
 * w.r.t. x -- NULL skips it (the discriminator update, where the input carries no gradient). */
int b200sr_disc_backward(b200sr_plan* plan, const float* dy, const void* packed, void* workspace, float* flat_grads_or_null,
                         float* dx_or_null, b200sr_stream stream);

const char* b200sr_last_error(void);
int b200sr_version(void);
/* timing probes for profiling only (results become wrong unless noted): bit 0 (1) no epilogue traffic, bit 1 (2) no MMAs,
 * bit 2 (4) no activation / weight loads, bit 3 (8) no bf16 output stores, bit 4 (16) no dependency waits, bit 6 (64) role
 * profiler and bit 7 (128) per-entry timeline (both harmless), bit 8 (256) no signaller fence, bit 9 (512) no proxy fence.
 * 0 = normal operation (default). */
void b200sr_debug_set(int flags);
/* bit 6 (64) of the debug flags makes the chain kernel record, per CTA, the cycles each warp role waited on each barrier
 * kind (12 counters per CTA, see conv_kernel.cuh); this copies the first n counters of the last launch to the host. */
int b200sr_debug_read_profile(unsigned long long* out_host, int n);
/* byte offset and size of a named workspace tensor of a plan (test / debugging use); B200SR_ERR_INVALID for a name the plan
 * does not have.  Discriminator plans name every tensor they keep: the ingested input "xin", the forward activations
 * "T0u" "T1u" "T2u" "T3" "B1" "A1" "B2" "A2" "B3" "A3" "S3" "A4" "A5" and, in training plans, the backward gradients "DYP" "G5"
 * "G4" "GS3" "G3" "GB3" "GS2" "GA2" "GB2" "GS1" "GA1" "GB1" "GT3" "GT2" "GT1" "G0" (build_disc_plan in b200sr.cu says what each
 * holds).  Generator plans name theirs too (build_plan in b200sr.cu; trunk plans only "TR" "C1" "C2", the "D" buffers and, in training
 * plans, "GR" "GC1" "GC2" and the "DYB" buffers): "xin", the fp32 carriers "T0" "TR" "C1" "C2" (tile-blocked),
 * the dense-block buffers "D0" ... "D{R-1}" (R = 3 * num_blocks; inference plans keep only the ping-pong pair "D0" "D1"), the
 * tail activations "SPLT" "SPL0" ... "SPL{n_up}" "SPLC" and, in training plans, "CMASK" (not in unclamped plans) "DYP" "G3"
 * "GU1" ... "GU{n_up}" "GT" "GTB" "GR" "GC1" "GC2" "GO1" "DYB0" ... "DYB{R-1}".  VGG plans (build_vgg_plan; l = conv index, h_l x w_l
 * its lattice, C_l its output channels, N = batch, NB = grad_images) name: "xin" [N, H, W, 64] bf16 [hi(3) | lo(3) | hi(3) | 0] of
 * (x - mean) / std; "A{l}" (l <= last_conv) [N, h_l, w_l, C_l] bf16, conv l's output after the ReLU; "P{l}" (l = 1, 3, 7, 11 and
 * l < last_conv) [N, h_l/2, w_l/2, C_l] bf16, its 2x2 max-pool; "F{l}" (feat_mask bit l) [N, h_l, w_l, C_l] fp32, the feature node
 * (before the ReLU for l == last_conv, after it otherwise); and in plans with a gradient request "G{l}" (l <= grad_conv)
 * [NB, h_l, w_l, C_l] bf16, the gradient w.r.t. conv l's pre-activation output, and "GP{l}" (pool after l, l < grad_conv)
 * [NB, h_l/2, w_l/2, C_l] bf16, that gradient on the pooled lattice. */
int b200sr_debug_buffer(const b200sr_plan* plan, const char* name, int64_t* offset_bytes, int64_t* bytes);

#ifdef __cplusplus
}
#endif
#endif /* B200SR_H_ */
