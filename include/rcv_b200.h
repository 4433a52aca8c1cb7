/*
 * rcv_b200.h -- C ABI of librcv_b200.so: the B200 (sm_100a) implementation of
 * RoboCupVision's one data-parallel hot path (encoder-decoder segmentation nets:
 * conv / transposed conv / BatchNorm / ReLU / max-pool / skip add, weighted
 * softmax cross-entropy, argmax + per-image confusion matrix, L1 + Adam tail).
 *
 * The reference has no FFI of its own: the arithmetic of this path lives behind
 * torch.nn calls in /root/reference/model.py.  Every entry point below names the
 * reference call site (file:line) whose arithmetic it replaces.  A maintainer
 * binds these with ctypes (see INTEGRATION.md); robocupvision_b200/_lib.py is
 * that binding.
 *
 * Conventions
 *   - plain C, POD structs, raw device pointers, sizes; no C++/torch types.
 *   - all tensors are fp32, NCHW, contiguous, unless stated; labels int64.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     makes no hidden synchronisation and allocates no device memory: the
 *     caller owns every buffer including workspaces.
 *   - return value: 0 = RCV_OK, negative = rcv_status.  Nothing throws or exits.
 *     rcv_last_error() returns a thread-local message for the last failure.
 *   - no fallbacks: an unsupported geometry is RCV_ERR_UNSUPPORTED, never a
 *     library/CPU path.
 */
#ifndef RCV_B200_H_
#define RCV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCV_ABI_VERSION 5

typedef enum rcv_status {
  RCV_OK = 0,
  RCV_ERR_BAD_ARG = -1,      /* null pointer / inconsistent sizes            */
  RCV_ERR_UNSUPPORTED = -2,  /* geometry outside the hot path (see DESIGN.md) */
  RCV_ERR_CUDA = -3,         /* launch / runtime error (message has detail)   */
  RCV_ERR_WORKSPACE = -4     /* workspace too small                           */
} rcv_status;

/* Epilogue applied to v = conv(x, w)[+bias] before it is stored
 * (model.py:116 `Conv`: bn(relu(conv)); model.py:175 `ConvPoolSimple` and
 * model.py:191-193 `upSampleTransposeConv`: relu(bn(conv)); model.py:137-138
 * `ConvPool`: relu(conv1)).  scale/shift are the folded eval-mode BatchNorm
 * (gamma/sqrt(var+eps), beta-mean*scale). */
typedef enum rcv_epilogue {
  RCV_EPI_NONE = 0,         /* y = v                         */
  RCV_EPI_RELU = 1,         /* y = max(v,0)                  */
  RCV_EPI_RELU_AFFINE = 2,  /* y = scale*max(v,0)+shift      */
  RCV_EPI_AFFINE_RELU = 3,  /* y = max(scale*v+shift,0)      */
  RCV_EPI_AFFINE = 4        /* y = scale*v+shift             */
} rcv_epilogue;

/* Math mode of the GEMM-shaped kernels. */
typedef enum rcv_math {
  RCV_MATH_FP32 = 0,     /* fp32 FFMA on CUDA cores (always available)          */
  RCV_MATH_TF32X3 = 1,   /* tcgen05 kind::tf32, 3-term error-compensated split,  *
                          * TMEM accumulators: fp32-level accuracy (~1e-6 of the *
                          * output range); needs packed weights (rcv_conv_pack)  */
  RCV_MATH_AUTO = 2,     /* the PARITY mode of the nets: TF32X3 where packed     *
                          * weights are given and the reduction is long enough   *
                          * to pay, else FP32 -- logits within 1e-4 of fp32      */
  /* Fast modes, reported separately from the parity mode (north_star: "bf16      *
   * variant stated separately"); engine choice as RCV_MATH_AUTO, the CUDA-core   *
   * layers (<= 16 output channels) stay exact fp32:                             */
  RCV_MATH_TF32 = 3,     /* one kind::tf32 MMA per product (operands rounded to  *
                          * 10 mantissa bits, fp32 accumulate): ~1e-3 per layer  */
  RCV_MATH_BF16 = 4      /* kind::f16 with bf16 operands (8 mantissa bits, fp32  *
                          * accumulate, activations stay fp32 in HBM) in the     *
                          * halo-staged stride-1 3x3 kernel where the reduced    *
                          * channel count is a multiple of 64; RCV_MATH_TF32 in  *
                          * the other tensor-core kernels.  The packed panel of  *
                          * a layer depends on the mode it was packed for.       */
} rcv_math;

/* Which operand a packed weight panel serves. */
typedef enum rcv_pack_dir {
  RCV_PACK_FWD = 0,      /* rcv_conv_fwd                                        */
  RCV_PACK_DGRAD = 1     /* rcv_conv_dgrad                                      */
} rcv_pack_dir;
#define RCV_DIR_WGRAD 2  /* rcv_conv_engine only: the weight gradient (no panel) */

/* One convolution-type layer.  transposed=0: nn.Conv2d(Cin,Cout,ksize,stride,
 * pad,dil) on x[N,Cin,H,W] (model.py:112,130-133,170,259,411,554).
 * transposed=1: nn.ConvTranspose2d(Cin,Cout,3,stride=2,padding=1,
 * output_padding=1) (model.py:186-187), x[N,Cin,H,W] -> y[N,Cout,2H,2W],
 * weight layout (Cin,Cout,3,3).  Supported: ksize 1 (stride 1, pad 0) and
 * ksize 3 with (stride,pad,dil) in {(1,1,1),(1,2,2),(2,1,1)}. */
typedef struct rcv_conv_desc {
  int32_t N, Cin, H, W; /* input tensor                                   */
  int32_t Cout;
  int32_t ksize, stride, pad, dil;
  int32_t transposed;
  int32_t epilogue;     /* rcv_epilogue (forward only)                    */
  int32_t math;         /* rcv_math                                       */
  /* Optional scratch for rcv_conv_fwd / rcv_conv_dgrad (NULL / 0: none).  Caller-owned device memory of at least
   * rcv_conv_workspace_bytes(d, direction) bytes, 128-byte aligned, ZERO-FILLED ONCE by the caller before its first
   * use (the kernels leave its counter area zeroed again), and used by one stream at a time.  With it the
   * halo-staged tensor-core kernel splits the reduction of the pixel tiles that do not fill a whole wave of SMs
   * across several CTAs (and of every tile when the layer has far fewer tiles than SMs: small batches);
   * without it, or when it is too small, the same layer runs unsplit -- results agree to accumulation order. */
  void* workspace;
  uint64_t workspace_bytes;
  /* rcv_conv_fwd: channels of the `residual` tensor (0 = Cout).  A value below Cout adds residual[N, res_channels,
   * Ho, Wo] to the FIRST res_channels output channels only -- the partial skip of LabelProp, `x[:, 0:8] += top`
   * (model.py:565) -- and is taken by the narrow-layer engine only (RCV_ERR_UNSUPPORTED elsewhere). */
  int32_t res_channels;
} rcv_conv_desc;

int rcv_version(void);
const char* rcv_last_error(void);

/* Programmatic dependent launch.  When on, every kernel of the library is launched with
 * cudaLaunchAttributeProgrammaticStreamSerialization: the next grid of the stream is set up while the current one
 * drains (every kernel starts with griddepcontrol.launch_dependents + griddepcontrol.wait, so data dependences stay
 * those of plain stream order; capture-safe).  Default: the RCV_PDL environment variable, else off.
 * rcv_set_pdl returns the previous setting. */
int rcv_set_pdl(int on);
int rcv_get_pdl(void);

/* Output spatial size of a layer (H_out, W_out). */
int rcv_conv_out_hw(const rcv_conv_desc* d, int32_t* Ho, int32_t* Wo);

/* ---- convolution family ------------------------------------------------- */

/* Weight panels for the tensor-core engine.  The nn.Conv2d / nn.ConvTranspose2d
 * weight tensor w (model.py:112,186) is re-laid out once per forward as the
 * engine's B operand: K-major rows in (tap, channel) order, split into tf32 hi
 * and lo parts, in the 128-byte-swizzled shared-memory image a CTA copies in
 * bulk.  packed must hold rcv_conv_packed_bytes(d, direction) bytes, 128-byte
 * aligned; it depends on the layer geometry only, not on N, H, W.  One launch. */
size_t rcv_conv_packed_bytes(const rcv_conv_desc* d, int direction);
/* 1 if rcv_conv_fwd / rcv_conv_dgrad (per direction) would run this layer on
 * the tensor cores under d->math when given packed weights, else 0: lets the
 * caller skip packing layers that stay on CUDA cores under RCV_MATH_AUTO. */
int rcv_conv_uses_tensor_cores(const rcv_conv_desc* d, int direction);
/* Bytes of scratch rcv_conv_fwd / rcv_conv_dgrad can use for this layer at this size (d->workspace; 0: none). */
size_t rcv_conv_workspace_bytes(const rcv_conv_desc* d, int direction);
int rcv_conv_pack(const rcv_conv_desc* d, int direction, const float* w,
                  void* packed, void* stream);

/* Which kernel family rcv_conv_fwd / rcv_conv_dgrad / rcv_conv_wgrad (direction RCV_PACK_FWD,
 * RCV_PACK_DGRAD, RCV_DIR_WGRAD) dispatches this layer to under d->math, given 16-byte aligned tensors and packed weights (tests and profiles name the
 * engine they measured).  Negative = rcv_status. */
typedef enum rcv_engine {
  RCV_ENGINE_SIMT = 0,    /* fp32 FFMA implicit GEMM (any geometry)                       */
  RCV_ENGINE_DIRECT = 1,  /* fp32 direct conv through L1 (<= 16 output channels, any width) */
  RCV_ENGINE_UMMA = 2,    /* tcgen05 3xTF32 implicit GEMM, TMEM accumulators               */
  RCV_ENGINE_NARROW = 3   /* fp32 FFMA2 direct conv / register-accumulating wgrad, TMA     *
                           * halo staging (<= 16 channels on the narrow side, widths that  *
                           * are multiples of 4)                                           */
} rcv_engine;
int rcv_conv_engine(const rcv_conv_desc* d, int direction);

/* Batched form: the panels of many layers in ONE launch (a train step re-packs every layer's
 * weights each step).  The caller builds a job table on the host once -- the weight and panel
 * device pointers must stay valid and unchanged -- copies it to device memory it owns
 * (rcv_conv_pack_table_bytes(n) bytes), and runs it on a stream whenever the weights changed.
 * njobs <= 128. */
size_t rcv_conv_pack_table_bytes(int32_t njobs);
int rcv_conv_pack_table_build(int32_t njobs, const rcv_conv_desc* descs,
                              const int32_t* directions, const float* const* weights,
                              void* const* packed, void* host_table, int64_t* total_chunks);
int rcv_conv_pack_table_run(const void* device_table, int32_t njobs,
                            int64_t total_chunks, void* stream);

/* y = EPI(conv(x,w) + bias) [+ residual].  wpacked (rcv_conv_pack of w,
 * RCV_PACK_FWD) may be NULL: the call then runs on CUDA cores (RCV_MATH_TF32X3
 * without it is RCV_ERR_BAD_ARG).  bias, scale, shift, residual,
 * stats may be NULL.  residual has the shape of y and is added after the
 * epilogue (decoder skip: model.py:300-307, 509).  If stats != NULL it is a
 * double[2*Cout] accumulator: stats[c] += sum(y_c), stats[Cout+c] += sum(y_c^2)
 * over this call's outputs (train-mode BatchNorm batch statistics of the
 * tensor BN consumes; caller zeroes it).
 * Replaces F.conv2d / F.conv_transpose2d (+ relu + eval batch_norm + add). */
int rcv_conv_fwd(const rcv_conv_desc* d, const float* x, const float* w,
                 const void* wpacked, const float* bias, const float* scale,
                 const float* shift,
                 const float* residual, float* y, double* stats, void* stream);

/* Normalise-on-load: rcv_conv_fwd on the tensor in_scale[c]*x + in_shift[c] (then ReLU if in_relu), i.e. on the
 * output of the BatchNorm block that produced x, without that output ever being written: the staging loop of the
 * halo-staged tensor-core kernel applies it to real pixels and keeps the zero padding zero.  in_scale / in_shift:
 * float[Cin] (rcv_bn_finalize's scale / shift).  Only layers for which rcv_conv_normalises_on_load(d) returns 1
 * (stride-1 3x3, Cin a multiple of 32, rows short enough for the kernel's patch) -- RCV_ERR_UNSUPPORTED otherwise.
 * Takes a training-mode BatchNorm apply pass (model.py:113, 171) off the forward critical path. */
int rcv_conv_normalises_on_load(const rcv_conv_desc* d);
int rcv_conv_fwd_nl(const rcv_conv_desc* d, const float* x, const float* in_scale,
                    const float* in_shift, int in_relu, const float* w, const void* wpacked,
                    const float* bias, const float* scale, const float* shift,
                    const float* residual, float* y, double* stats, void* stream);

/* dx = d(conv)/dx applied to dy (shape of y) [+ residual].  residual (may be
 * NULL, may alias dx) has the shape of dx: the gradient arriving at the same
 * tensor from a second consumer (the decoder skip), summed in the epilogue.
 * wpacked: rcv_conv_pack of w with RCV_PACK_DGRAD, or NULL (CUDA cores).
 * Replaces convolution_backward's input gradient (+ autograd's add). */
int rcv_conv_dgrad(const rcv_conv_desc* d, const float* dy, const float* w,
                   const void* wpacked, const float* residual, float* dx,
                   void* stream);

/* dw += d(conv)/dw, dbias += sum(dy) (dbias may be NULL).  Split over pixels
 * with fp32 atomic accumulation: the caller zeroes dw/dbias beforehand.
 * Replaces convolution_backward's weight/bias gradients. */
int rcv_conv_wgrad(const rcv_conv_desc* d, const float* x, const float* dy,
                   float* dw, float* dbias, void* stream);

/* Normalise-on-load for the weight gradient: rcv_conv_wgrad with in_scale[c]*x + in_shift[c] (then ReLU if
 * in_relu) in place of x -- the companion of rcv_conv_fwd_nl, so that the BatchNorm output the forward pass never
 * wrote does not have to be written for the backward pass either.  Only layers for which
 * rcv_conv_wgrad_normalises_on_load(d) returns 1 (tensor-core weight gradient with the quad gather: stride-1 3x3,
 * rows a multiple of 4 pixels wide, not transposed) -- RCV_ERR_UNSUPPORTED otherwise. */
int rcv_conv_wgrad_normalises_on_load(const rcv_conv_desc* d);
int rcv_conv_wgrad_nl(const rcv_conv_desc* d, const float* x, const float* in_scale,
                      const float* in_shift, int in_relu, const float* dy, float* dw,
                      float* dbias, void* stream);

/* ---- BatchNorm2d, training mode (model.py:113,134,171,188) --------------- */

/* From stats (sum, sum of squares over count = N*H*W elements per channel):
 * mean, biased var -> scale = gamma/sqrt(var+eps), shift = beta-mean*scale;
 * running_mean = (1-m)*running_mean + m*mean, running_var likewise with the
 * unbiased variance (either may be NULL); save_mean / save_invstd for the
 * backward pass; *num_batches_tracked += 1 (BatchNorm2d's int64 buffer; may be
 * NULL).  One tiny launch. */
int rcv_bn_finalize(int32_t C, int64_t count, const double* stats,
                    const float* gamma, const float* beta, float* running_mean,
                    float* running_var, float momentum, float eps, float* scale,
                    float* shift, float* save_mean, float* save_invstd,
                    int64_t* num_batches_tracked, void* stream);

/* Eval-mode fold (model.eval(), running statistics):
 * scale = gamma/sqrt(var+eps), shift = beta - mean*scale. */
int rcv_bn_fold(int32_t C, const float* gamma, const float* beta,
                const float* mean, const float* var, float eps, float* scale,
                float* shift, void* stream);

/* y = act(scale_c*z + shift_c) [+ residual], act = relu if relu!=0.
 * z,y: [N,C,HW].  res_channels: channels of residual (0 = C); below C, residual[N,res_channels,HW] is added to the
 * first res_channels channels only (LabelProp's partial skip, model.py:565). */
int rcv_bn_apply(int32_t N, int32_t C, int64_t HW, const float* z,
                 const float* scale, const float* shift, int relu,
                 const float* residual, int32_t res_channels, float* y, void* stream);

/* rcv_bn_finalize + rcv_bn_apply in one launch (the train-mode forward of a BatchNorm node):
 * every block derives scale/shift from stats; block 0 also writes scale, shift, save_mean,
 * save_invstd (for the backward pass), updates the running statistics and bumps
 * *num_batches_tracked (may be NULL). */
int rcv_bn_finalize_apply(int32_t N, int32_t C, int64_t HW, const double* stats,
                          const float* gamma, const float* beta, float* running_mean,
                          float* running_var, float momentum, float eps, const float* z,
                          int relu, const float* residual, int32_t res_channels, float* y, float* scale,
                          float* shift, float* save_mean, float* save_invstd,
                          int64_t* num_batches_tracked, void* stream);

/* Backward of y = act(scale*z+shift) composed with the producer's own ReLU.
 * order = RCV_EPI_RELU_AFFINE: z = relu(conv), y = bn(z)      (model.py:116)
 * order = RCV_EPI_AFFINE_RELU: z = conv,       y = relu(bn(z)) (model.py:175)
 * Pass 1 (reduce): sums[c] += sum(g), sums[C+c] += sum(g*xhat) with
 *   g = dy (RELU_AFFINE) or dy*[scale*z+shift>0] (AFFINE_RELU),
 *   xhat = (z-mean)*invstd.  sums is double[2*C], caller zeroes.
 * Pass 2 (apply): dz = scale*(g - sums[c]/cnt - xhat*sums[C+c]/cnt), then for
 *   RELU_AFFINE dz *= [z>0]; writes dconv (gradient w.r.t. the conv output),
 *   and accumulates dgamma[c] += sums[C+c], dbeta[c] += sums[c] (once, by the
 *   first block), dbias[c] += sum(dconv) if dbias != NULL.
 * Replaces native_batch_norm_backward + threshold_backward. */
int rcv_bn_bwd_reduce(int32_t N, int32_t C, int64_t HW, int order,
                      const float* dy, const float* z, const float* scale,
                      const float* shift, const float* save_mean,
                      const float* save_invstd, double* sums, void* stream);
int rcv_bn_bwd_apply(int32_t N, int32_t C, int64_t HW, int order,
                     const float* dy, const float* z, const float* scale,
                     const float* shift, const float* save_mean,
                     const float* save_invstd, const double* sums,
                     float* dconv, float* dgamma, float* dbeta, float* dbias,
                     void* stream);

/* rcv_bn_bwd_reduce + rcv_bn_bwd_apply as ONE call: a single launch (one thread-block cluster per channel, the
 * partial sums exchanged through distributed shared memory and added in rank order: bitwise reproducible) where the
 * channels split into <= 8 CTA-sized slices, else the two passes.  sums is only touched by the two-pass form. */
int rcv_bn_bwd_is_fused(int32_t N, int32_t C, int64_t HW);   /* host query: 1 = one launch, 0 = two */
int rcv_bn_bwd(int32_t N, int32_t C, int64_t HW, int order, const float* dy, const float* z,
               const float* scale, const float* shift, const float* save_mean, const float* save_invstd,
               double* sums, float* dconv, float* dgamma, float* dbeta, float* dbias, void* stream);

/* dx = dy * [y > 0] (threshold_backward for a stored ReLU output y). */
int rcv_relu_bwd(int64_t n, const float* dy, const float* y, float* dx,
                 void* stream);

/* dbias[c] += sum over (n, hw) of dy[n,c,hw]. */
int rcv_channel_sum(int32_t N, int32_t C, int64_t HW, const float* dy,
                    float* dbias, void* stream);

/* ---- MaxPool2d(2,2) (model.py:92-100) ----------------------------------- */
/* y[N,C,H/2,W/2]; idx (may be NULL) = int64 flat index h*W+w inside the (n,c)
 * plane, first maximum in row-major window order, NaN wins -- the convention
 * of F.max_pool2d(return_indices=True); code (may be NULL) = uint8 window
 * position 0..3 for the backward pass. */
int rcv_maxpool2x2_fwd(int32_t N, int32_t C, int32_t H, int32_t W,
                       const float* x, float* y, int64_t* idx, uint8_t* code,
                       void* stream);
/* dx[N,C,H,W] = scatter of dy through code (every dx element is written). */
int rcv_maxpool2x2_bwd(int32_t N, int32_t C, int32_t H, int32_t W,
                       const float* dy, const uint8_t* code, float* dx,
                       void* stream);

/* ---- decoder-side resampling extras (north_star: "a fused pool-index/unpool
 * pair", "transposed-conv/bilinear upsampling").  The reference has neither an
 * unpool nor a bilinear layer (model.py:178-194 is its only upsampler; "bilinear"
 * occurs only as a PIL resize, transform.py:8-19), so these replace the
 * torch.nn.functional calls a decoder variant would make and are pinned
 * against them. ------------------------------------------------------------- */
/* out[N,C,H,W] = F.max_unpool2d(y[N,C,H/2,W/2], idx, 2, 2) (+ skip[N,C,H,W] if
 * not NULL): positions from idx (int64 plane index, as rcv_maxpool2x2_fwd
 * writes) or, when idx is NULL, from the uint8 window codes.  Every element of
 * out is written. */
int rcv_maxunpool2x2_fwd(int32_t N, int32_t C, int32_t H, int32_t W,
                         const float* y, const int64_t* idx, const uint8_t* code,
                         const float* skip, float* out, void* stream);
/* dy[N,C,H/2,W/2] = dout[N,C,H,W] gathered at the stored positions. */
int rcv_maxunpool2x2_bwd(int32_t N, int32_t C, int32_t H, int32_t W,
                         const float* dout, const int64_t* idx,
                         const uint8_t* code, float* dy, void* stream);
/* out[N,C,2H,2W] = F.interpolate(x[N,C,H,W], scale_factor=2, mode="bilinear",
 * align_corners=False) (+ skip[N,C,2H,2W] if not NULL). */
int rcv_upsample_bilinear2x_fwd(int32_t N, int32_t C, int32_t H, int32_t W,
                                const float* x, const float* skip, float* out,
                                void* stream);
/* dx[N,C,H,W] = the adjoint applied to dout[N,C,2H,2W]. */
int rcv_upsample_bilinear2x_bwd(int32_t N, int32_t C, int32_t H, int32_t W,
                                const float* dout, float* dx, void* stream);

/* ---- classifier head of a training step, one pass ----------------------- */
/* The 1x1 classifier conv (model.py:259 UltClassifier / :411 / :554), CrossEntropyLoss2d (model.py:76-82), the
 * argmax / correct-pixel count (train.py:70-71) and the backward of all three in ONE pass over the decoder's last
 * feature map: logits = weight feat + bias; loss_sums[0] += sum_p w[y_p] nll_p; correct += #(argmax == y);
 * dlogits = gscale w[y_p] (softmax - onehot) / loss_sums[1]; dfeat = weight^T dlogits; dweight += dlogits feat^T;
 * dbias += dlogits.  Logits and their gradient never exist in memory.  Replaces, inside TrainStep, the sequence
 * rcv_conv_fwd (head) -> rcv_ce_fwd -> rcv_ce_bwd -> rcv_conv_dgrad + rcv_conv_wgrad (head).
 * loss_sums[1] must already hold sum_p w[y_p]: it depends on the labels only, rcv_ce_weight_sum adds it (to a zeroed
 * cell) any time before.  feat, dfeat [N,Cin,HW]; weight, dweight [C,Cin]; bias, dbias [C] or NULL; target int64
 * [N,HW] (labels outside [0,C) contribute nothing); class_w [C] or NULL; gscale device float or NULL (1).
 * Supported (rcv_head_ce_supported): 2..8 classes over 8 or 16 channels; anything else RCV_ERR_UNSUPPORTED and the
 * caller keeps the unfused sequence. */
int rcv_head_ce_supported(int32_t Cin, int32_t C);
int rcv_ce_weight_sum(int32_t C, int64_t count, const int64_t* target, const float* class_w, double* out,
                      void* stream);
int rcv_head_ce_train(int32_t N, int32_t Cin, int32_t C, int64_t HW, const float* feat, const float* weight,
                      const float* bias, const int64_t* target, const float* class_w, const float* gscale,
                      double* loss_sums, int64_t* correct, float* dfeat, float* dweight, float* dbias,
                      void* stream);

/* ---- classifier head of a Dice-loss training step, two passes ------------ */
/* The 1x1 classifier conv, DiceLoss (model.py:5-43, the --useDice option), the argmax / correct-pixel count and their
 * backward in TWO passes over the decoder's last feature map (the Dice gradient of every pixel depends on the
 * batch-wide sums, so one pass cannot do it).  Replaces, inside TrainStep(loss="dice"), the sequence rcv_conv_fwd
 * (head) -> rcv_dice_fwd -> rcv_dice_bwd -> rcv_conv_dgrad + rcv_conv_wgrad (head); the logits and their gradient
 * never exist in memory.  Shapes as rcv_head_ce_train: feat, dfeat [N,Cin,HW]; weight, dweight [C,Cin]; bias, dbias
 * [C] or NULL; target int64 [N,HW].  Pixels labelled outside [0,C) contribute nothing, to the sums or to the
 * gradient (rcv_dice_fwd adds their softmax to the cardinality).  Supported: what rcv_head_ce_supported accepts (2..8
 * classes over 8 or 16 channels); anything else RCV_ERR_UNSUPPORTED.
 * Pass 1, rcv_head_dice_fwd: logits = weight feat + bias; sums (double[2*C], caller zeroes) as rcv_dice_fwd:
 * sums[c] += sum_p softmax_c(p)*[y_p==c], sums[C+c] += sum_p (softmax_c(p) + [y_p==c]); correct (int64[1] or NULL)
 * += #(argmax == y), lowest class index among equal maxima. */
int rcv_head_dice_fwd(int32_t N, int32_t Cin, int32_t C, int64_t HW, const float* feat, const float* weight,
                      const float* bias, const int64_t* target, double* sums, int64_t* correct, void* stream);
/* Pass 2, rcv_head_dice_train, after pass 1 on the same stream: with the finished sums, a_c = 2 w_c / (C (K_c+eps)),
 * b_c = 2 w_c I_c / (C (K_c+eps)^2) (I_c = sums[c], K_c = sums[C+c]), g_c = -a_c [y==c] + b_c and
 * dlogits_j = gscale p_j (g_j - sum_c p_c g_c), exactly rcv_dice_bwd's arithmetic; dfeat = weight^T dlogits (written);
 * dweight += dlogits feat^T; dbias += dlogits.  weights: the normalised w (device float[C], w = weights/sum*C on the
 * host as DiceLoss does; NULL = 1); gscale device float or NULL (1).  loss (double[2] or NULL) = [1 - mean_c(2 w_c
 * I_c / (K_c+eps)), 1.0]: a numerator / denominator pair, so readers of the CE loss sums read it unchanged. */
int rcv_head_dice_train(int32_t N, int32_t Cin, int32_t C, int64_t HW, const float* feat, const float* weight,
                        const float* bias, const int64_t* target, const float* weights, const double* sums, float eps,
                        const float* gscale, double* loss, float* dfeat, float* dweight, float* dbias, void* stream);
/* loss (double[2]) = [1 - mean_c(2 w_c sums[c] / (sums[C+c] + eps)), 1.0] from the sums of rcv_dice_fwd: the loss
 * cell of rcv_head_dice_train for the unfused Dice step, one single-thread launch.  weights as above, C = 2..8. */
int rcv_dice_loss(int32_t C, const double* sums, const float* weights, float eps, double* loss, void* stream);

/* dst[n, dst_offset + c, :] = src[n, src_offset + c, :] for c < count; src [N,src_channels,HW], dst
 * [N,dst_channels,HW].  The channel moves of the skip wiring that no producer can fold: ROBO_UNet --v2's
 * torch.cat([layer(up), downs[-(i+2)]], 1) (model.py:507; two calls fill the concatenated tensor), the gradient
 * halves autograd slices back out of it, and the gradient of LabelProp's partial skip (model.py:565). */
int rcv_channel_copy(int64_t N, int64_t HW, int32_t count, const float* src, int32_t src_channels,
                     int32_t src_offset, float* dst, int32_t dst_channels, int32_t dst_offset, void* stream);

/* ---- weighted softmax cross-entropy + argmax + confusion ----------------- */
/* CrossEntropyLoss2d (model.py:76-82), torch.max(pred,1) (train.py:70,128) and
 * the per-image confusion loop (train.py:133-153) in one pass over the logits.
 * logits [N,C,HW] (C <= 8), target int64 [N,HW] in [0,C), class_w [C] or NULL.
 * loss_sums: double[2]: += sum_p w[y_p]*nll_p, += sum_p w[y_p]  (caller zeroes;
 *   loss = loss_sums[0]/loss_sums[1]).
 * argmax   : int64 [N,HW] or NULL; lowest class index among equal maxima.
 * conf     : int64 [N,C,C] or NULL; conf[n,p,l] += #(argmax==p and target==l).
 * correct  : int64[1] or NULL; += #(argmax==target).  */
int rcv_ce_fwd(int32_t N, int32_t C, int64_t HW, const float* logits,
               const int64_t* target, const float* class_w, double* loss_sums,
               int64_t* argmax, int64_t* conf, int64_t* correct, void* stream);
/* dlogits = gscale * w[y_p]*(softmax(z_p) - onehot(y_p)) / loss_sums[1];
 * gscale (device float, may be NULL = 1) is the upstream gradient. */
int rcv_ce_bwd(int32_t N, int32_t C, int64_t HW, const float* logits,
               const int64_t* target, const float* class_w,
               const double* loss_sums, const float* gscale, float* dlogits,
               void* stream);
/* conf[n,p,l] += #(pred==p and target==l) from two int64 label maps. */
int rcv_confusion(int32_t N, int32_t C, int64_t HW, const int64_t* pred,
                  const int64_t* target, int64_t* conf, void* stream);

/* The tail of the validation loops (train.py:148-163) on the device: iou_sum[c] (double[C], overwritten) = sum over
 * the N images of inter/union per class from the per-image confusion counts conf int64[N,C,C] (union = row + column
 * - diagonal; an image without the class counts 1, train.py:152-153), and *loss (double, may be NULL) =
 * loss_sums[0] / loss_sums[1] of rcv_ce_fwd.  One launch, no host round trip (the reference does 25*B .item() calls). */
int rcv_metric_tail(int32_t N, int32_t C, const int64_t* conf, const double* loss_sums,
                    double* iou_sum, double* loss, void* stream);

/* ---- input-side label ops of the callers --------------------------------- */
/* labels[i] = lut[labels[i]] in place for 0 <= labels[i] < nlut (nlut <= 64): maskLabel,
 * transform.py:26-49 (the class-drop relabel is a permutation-with-merges of 0..4). */
int rcv_label_lut(int64_t n, int64_t* labels, int32_t nlut, const int64_t* lut, void* stream);
/* out[b,c,p] = labels[b,p]==c ? +1 : -1, float [B,C,HW]: labelToPred, transform.py:172-183. */
int rcv_label_to_pred(int64_t B, int32_t C, int64_t HW, const int64_t* labels, float* out,
                      void* stream);
/* The two mirrored LabelProp samples of each of P frame pairs (labelPropTrain.py:178-193):
 * inputs[2q]   = (Y_a, Y_b, Y_a-Y_b, labelToPred(lab_b)), targets[2q]   = lab_a
 * inputs[2q+1] = (Y_b, Y_a, Y_b-Y_a, labelToPred(lab_a)), targets[2q+1] = lab_b
 * ya, yb float [P,HW]; la, lb int64 [P,HW]; inputs float [2P,3+C,HW]; targets int64 [2P,HW]. */
int rcv_lp_assemble(int64_t P, int32_t C, int64_t HW, const float* ya, const float* yb,
                    const int64_t* la, const int64_t* lb, float* inputs, int64_t* targets,
                    void* stream);

/* Training-split augmentation of SSYUVDataset.__getitem__ (dataset.py:123-131) over a whole batch:
 * Normalize ((x - mean[c]) / std[c], mean / std: HOST arrays of 3 floats), horizontal flip of image and
 * label (img.flip(2)), ColorJitter (dataset.py:19-39: y0 = (y0 + b) * c; (u, v) = M (u, v)).  Per-image
 * parameters in DEVICE memory, params[n] = {flip (0/1), b, c, m00, m01, m10, m11, unused}: the caller draws
 * them (random.uniform in the reference) -- the kernel is deterministic.  x, y float [N,3,H,W] (not in
 * place); labels_in / labels_out int64 [N,H,W] or both NULL. */
int rcv_augment(int32_t N, int32_t H, int32_t W, const float* x, float* y,
                const int64_t* labels_in, int64_t* labels_out, const float* params,
                const float* mean, const float* std_, void* stream);

/* ---- DiceLoss (model.py:5-43, the --useDice option), C = 2..8 classes ----- */
/* sums (double[2*C], caller zeroes): sums[c] += sum_p softmax_c(p)*[y_p==c] (intersection),
 * sums[C+c] += sum_p (softmax_c(p) + [y_p==c]) (cardinality).
 * loss = 1 - mean_c(2*w_c*sums[c] / (sums[C+c] + eps)), w = weights/sum(weights)*C (host side). */
int rcv_dice_fwd(int32_t N, int32_t C, int64_t HW, const float* logits,
                 const int64_t* target, double* sums, void* stream);
/* dlogits = gscale * dloss/dlogits through the softmax; weights: the normalised w (device, may be NULL = 1),
 * gscale: device float or NULL (= 1). */
int rcv_dice_bwd(int32_t N, int32_t C, int64_t HW, const float* logits,
                 const int64_t* target, const float* weights, const double* sums,
                 float eps, const float* gscale, float* dlogits, void* stream);

/* ---- train-step tail: L1 regulariser + pruning mask + Adam --------------- */
/* One fused pass over a flat parameter range (train.py:23-27 l1reg, 59-65 grad
 * mask, torch.optim.Adam defaults amsgrad=False, weight_decay=0):
 *   g = grad_scale*g + l1_decay*sign(p); if mask && mask[i]: g = 0;
 *   m = b1*m+(1-b1)*g; v = b2*v+(1-b2)*g*g;
 *   p -= lr * (m/(1-b1^t)) / (sqrt(v/(1-b2^t)) + eps)
 * l1_sum (double[1], may be NULL) += sum |p| (before the update).  step = t>=1. */
int rcv_adam_l1_step(int64_t n, float* p, const float* g, float* m, float* v,
                     const uint8_t* mask, float lr, float beta1, float beta2,
                     float eps, int32_t step, float l1_decay, float grad_scale,
                     double* l1_sum, const int32_t* step_dev, const float* lr_dev,
                     void* stream);
/* *counter += inc on the stream (the device-resident Adam step count used when
 * the train step is replayed from a CUDA graph: step_dev / lr_dev above, when
 * non-NULL, override the host `step` / `lr`). */
int rcv_counter_add(int32_t* counter, int32_t inc, void* stream);
/* SGD with momentum/dampening=0/weight decay (trainer.py:182-184), with the same
 * optional L1 sub-gradient, pruning mask and device-resident learning rate as
 * rcv_adam_l1_step:
 *   g = grad_scale*g + l1_decay*sign(p); masked -> 0; g += wd*p;
 *   buf = mom*buf + g (buf = g at first_step; a zero-filled buf gives the same
 *   first step, so graph replays pass first_step = 0); p -= lr*buf.
 * l1_sum (double[1], may be NULL) += sum |p| before the update; lr_dev (device
 * float, may be NULL) overrides lr. */
int rcv_sgd_step(int64_t n, float* p, const float* g, float* buf,
                 const uint8_t* mask, float lr, float momentum,
                 float weight_decay, float grad_scale, int first_step,
                 float l1_decay, double* l1_sum, const float* lr_dev,
                 void* stream);

/* Stream-ordered zero fill of `bytes` bytes (cudaMemsetAsync: a memset node, not a
 * kernel, inside a captured graph): the accumulators a step sums into -- gradient
 * arena (optimizer.zero_grad(), train.py:45), BatchNorm statistics, loss sums. */
int rcv_zero(void* ptr, size_t bytes, void* stream);

/* ---- deterministic (fixed-order) reductions ------------------------------ */
/* The entry points above add each CTA's partial sums into their destination with floating-point atomics, so the
 * order of the additions, and the last bits of the result, change from run to run.  Each _det variant below computes
 * exactly what its plain form computes, with one difference: every CTA parks its partial vector in a slot of
 * `scratch` fixed by the launch geometry, and the CTA that arrives last adds the slots into the destination in an
 * order fixed by the launch geometry (never by the arrival order).  Same inputs on the same device: bitwise the same result, run after run (torch.use_deterministic_algorithms,
 * the reference's seeded CPU runs).  It differs from the plain form in summation order only.
 * scratch: caller-owned device memory of at least rcv_det_scratch_bytes(op, ...) bytes, 128-byte aligned,
 * ZERO-FILLED ONCE by the caller before its first use (the kernels leave it ready for the next call), used by one
 * stream at a time; too small is RCV_ERR_WORKSPACE.  The scratch needed depends on the grid, which follows the
 * problem size and the device. */
typedef enum rcv_det_op {
  RCV_DET_CE_FWD = 0,         /* rcv_ce_fwd_det: N images of HW pixels (C ignored)                  */
  RCV_DET_CE_WEIGHT_SUM = 1,  /* rcv_ce_weight_sum_det: count = N*HW labels (C ignored)             */
  RCV_DET_DICE_FWD = 2,       /* rcv_dice_fwd_det: N images of HW pixels, C classes                 */
  RCV_DET_L1_SUM = 3          /* rcv_adam_l1_step_det / rcv_sgd_step_det: n = N*HW parameters      */
} rcv_det_op;
/* Bytes of scratch the _det entry point of `op` needs for this problem; 0 for an unknown op or a problem the entry
 * point refuses.  Host only: needs no GPU. */
size_t rcv_det_scratch_bytes(int op, int32_t N, int32_t C, int64_t HW);

/* rcv_ce_fwd with loss_sums in fixed order: CrossEntropyLoss2d (model.py:76-82).  argmax / conf / correct are integer counts and exact either way.  scratch may be NULL when
 * loss_sums is NULL. */
int rcv_ce_fwd_det(int32_t N, int32_t C, int64_t HW, const float* logits,
                   const int64_t* target, const float* class_w, double* loss_sums,
                   int64_t* argmax, int64_t* conf, int64_t* correct, void* scratch,
                   uint64_t scratch_bytes, void* stream);
/* rcv_ce_weight_sum in fixed order: the normaliser sum_p w[y_p] of CrossEntropyLoss2d's weighted mean
 * (model.py:76-82); the atomic form is exact only when the class weights are integers. */
int rcv_ce_weight_sum_det(int32_t C, int64_t count, const int64_t* target, const float* class_w,
                          double* out, void* scratch, uint64_t scratch_bytes, void* stream);
/* rcv_dice_fwd in fixed order: DiceLoss's intersection and cardinality sums (model.py:5-43). */
int rcv_dice_fwd_det(int32_t N, int32_t C, int64_t HW, const float* logits,
                     const int64_t* target, double* sums, void* scratch,
                     uint64_t scratch_bytes, void* stream);
/* rcv_adam_l1_step / rcv_sgd_step with l1_sum in fixed order: the L1 term the reference adds to the reported loss
 * (train.py:23-27).  The parameter updates are element-wise and identical to the plain forms.  scratch may be
 * NULL when l1_sum is NULL. */
int rcv_adam_l1_step_det(int64_t n, float* p, const float* g, float* m, float* v,
                         const uint8_t* mask, float lr, float beta1, float beta2,
                         float eps, int32_t step, float l1_decay, float grad_scale,
                         double* l1_sum, const int32_t* step_dev, const float* lr_dev,
                         void* scratch, uint64_t scratch_bytes, void* stream);
int rcv_sgd_step_det(int64_t n, float* p, const float* g, float* buf,
                     const uint8_t* mask, float lr, float momentum,
                     float weight_decay, float grad_scale, int first_step,
                     float l1_decay, double* l1_sum, const float* lr_dev,
                     void* scratch, uint64_t scratch_bytes, void* stream);

/* ---- data-parallel gradient exchange over NVLink peer memory ------------- */
/* The one exchange of batch-sharded training: the sum all-reduce of the flat gradient arena after
 * `loss.backward()` (train.py:66; what DistributedDataParallel adds to the reference's loop), as ONE kernel per
 * bucket over peer-mapped arenas instead of a collective-library call: a ready barrier (flags in peer memory), each
 * rank sums its 1/N share of the range over all ranks' arenas IN RANK ORDER (bitwise the same result whichever rank
 * computes it) and stores the sums into every arena, then a done barrier.  When the launch completes, the range of
 * the local arena holds the sums and no peer touches it until the next launch on the same slot.
 *
 * Setup, once per rank: rcv_peer_alloc (a zero-filled cudaMalloc block + its 64-byte cudaIpc handle), exchange the
 * handles through any host channel, rcv_peer_open each peer's handle.  The block holds the arena followed by
 * rcv_peer_flag_bytes() of flags (16-byte aligned); a rank passes its OWN block for its own index. */
uint64_t rcv_peer_flag_bytes(void);
int rcv_peer_alloc(uint64_t bytes, void** ptr, void* handle64);
int rcv_peer_open(const void* handle64, void** ptr);
int rcv_peer_close(void* ptr);   /* a pointer rcv_peer_open returned  */
int rcv_peer_free(void* ptr);    /* a pointer rcv_peer_alloc returned */
/* arenas[world], flags[world]: HOST arrays of device pointers in rank order (own block included).  slot: 0..15, one
 * per concurrently outstanding range (every rank must issue the same sequence of launches per slot).  offset, count:
 * floats, multiples of 4.  status: device int32 in local memory, set to 1 if a peer did not arrive within
 * RCV_PEER_TIMEOUT_S (default 30) seconds -- the launch then returns without hanging and the sums are invalid.
 * world = 1 is legal (flags and barriers run, the sums are the gradients themselves). */
int rcv_peer_allreduce(int32_t world, int32_t rank, int32_t slot, float* const* arenas, uint32_t* const* flags,
                       int64_t offset, int64_t count, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RCV_B200_H_ */
