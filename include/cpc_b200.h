/*
 * cpc_b200.h -- C-ABI of the B200-native CPC training hot path.
 *
 * The reference (vincentherrmann/constrastive-predictive-coding-audio) is pure Python/PyTorch and has
 * no FFI of its own; this header is the boundary the new implementation defines (SURVEY.md 8b).  Each
 * entry point replaces the ATen library calls the reference makes at the cited file:line.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name says `host`;
 *   - the caller owns every buffer (PyTorch's caching allocator in practice); nothing is allocated,
 *     freed or cached inside; no global or thread-local state (autograd calls backward from another
 *     thread than forward);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it, no host
 *     synchronisation inside;
 *   - `workspace` / `workspace_bytes`: scratch the caller provides, size from the matching
 *     *_workspace_bytes(); contents are undefined before and after the call;
 *   - return value: CPC_OK (0) or a negative cpc_status; cpc_status_string() names it.  On error nothing
 *     has been enqueued.
 *   - the library only runs on compute capability 10.x (sm_100a); CPC_ERR_ARCH otherwise.  There is no
 *     CPU fallback anywhere.
 */
#ifndef CPC_B200_H
#define CPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cpc_status {
    CPC_OK = 0,
    CPC_ERR_BAD_SHAPE = -1,     /* a dimension is non-positive / inconsistent            */
    CPC_ERR_ALIGNMENT = -2,     /* pointer or pitch violates the stated alignment        */
    CPC_ERR_WORKSPACE = -3,     /* workspace too small or NULL                           */
    CPC_ERR_ARCH = -4,          /* current device is not sm_100                          */
    CPC_ERR_CUDA = -5,          /* a CUDA runtime call (launch) failed                   */
    CPC_ERR_UNSUPPORTED = -6,   /* valid request this build has no kernel for            */
    CPC_ERR_NULL = -7           /* required pointer is NULL                              */
} cpc_status;

const char* cpc_status_string(int status);
/* ABI version; bumped on any signature change. */
int cpc_abi_version(void);
/* CPC_OK when the current CUDA device can run this library (sm_100), else CPC_ERR_ARCH / CPC_ERR_CUDA. */
int cpc_runtime_check(void);
/* Number of kernels this library has launched since load (process-wide atomic counter; bench.py's
 * "gpu_launches").  cpc_launch_count_reset() zeroes it. */
uint64_t cpc_launch_count(void);
void cpc_launch_count_reset(void);

/* ------------------------------------------------------------------------------------------------
 * 1. Constant-Q front end: complex filterbank correlation (+ fused log-power / phase / pooling).
 *    Replaces CQT.forward (constant_q_transform.py:161-172: 9 strided F.conv1d + chunk/cat/stack) and
 *    PreprocessingModule.forward (scalogram_model.py:75-102: abs, pow, log, atan2, phase difference,
 *    unwrap, max_pool2d, scale, power -- about 20 ATen launches) .
 * ---------------------------------------------------------------------------------------------- */
#define CPC_CQT_MAX_GROUPS 16

typedef enum cpc_cqt_mode {
    CPC_CQT_COMPLEX = 0,   /* out (B, n_bins, T, 2) fp32: what CQT.forward returns                         */
    CPC_CQT_LOGPOW = 1,    /* out (B, 1, n_bins, T/pool_t): ((log(re^2+im^2+eps)+log_offset)*norm)^power   */
    CPC_CQT_LOGPOW_PHASE = 2 /* out (B, 2, n_bins, (T-1)/pool_t): channel 0 as above on frames 1..T-1,
                                channel 1 = unwrap(phi_t - phi_{t-1} + fixed[f]) * scale[f], then *norm, ^power */
} cpc_cqt_mode;

typedef struct cpc_cqt_params {
    int32_t batch;          /* B                                                                      */
    int32_t n_samples;      /* L: samples per item (the last one is never read, as in the reference)   */
    int32_t x_pitch;        /* elements between consecutive items of x (>= L)                          */
    int32_t n_bins;         /* F                                                                      */
    int32_t hop;            /* hop_length                                                             */
    int32_t n_frames;       /* T = floor((L - 1 - kernel_size[0]) / hop) + 1                           */
    int32_t n_groups;       /* octave groups, <= CPC_CQT_MAX_GROUPS                                    */
    int32_t kernel_size[CPC_CQT_MAX_GROUPS];  /* K_g, non-increasing; group g reads x[off_g + hop*t + n],
                                                 off_g = (K_0 - K_g)/2  (constant_q_transform.py:165-166) */
    int32_t bin_lo[CPC_CQT_MAX_GROUPS];       /* group g covers bins [bin_lo, bin_hi)                  */
    int32_t bin_hi[CPC_CQT_MAX_GROUPS];
    int64_t weight_offset[CPC_CQT_MAX_GROUPS];/* element offset inside `weights` of group g's block:
                                                 (2*n_g, K_g) row-major fp32, rows [real bins; imag bins] */
    int32_t mode;           /* cpc_cqt_mode                                                           */
    int32_t pool_t;         /* 1, or 2 = max over adjacent frame pairs (scalogram_pooling=[1,2])       */
    float eps;              /* added to the power before log (0 or 1e-9)                              */
    float log_offset;       /* added after log                                                       */
    float norm;             /* multiplied after the offset                                           */
    float power;            /* exponent applied last (1 = skipped)                                   */
    int32_t flags;          /* CPC_CQT_FLAG_*: kernel selection switches (A/B tests); 0 = default     */
} cpc_cqt_params;
#define CPC_CQT_FLAG_NO_TENSOR 1   /* every octave group on the fp32 CUDA-core kernels                  */
#define CPC_CQT_FLAG_HALF_OPERANDS 2 /* tensor-core groups on ONE fp16 plane per operand (11-bit mantissas after the exact
                                      power-of-two scaling; ~2e-4 relative) instead of the fp32-accurate hi/lo pair: the front
                                      end of the bf16 operand mode (cpc_conv_params.precision = 1 downstream)            */

size_t cpc_cqt_workspace_bytes(const cpc_cqt_params* p);
/* x (B, x_pitch) fp32; weights: packed group blocks, fp32; phase_fixed / phase_scale: (n_bins) fp32, only
 * read in CPC_CQT_LOGPOW_PHASE (PhaseDifference, constant_q_transform.py:275-286); out: see cpc_cqt_mode. */
int cpc_cqt_fwd(const float* x, const float* weights, const float* phase_fixed, const float* phase_scale,
                float* out, const cpc_cqt_params* p, void* workspace, size_t workspace_bytes, void* stream);
/* The tensor-core filterbank reads the filters as scaled fp16 hi/lo planes.  That form only depends on the weights
 * (fixed after CQT.__init__, constant_q_transform.py:141-146, unless trainable): cpc_cqt_pack_filters writes it once
 * into a caller-owned buffer of cpc_cqt_packed_filter_bytes (0 = this configuration has no tensor-core path) and
 * cpc_cqt_fwd_ex takes it back on every call (packed_filters == NULL: packed into the workspace per call, as cpc_cqt_fwd
 * does).  The packed form depends on the filterbank fields of p only (groups, bins, hop), not on batch / length. */
size_t cpc_cqt_packed_filter_bytes(const cpc_cqt_params* p);
int cpc_cqt_pack_filters(const float* weights, void* packed, const cpc_cqt_params* p, void* stream);
int cpc_cqt_fwd_ex(const float* x, const float* weights, const void* packed_filters, const float* phase_fixed,
                   const float* phase_scale, float* out, const cpc_cqt_params* p, void* workspace, size_t workspace_bytes,
                   void* stream);

/* ------------------------------------------------------------------------------------------------
 * 2. Strided convolution, forward / data gradient / weight gradient.  conv1d is h = 1.
 *    Replaces nn.Conv1d in AudioEncoder (audio_model.py:30-44) and nn.Conv2d (+ the preceding
 *    nn.ZeroPad2d) in ScalogramEncoder / ScalogramEncoderBlock (scalogram_model.py:155-201, 387-431),
 *    and their autograd (cuDNN dgrad / wgrad) in loss.backward() (contrastive_estimation_training.py:161).
 *    Tensors are NCHW fp32, contiguous.  Cross-correlation (PyTorch convention), groups = 1, dilation 1.
 * ---------------------------------------------------------------------------------------------- */
typedef struct cpc_conv_params {
    int32_t batch;
    int32_t c_in, h_in, w_in;
    int32_t c_out, h_out, w_out;
    int32_t kh, kw;
    int32_t stride_h, stride_w;
    int32_t pad_top, pad_left;   /* zero rows above / columns left of the input (ZeroPad2d top padding is
                                    folded in here); bottom / right padding is implied by h_out / w_out   */
    int32_t relu;                /* forward only: fuse max(.,0) into the epilogue                          */
    int32_t precision;           /* 0 = fp32-faithful (error <= 1e-5 relative), 1 = bf16 operands           */
    int32_t flags;               /* CPC_CONV_FLAG_*: kernel selection switches (A/B tests); 0 = default     */
} cpc_conv_params;
#define CPC_CONV_FLAG_CUDA_CORE 1        /* no tensor-core kernel at all: the fp32 CUDA-core kernels          */
#define CPC_CONV_FLAG_NO_TALL 2          /* kh x 1 convolutions on the generic tcgen05 kernel                 */
#define CPC_CONV_FLAG_NO_SMALLK 4        /* tiny-K convolutions on the tiled kernels                          */
#define CPC_CONV_FLAG_NO_FUSED_DGRAD 8   /* stride-2 data gradient as one launch per parity class             */
#define CPC_CONV_FLAG_NO_MMA_SMALL_WGRAD 16 /* tiny-K weight gradient on the FMA kernel instead of mma.sync      */

size_t cpc_conv_workspace_bytes(const cpc_conv_params* p, int which /* 0 fwd, 1 dgrad, 2 wgrad */);
/* y = conv(x, w) + bias (bias may be NULL). */
int cpc_conv_fwd(const float* x, const float* w, const float* bias, float* y, const cpc_conv_params* p,
                 void* workspace, size_t workspace_bytes, void* stream);
/* dx = conv_transpose(dy, w); every element of dx is written. */
int cpc_conv_dgrad(const float* dy, const float* w, float* dx, const cpc_conv_params* p,
                   void* workspace, size_t workspace_bytes, void* stream);
/* dw (c_out, c_in, kh, kw) and, when dbias != NULL, dbias (c_out); both overwritten (not accumulated). */
int cpc_conv_wgrad(const float* x, const float* dy, float* dw, float* dbias, const cpc_conv_params* p,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Depthwise convolution (groups = channels, c_out == c_in, weight (C, 1, kh, kw), no bias): the first half of
 * Conv2dSeparable (scalogram_model.py:532-544; the 1x1 half is cpc_conv_*).  Same geometry fields as above;
 * relu / precision / flags are ignored (fp32 CUDA-core arithmetic, memory-bound). */
int cpc_dwconv_fwd(const float* x, const float* w, float* y, const cpc_conv_params* p, void* stream);
int cpc_dwconv_dgrad(const float* dy, const float* w, float* dx, const cpc_conv_params* p, void* stream);
int cpc_dwconv_wgrad(const float* x, const float* dy, float* dw, const cpc_conv_params* p, void* stream);

/* Which kernel family serves this configuration (for profiling / reporting; which: 0 fwd, 1 dgrad, 2 wgrad):
 * 0 tiled fp32 CUDA-core GEMM, 1 direct small-K kernel, 2 row-streaming tcgen05 (32 -> 32 channels, conv_tall.cu),
 * 3 row-streaming tcgen05 (128 output channels, conv_tall128.cu), 4 generic implicit-GEMM tcgen05; -1 bad params. */
int cpc_conv_kernel_family(const cpc_conv_params* p, int which);

/* Optional operand caching.  The tensor-core kernels read bf16 hi/lo planes of their activation operand; by
 * default every call re-packs its fp32 inputs into the workspace.  A caller that keeps tensors across calls (an
 * autograd Function keeps x from forward to backward, and uses dy for both gradients) can pack each operand
 * once with cpc_conv_pack() and hand the result to the *_ex entry points (a NULL packed pointer = pack
 * internally; the fp32 tensor must always be passed too, some kernel families read it directly).
 *   operand 0: x   operand 1: dy.   cpc_conv_packed_bytes() == 0: this configuration does not use a packed copy.
 *   `packed` must be 16-byte aligned (it becomes a TMA global base address). */
size_t cpc_conv_packed_bytes(const cpc_conv_params* p, int operand);
int cpc_conv_pack(const float* src, void* packed, const cpc_conv_params* p, int operand, void* stream);
/* cpc_conv_pack(dy, ..., operand = 1) that also writes the bias gradient dbias[c_out] = sum over (b, h, w) of dy when
 * dbias is non-NULL: dy is read once for both (contrastive_estimation_training.py:161, autograd of the conv biases). */
int cpc_conv_pack_dy(const float* dy, void* packed, float* dbias, const cpc_conv_params* p, void* stream);
int cpc_conv_fwd_ex(const float* x, const float* w, const float* bias, float* y, const cpc_conv_params* p,
                    const void* packed_x, void* workspace, size_t workspace_bytes, void* stream);
int cpc_conv_dgrad_ex(const float* dy, const float* w, float* dx, const cpc_conv_params* p, const void* packed_dy,
                      void* workspace, size_t workspace_bytes, void* stream);
int cpc_conv_wgrad_ex(const float* x, const float* dy, float* dw, float* dbias, const cpc_conv_params* p,
                      const void* packed_x, const void* packed_dy, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 2b. Fused BatchNorm2d + ReLU (+ centre-cropped residual add + ReLU), forward and backward.
 *    Replaces nn.BatchNorm2d / nn.ReLU after each conv of ScalogramEncoderBlock (scalogram_model.py:399-431),
 *    the residual crop-and-add (scalogram_model.py:451-472) and the F.relu between blocks (:523-527), and
 *    their autograd (cuDNN batch-norm backward, threshold_backward, slice_backward, add).
 *        v   = relu_if(relu, gamma * (x - mean) * rstd + beta)
 *        out = relu_if(outer_relu, v + residual[:, :, res_off_h : res_off_h + H, res_off_w : res_off_w + W])
 *    x / out / dout / dx: (B, C, H, W) contiguous fp32; residual / d_residual: (B, C, res_height, res_width).
 * ---------------------------------------------------------------------------------------------- */
typedef struct cpc_bn_params {
    int32_t batch, channels, height, width;
    int32_t res_height, res_width;   /* 0, 0: no residual operand                                          */
    int32_t res_off_h, res_off_w;    /* crop origin inside the residual plane                              */
    int32_t relu;                    /* ReLU directly after the normalisation                              */
    int32_t outer_relu;              /* ReLU after the residual add (ignored without residual)             */
    int32_t training;                /* 1: batch statistics, running stats updated (nn.BatchNorm2d.train());
                                        0: running statistics (eval())                                     */
    float eps, momentum;
    int32_t packed_planes;           /* *_packed variants only: 0 or 2 = bf16 hi + lo planes (operands of an fp32-faithful
                                        conv, precision 0); 1 = the hi plane only (operand of a precision-1 conv)     */
} cpc_bn_params;

size_t cpc_bn_relu_workspace_bytes(const cpc_bn_params* p);
/* gamma / beta (C) may be NULL (affine=False).  running_mean / running_var (C): updated in place when
 * training (may be NULL then), read when not.  save_mean / save_rstd (C): outputs, inputs of bwd. */
int cpc_bn_relu_fwd(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var,
                    const float* residual, float* out, float* save_mean, float* save_rstd, const cpc_bn_params* p,
                    void* workspace, size_t workspace_bytes, void* stream);
/* dx overwritten; dgamma / dbeta (C) overwritten when non-NULL; d_residual (full residual shape, zero outside
 * the crop) overwritten when non-NULL. */
int cpc_bn_relu_bwd(const float* dout, const float* x, const float* gamma, const float* beta, const float* save_mean,
                    const float* save_rstd, const float* residual, float* dx, float* dgamma, float* dbeta,
                    float* d_residual, const cpc_bn_params* p, void* workspace, size_t workspace_bytes, void* stream);

/* Packed-output variants: when the only consumer of the activation (forward) or of the gradient (backward) is a
 * tensor-core conv that reads the bf16 hi/lo operand planes of cpc_conv_pack ([plane][B*C*H][round8(W)], fp32-faithful
 * mode), the batch norm writes that form directly -- no fp32 tensor, no packing pass.  cpc_bn_packed_bytes gives the
 * buffer size.  dx_sum (optional, C floats) receives the per-channel sum of dx = the bias gradient of the conv that
 * feeds this batch norm.  The conv entry points accept a NULL fp32 operand when its packed form is supplied and
 * cpc_conv_kernel_family is a row-streaming family (2, 3). */
size_t cpc_bn_packed_bytes(const cpc_bn_params* p);
int cpc_bn_relu_fwd_packed(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var,
                           const float* residual, void* packed_out, float* save_mean, float* save_rstd,
                           const cpc_bn_params* p, void* workspace, size_t workspace_bytes, void* stream);
int cpc_bn_relu_bwd_packed(const float* dout, const float* x, const float* gamma, const float* beta, const float* save_mean,
                           const float* save_rstd, const float* residual, void* packed_dx, float* dx_sum, float* dgamma,
                           float* dbeta, float* d_residual, const cpc_bn_params* p, void* workspace, size_t workspace_bytes,
                           void* stream);

/* Saved outer-ReLU mask: with a residual operand and outer_relu, the backward pass needs sign(v + residual).  The plain
 * entry points recompute it (re-reading the residual in both backward kernels); the *_mask variants exchange it as one
 * bit per element -- bit (i % 32) of word plane * ceil(H*W / 32) + i / 32, i the row-major index inside a (b, c) plane --
 * written by the forward call and read by the backward ones (residual itself is then not read).  cpc_bn_mask_bytes is
 * the buffer size, 0 when the shape has no such mask (no residual / no outer ReLU / planes served by the small-plane
 * kernels): pass NULL then, which makes every *_mask call identical to its plain counterpart. */
size_t cpc_bn_mask_bytes(const cpc_bn_params* p);
int cpc_bn_relu_fwd_mask(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var,
                         const float* residual, float* out, float* save_mean, float* save_rstd, void* relu_mask,
                         const cpc_bn_params* p, void* workspace, size_t workspace_bytes, void* stream);
int cpc_bn_relu_bwd_mask(const float* dout, const float* x, const float* gamma, const float* beta, const float* save_mean,
                         const float* save_rstd, const float* residual, const void* relu_mask, float* dx, float* dgamma,
                         float* dbeta, float* d_residual, const cpc_bn_params* p, void* workspace, size_t workspace_bytes,
                         void* stream);
int cpc_bn_relu_bwd_packed_mask(const float* dout, const float* x, const float* gamma, const float* beta,
                                const float* save_mean, const float* save_rstd, const float* residual,
                                const void* relu_mask, void* packed_dx, float* dx_sum, float* dgamma, float* dbeta,
                                float* d_residual, const cpc_bn_params* p, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ------------------------------------------------------------------------------------------------
 * 2c. Non-overlapping max pooling (kernel = stride, no padding), forward and backward.
 *    Replaces nn.MaxPool2d on the residual branch (scalogram_model.py:434-441, ceil_mode=True) and the main-path
 *    poolings (:402-403, :424-425) and max_pool2d_with_indices_backward.  x / dx (B, C, h_in, w_in),
 *    y / dy (B, C, h_out, w_out); h_out = ceil_mode ? ceil(h_in / kernel) : floor(h_in / kernel), same for w.
 *    The backward pass re-derives the arg-max from x (first maximum in row-major window order).
 * ---------------------------------------------------------------------------------------------- */
typedef struct cpc_pool_params {
    int32_t batch, channels, h_in, w_in, h_out, w_out;
    int32_t kernel;
    int32_t ceil_mode;
} cpc_pool_params;

int cpc_maxpool_fwd(const float* x, float* y, const cpc_pool_params* p, void* stream);
int cpc_maxpool_bwd(const float* x, const float* dy, float* dx, const cpc_pool_params* p, void* stream);
/* dx += max-pool gradient.  For a tensor that feeds both a pooling and another operator (the input of a residual
 * encoder block, scalogram_model.py:446-450): the other operator's backward writes dx, this call adds the pooling's share
 * in place -- what autograd's accumulation would do with a zero-filled pooling gradient and a separate add pass. */
int cpc_maxpool_bwd_accumulate(const float* x, const float* dy, float* dx, const cpc_pool_params* p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 3. InfoNCE scoring + loss, forward and backward, scores never written to HBM.
 *    Replaces score_function + the loss block of ContrastiveEstimationTrainer.train
 *    (contrastive_estimation_training.py:12-22, 106-122, 141, 166) and its autograd.
 *    pred (B, K, E) contiguous fp32; targets is the *strided view* z[:, :, -K:] of the encoder output
 *    (audio_model.py:197): element (t, e, k) at targets[t*tgt_stride_b + e*tgt_stride_e + k*tgt_stride_k].
 * ---------------------------------------------------------------------------------------------- */
typedef enum cpc_score_kind {
    CPC_SCORE_LINEAR = 0,
    CPC_SCORE_SOFTPLUS = 1,
    /* difference_score_function (contrastive_estimation_training.py): S = 1 / sum_e (P[r,e] - Z[c,e])^2.  Always on
     * the fp32 CUDA-core kernels (also with precision = bf16), with the squared differences accumulated in fp32, never
     * expanded as |p|^2 + |z|^2 - 2 p.z; a prediction equal to a target gives S = +inf and a NaN loss. */
    CPC_SCORE_DIFFERENCE = 2
} cpc_score_kind;

typedef struct cpc_infonce_params {
    int32_t batch;          /* B */
    int32_t steps;          /* K prediction steps */
    int32_t enc;            /* E encoding size */
    int32_t all_steps;      /* 1: softmax over all (d,k) for each (t,k') (score_over_all_timesteps=True);
                               0: per step k, softmax over d for each t                                 */
    int32_t score_kind;     /* cpc_score_kind */
    float regularization;   /* lambda of  lambda * mean((mean_k S)^2)  (:141) */
    int64_t tgt_stride_b, tgt_stride_e, tgt_stride_k;   /* in elements */
    int32_t precision;      /* as in cpc_conv_params */
    int32_t flags;          /* CPC_INFONCE_FLAG_*; 0 = default */
} cpc_infonce_params;
#define CPC_INFONCE_FLAG_NO_TENSOR 1     /* everything on the fp32 CUDA-core kernels                          */

/* Layout of the forward's `out` (fp32): [0] loss, [1] max score, [2] loss without regulariser,
 * [3] mean score; `lse`: per softmax column, all_steps ? (B*K) indexed t*K+k' : (K*B) indexed k*B+t.
 * `lse` is an output of fwd and an input of bwd (the saved-for-backward tensor). */
#define CPC_INFONCE_OUT_FLOATS 4
size_t cpc_infonce_workspace_bytes(const cpc_infonce_params* p, int which /* 0 fwd, 1 bwd */);
int cpc_infonce_fwd(const float* pred, const float* targets, float* out, float* lse,
                    const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, void* stream);
/* grad_loss: device pointer to one fp32 (dL/dloss).  d_pred (B,K,E) contiguous; d_targets (B,E,K)
 * contiguous; both overwritten. */
int cpc_infonce_bwd(const float* pred, const float* targets, const float* lse, const float* grad_loss,
                    float* d_pred, float* d_targets, const cpc_infonce_params* p,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Validation metrics of ContrastiveEstimationTrainer.validate (contrastive_estimation_training.py:224-247):
 * per-step losses (K) with the reference's view semantics, per-step accuracy (K), mean score (1).
 * metrics: (2*K + 1) fp32. */
int cpc_infonce_validate(const float* pred, const float* targets, float* metrics,
                         const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 5. Adam update of all parameter tensors (torch.optim.Adam semantics, amsgrad off) in one pass.
 *    Replaces optimizer.step() of ContrastiveEstimationTrainer.train
 *    (contrastive_estimation_training.py:162; optimizer class from the ctor, :41,59).
 *    params / grads / exp_avg / exp_avg_sq: HOST arrays of n_tensors device pointers (fp32, contiguous,
 *    numel[i] elements each).  step_state: 4 device floats owned by the caller; [0] is the step count t
 *    (0 before the first update; advanced by every call, so CUDA-graph replays keep counting), [1..2]
 *    are scratch (bias corrections of the current step).
 *      g = grad_scale * grad (+ weight_decay * p);  m += (1-beta1)(g-m);  v = beta2 v + (1-beta2) g^2
 *      p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps)
 * ---------------------------------------------------------------------------------------------- */
typedef struct cpc_adam_params {
    double lr, beta1, beta2, eps, weight_decay;   /* doubles, as the Python optimizer holds them: 1 - beta is
                                                     formed in double and rounded once, like torch does */
    float grad_scale;       /* 1/world_size when grads hold the all-reduced SUM, else 1 */
    int32_t maximize;
} cpc_adam_params;

int cpc_adam_step(int32_t n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                  void* const* exp_avg_sq, const int64_t* numel, float* step_state,
                  const cpc_adam_params* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CPC_B200_H */
