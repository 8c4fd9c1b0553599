/*
 * libb200np -- C ABI of the B200-native (sm_100a) neural-process hot path.
 *
 * The reference (boschresearch/what-matters-for-meta-learning) has no FFI: its hot path is Python
 * nn.Modules calling ATen/cuDNN/cuBLAS.  This header is the boundary a maintainer binds instead
 * (ctypes stub: what-matters-for-meta-learning_b200/b200np/lib.py; see INTEGRATION.md).  Each
 * entry point names the reference call site(s) it replaces.  File:line are relative to the
 * reference checkout.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous fp32 (or int32 where stated); the caller
 *     owns all memory, including workspaces (size them with the *_workspace functions);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous, never synchronise,
 *     never allocate, and are CUDA-graph capturable;
 *   - return value 0 = success, negative = B200NP_E_* (b200np_strerror gives the text);
 *   - CNN activations are NHWC ("pixel-major": [image][y][x][channel]); network inputs stay NCHW
 *     as the reference's datasets deliver them.
 */
#ifndef B200NP_H
#define B200NP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200NP_OK 0
#define B200NP_E_BADARG (-1)    /* dimension / pointer / alignment precondition violated */
#define B200NP_E_LAUNCH (-2)    /* cudaLaunch / cudaGetLastError reported a failure        */
#define B200NP_E_WORKSPACE (-3) /* workspace too small                                     */
#define B200NP_E_UNSUPPORTED (-4)

/* precision of tensor-core contractions: fp32-grade split (3 tf32 passes) or one tf32 pass,
 * or the CUDA-core fp32 kernels (used for validation and for shapes tensor cores do not fit) */
#define B200NP_PREC_FP32_SIMT 0
#define B200NP_PREC_TF32X3 1
#define B200NP_PREC_TF32 2

#define B200NP_ACT_NONE 0
#define B200NP_ACT_RELU 1
#define B200NP_ACT_TANH 2

const char* b200np_strerror(int code);
int b200np_version(void);
/* 1 if the current device is compute capability 10.x, 0 otherwise, negative on CUDA error */
int b200np_device_ok(void);
/* number of CUDA kernels this library has enqueued in this process (bench.py's gpu_launches) */
long long b200np_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Small-Cin direct convolution (stem).  Replaces nn.Conv2d 5x5 s2 p2 + ReLU at
 * networks/models.py:93-95,160-162 and the first conv of encoder_w0
 * (networks/CNPShapeNet1D.py:47-48).  x NCHW [N,Cin,H,W] (Cin<=4), w torch layout
 * [Cout,Cin,R,R], y NHWC [N,H/stride,W/stride,Cout].
 * ------------------------------------------------------------------------------------------ */
/* precision (B200NP_PREC_*): the 1-channel 5x5 stem runs on tcgen05 in the TF32 modes (im2col tile built
 * in shared memory, K = 25 padded to one 32-wide K-block); every other variant and fp32 mode run on
 * CUDA cores in exact fp32. */
/* relu_bits (nullable, tcgen05 stem only): the ReLU gates of y as 1 bit per element, [pixel][Cout/32] words,
 * bit j of word h = channel 32 h + j -- what b200np_conv_dgrad takes as `mask_bits` (8 B per pixel instead of
 * re-reading the 256 B activation). */
int b200np_conv_small_fwd(const float* x, const float* w, const float* bias, float* y, int N,
                          int Cin, int H, int W, int Cout, int R, int stride, int pad, int relu,
                          int precision, uint32_t* relu_bits, void* stream);
size_t b200np_conv_small_wgrad_workspace(int N, int Cin, int H, int W, int Cout, int R, int stride,
                                         int pad, int precision);
/* dy NHWC is the gradient w.r.t. the pre-activation output; writes dw [Cout,Cin,R,R], db [Cout] */
int b200np_conv_small_wgrad(const float* x, const float* dy, float* dw, float* db, int N, int Cin,
                            int H, int W, int Cout, int R, int stride, int pad, int precision,
                            void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Channel-dense NHWC convolutions as implicit GEMM (pixels x Cout x taps*Cin).
 * Replace the cuDNN calls behind BasicBlock.forward (networks/ResNet.py:58-74), the residual
 * 1x1 projection (:200-204), encoder_w0's 2nd/3rd convs (networks/CNPShapeNet1D.py:49-53) and
 * their autograd backward.
 *
 * Packed weights (made by b200np_pack_conv_weight from torch [Cout,Cin,R,R]) are opaque buffers of
 * b200np_packed_weight_floats(Cout,Cin,R) floats each:
 *   wf: [R*R][Cout][Cin] forward order,  wd: [R*R][Cin][Cout] data-gradient order,
 *   followed (64x64 layers) by the tensor-core image of the same slabs: tf32 hi/lo split,
 *   pre-swizzled 8 KB tiles that the tcgen05 kernels fetch with one bulk copy per K-block.
 * ------------------------------------------------------------------------------------------ */
size_t b200np_packed_weight_floats(int Cout, int Cin, int R);
int b200np_pack_conv_weight(const float* w, float* wf, float* wd, int Cout, int Cin, int R,
                            void* stream);

/* y = act( conv_RxR(x; wf, stride, pad=R/2) + bias  [+ conv_1x1(xs; wsf, stride_s) + bias_s] )
 * x  [N,H,W,Cin], y [N,H/stride,W/stride,Cout]; optional skip source xs [N,OH*stride_s,OW*stride_s,Cs]
 * (pass xs = NULL to disable).  This one call is conv1 (+ReLU) or conv2 + downsample + add + ReLU
 * of a BasicBlock. */
/* relu_bits (nullable; 64-channel tensor-core modes only): the gates (y > 0) of the output as 1 bit per element in
 * the format b200np_conv_dgrad takes as `mask_bits`. */
int b200np_conv_fwd(const float* x, const float* wf, const float* bias, float* y, int N, int H, int W,
                    int Cin, int Cout, int R, int stride, const float* xs, const float* wsf,
                    const float* bias_s, int Cs, int stride_s, int act, int precision, uint32_t* relu_bits, void* stream);

/* dx = relu_mask(act_saved) * ( dgrad_RxR(dy; wd, stride) [+ dgrad_1x1(dys; wsd, stride_s)] )
 * dy [N,H/stride,W/stride,Cout] -> dx [N,H,W,Cin]; `mask_src` (same shape as dx, may be NULL) is
 * the saved post-ReLU activation whose positivity gates the gradient; optional second gradient
 * source dys [N,H/stride_s,W/stride_s,Cs] through a 1x1 stride_s conv (the skip projection).
 * `mask_bits` (nullable, 64-channel dx only) is the same gate packed 1 bit per element (see
 * b200np_conv_small_fwd) and takes precedence over mask_src. */
int b200np_conv_dgrad(const float* dy, const float* wd, float* dx, const float* mask_src,
                      const uint32_t* mask_bits, int N, int H, int W, int Cin, int Cout, int R, int stride,
                      const float* dys, const float* wsd, int Cs, int stride_s, int precision, void* stream);

size_t b200np_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int R, int stride);
/* dw [Cout,Cin,R,R] (torch layout) = sum over pixels of dy (x) im2col(x);  db [Cout] = sum dy
 * (db may be NULL).  x [N,H,W,Cin], dy [N,H/stride,W/stride,Cout].
 * Optional fused skip projection (64x64 layers): xs [N,OH*stride_s,OW*stride_s,64] is the input of the
 * 1x1 stride_s conv that was added to this conv's output, dws [64,64] receives its weight gradient
 * (it sees the same dy); pass xs = dws = NULL to disable. */
int b200np_conv_wgrad(const float* x, const float* dy, float* dw, float* db, int N, int H, int W,
                      int Cin, int Cout, int R, int stride, const float* xs, float* dws, int stride_s,
                      int precision, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pooling / flatten at the end of the CNN (networks/models.py:105-113, networks/ResNet.py:151-152)
 * and encoder_w0's MaxPool2d(2,2) + nn.Flatten (networks/CNPShapeNet1D.py:51,54).
 * ------------------------------------------------------------------------------------------ */
/* AdaptiveMaxPool2d((2,2)) on NHWC [N,H,W,C] (H,W even) + NCHW-order flatten:
 * out[n, c*4 + oh*2 + ow]; idx (int32, same shape) = h*W + w of the FIRST maximum (torch rule) */
int b200np_adaptive_maxpool2x2_flatten_fwd(const float* x, float* out, int32_t* idx, int N, int H,
                                           int W, int C, void* stream);
/* dx [N,H,W,C] = relu_mask(x_saved) * scatter(dout by idx) (zero elsewhere) */
int b200np_adaptive_maxpool2x2_flatten_bwd(const float* dout, const int32_t* idx, const float* x_saved,
                                           float* dx, int N, int H, int W, int C, void* stream);
/* NHWC [N,H,W,C] <-> NCHW-order flatten [N, C*H*W]  (img_agg == "reshape"; nn.Flatten) */
int b200np_nhwc_to_nchw_flat(const float* x, float* out, int N, int H, int W, int C, void* stream);
/* dx = relu_mask(x_saved) * unflatten(dout); x_saved may be NULL (no mask) */
int b200np_nchw_flat_to_nhwc(const float* dout, const float* x_saved, float* dx, int N, int H, int W,
                             int C, void* stream);
/* MaxPool2d(2,2) NHWC [N,H,W,C] -> [N,H/2,W/2,C]; idx int8 in {0,1,2,3} (= dy*2+dx, first max) */
int b200np_maxpool2x2_fwd(const float* x, float* y, int8_t* idx, int N, int H, int W, int C,
                          void* stream);
/* dx [N,H,W,C] = relu_mask(x_saved) * scatter(dy by idx) */
int b200np_maxpool2x2_bwd(const float* dy, const int8_t* idx, const float* x_saved, float* dx, int N,
                          int H, int W, int C, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense layers.  Replace nn.Linear / torch.cat / ReLU / Tanh chains:
 * transform_y, task_encoder, mu, fc_mu (networks/CNPDistractor.py:43-57, models.py:139-145),
 * EncoderFC, r_to_z, decoder0 (models.py:27-60, CNPShapeNet1D.py:58-72), the per-head
 * AttnLinear projections and _W (ANPDistractor.py:83-100), FAVOR+ feature GEMMs.
 *
 * One strided, grouped GEMM covers all of them:
 *   for g in [0,groups):  C_g[m,n] = act( alpha * sum_k A_g(m,k) * B_g(k,n)
 *                                         + bias_g[n] + beta * C_g[m,n]
 *                                         + row_scale[m] * addend[m,n] )
 *   A_g(m,k) = A[g][m*a_rs + k*a_cs],  B_g(k,n) = B[g][k*b_rs + n*b_cs],  C row stride ldc.
 * One of (a_rs,a_cs) and one of (b_rs,b_cs) must be 1.  Pointer tables are HOST arrays of
 * `groups` device pointers (groups <= 8); bias / addend / row_scale may be NULL.
 * ------------------------------------------------------------------------------------------ */
typedef struct b200np_gemm_desc {
  const float* A[8];
  const float* B[8];
  float* C[8];
  const float* bias[8];
  int groups;
  int M, N, K;
  long long a_rs, a_cs, b_rs, b_cs, ldc;
  float alpha, beta;
  int act;
  const float* row_scale; /* [M] (group 0 only), with addend [M,N] row stride ld_add */
  const float* addend;
  long long ld_add;
  int precision;
  void* workspace;        /* optional split-K scratch (b200np_gemm_workspace bytes); NULL: single pass */
  size_t workspace_bytes;
  int sum_groups;         /* nonzero: the groups are concatenated along K into ONE product,
                             C_0 = act(alpha * sum_g sum_k A_g(m,k) B_g(k,n) + ...)  (K % 32 == 0) */
  /* Implicit 3x3 stride-2 pad-1 convolution (tensor-core modes, groups == 1): operand A (conv_operand = 1, a_cs == 1) or
   * B (conv_operand = 2, b_cs == 1) is not a matrix in memory but the VIRTUAL im2col matrix of the NHWC tensor
   * [n, conv_H, conv_W, conv_C] the pointer addresses: element (m, k) with m = (image, oy, ox) over conv_H/2 x conv_W/2
   * outputs and k = tap * conv_C + ci (TAP-major, tap = r*3 + s) is x[image, 2*oy + r - 1, 2*ox + s - 1, ci], zero outside
   * the image; conv_C % 4 == 0.  The row stride of that operand is ignored.  Forward: A virtual, B = tap-major weight
   * [Cout][9*Cin] (b200np_conv_weight_tapmajor); weight gradient: A = dY^T, B virtual.  No column matrix is written. */
  int conv_operand;
  int conv_H, conv_W, conv_C;
} b200np_gemm_desc;
/* bytes of scratch with which b200np_gemm spreads the K range of a GEMM with few output tiles over the idle
 * SMs (deterministic: partial tiles are reduced in a fixed order); 0 when the shape does not profit */
size_t b200np_gemm_workspace(const b200np_gemm_desc* d);
int b200np_gemm(const b200np_gemm_desc* d, void* stream);

/* dz = dy * act'(y)  (ReLU: y>0; Tanh: 1-y^2), elementwise over n floats; dz may alias dy */
int b200np_act_bwd(const float* dy, const float* y, float* dz, long long n, int act, void* stream);
/* out[c] = sum_r x[r*ld + c], r<rows, c<cols  (bias gradients); deterministic two-stage */
size_t b200np_colsum_workspace(long long rows, int cols);
int b200np_colsum(const float* x, float* out, long long rows, int cols, long long ld, void* ws,
                  size_t ws_bytes, void* stream);
/* utility elementwise ops used between kernels (no library calls on the hot path) */
int b200np_fill(float* x, long long n, float value, void* stream);
int b200np_axpy(float* y, const float* x, long long n, float a, void* stream); /* y += a*x */
/* dst[dst_off[i] .. +numel[i]) = src[i] (zeros where src[i] is NULL) for nseg segments: the per-parameter
 * gradients of one backward pass gathered into the flat gradient buffer with one launch per 64 segments
 * (replaces autograd's per-parameter accumulate kernels).  src / dst_off / numel are HOST arrays. */
int b200np_multi_copy(const float* const* src, const long long* dst_off, const long long* numel, int nseg,
                      float* dst, void* stream);

/* Device-side task assembly: out [M,C,H,W] fp32 = (255 - bank[rows[m]]) / 255 from a uint8 channel-last image bank
 * [n,H,W,C] resident in HBM (dataset/shapenet_distractor.py:233-234,256-259 + utils/utils.py:26-30: `255 - x`,
 * `astype(float32) / 255.0`, channel-last -> NCHW).  With the bank on the device a training step uploads the few KB
 * of row indices and labels instead of 47 MB of images.  H*W must be a multiple of 4. */
int b200np_gather_images_u8(const uint8_t* bank, const int32_t* rows, float* out, long long M, int H, int W,
                            int C, void* stream);
/* y[r, :] = x[r / rep, :] (rep consecutive copies of each row; the reference's .repeat) */
int b200np_repeat_rows(const float* x, float* y, long long rows_in, int rep, int cols, void* stream);
/* x[r,:] = sum over the rep copies of dy (backward of repeat_rows) */
int b200np_repeat_rows_bwd(const float* dy, float* dx, long long rows_in, int rep, int cols,
                           void* stream);
/* y = scale[0] * x  with the scalar read from device memory (no host sync) */
int b200np_scale_by_device_scalar(const float* x, const float* scale, float* y, long long n,
                                  void* stream);

/* ------------------------------------------------------------------------------------------
 * CNP context aggregation (networks/CNPDistractor.py:96-103, CNPShapeNet1D.py:115-120,
 * CondNeuralProcess.py:94-101): feats [T,nc,D] -> out [T,D].
 * mode 0 = mean, 1 = max (idx int32 [T,D] = FIRST maximal context index, bit-exact with
 * torch.max(dim=1)).
 * ------------------------------------------------------------------------------------------ */
int b200np_ctx_aggregate_fwd(const float* feats, float* out, int32_t* idx, int T, int nc, int D,
                             int mode, void* stream);
int b200np_ctx_aggregate_bwd(const float* dout, const int32_t* idx, float* dfeats, int T, int nc, int D,
                             int mode, void* stream);
/* Bayesian context aggregation "baco" (networks/CNPDistractor.py:60-75,104-110): mu, s [T,nc,D] (s = the
 * pre-softplus output of latent_var) -> r [T,D];  var = 1e-5 + softplus(s), prior N(0,1).  The backward
 * recomputes the sums from mu, s and r. */
int b200np_baco_fwd(const float* mu, const float* s, float* r, int T, int nc, int D, void* stream);
int b200np_baco_bwd(const float* dr, const float* mu, const float* s, const float* r, float* dmu, float* ds,
                    int T, int nc, int D, void* stream);

/* ------------------------------------------------------------------------------------------
 * FAVOR+ (Performer) attention exactly as networks/fast_attention.py:74-99,151-156 computes it
 * (math: SURVEY.md appendix A; constants c = d^-1/4, rho = M^-1/2, eps = 1e-4 derived inside).
 * Head-projected inputs are laid out [T, n, H, d]: row r = (t*n + i)*H + h.  The feature
 * pre-activations U = c*xq*P^T [T*nt*H, M] and W = c*xk*P^T [T*nc*H, M] come from b200np_gemm
 * (row stride ldu >= M).  The exp / eps / normalised product are fused into the attention
 * kernels; the reference's [T,H,M,d] "context" tensor (232 MB) is never built.
 * ------------------------------------------------------------------------------------------ */
/* per row of x [R,d] and U [R,ldu]: diag = c^2 |x|^2 / 2 (:86-89), rowmax = max_f U, argmax = first
 * maximal feature (:93).  For keys, b200np_reduce(rowmax, op=max) gives the global stabiliser (:97). */
int b200np_favor_rowstats(const float* x, const float* U, float* diag, float* rowmax, int32_t* argmax,
                          long long R, int d, int M, long long ldu, void* stream);
/* out[0] = max (op 0) or sum (op 1) of x[0..n) -- single block, deterministic */
int b200np_reduce(const float* x, long long n, float* out, int op, void* stream);
/* One CTA per (task, head).  A = Q'K'^T [T,H,nt,nc] and Dn = rowsum(A) [T,H,nt] are saved for the
 * backward; out [T,nt,d,H] (feature-major, head-minor: the order `_W` consumes,
 * networks/ANPDistractor.py:98-99).  g = device scalar holding the (all-reduced) key max.
 * ties (device float, accumulated) counts elements of W equal to g (torch.max() tie rule). */
/* nt * nc <= 1024 (the training and evaluation shapes reach 36 x 25 = 900); larger tiles return B200NP_E_UNSUPPORTED. */
int b200np_favor_attn_fwd(const float* U, const float* W, const float* sq, const float* mq,
                          const float* tk, const float* g, const float* v, float* out, float* A,
                          float* Dn, float* ties, int T, int H, int nt, int nc, int d, int M,
                          long long ldu, void* stream);
/* Gradients of the fused part.  dU [T*nt*H, ldu], dW [T*nc*H, ldu] are gradients w.r.t. the
 * pre-activations INCLUDING the row-argmax routing for queries; ds_c2 [Rq] = c^2 * ds and
 * dt_c2 [Rk] = c^2 * dt multiply xq / xk in the final GEMM epilogue; dg_part [T*H] = per-(task,head)
 * shares of d loss / d g (sum them with b200np_reduce, all-reduce across ranks, then fix up). */
int b200np_favor_attn_bwd(const float* d_out, const float* U, const float* W, const float* sq,
                          const float* mq, const int32_t* amq, const float* tk, const float* g,
                          const float* v, const float* out, const float* A, const float* Dn, float* dU,
                          float* dW, float* dv, float* ds_c2, float* dt_c2, float* dg_part, int T, int H,
                          int nt, int nc, int d, int M, long long ldu, void* stream);
/* dW[r,f] += dg[0] / ties[0] wherever W[r,f] == g[0]  (global-argmax routing, even tie split) */
int b200np_favor_key_fixup(float* dW, const float* W, const float* g, const float* dg, const float* ties,
                           long long R, int M, long long ldu, void* stream);

/* ------------------------------------------------------------------------------------------
 * Losses (trainer/losses.py:32-80).  mu [R,out], y [R,L]; loss (device scalar) = mean over R rows;
 * dmu [R,out] = d loss / d mu (may be NULL for evaluation).
 *   kind 0: distractor  mean ||y - mu||_2            (:35-36)
 *   kind 1: quaternion  mean min(|q-mu^|_1,|-q-mu^|_1), mu^ = mu/||mu||   (:50-57)
 *   kind 2: azimuth     mean sum (y[:2]-mu)^2        (:59-61)
 *   kind 3: degree error (evaluation only, no gradient)                  (:63-76)
 * ------------------------------------------------------------------------------------------ */
int b200np_loss_fwd_bwd(const float* mu, const float* y, float* loss, float* dmu, long long R, int out,
                        int L, int kind, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused Adam over a flat fp32 parameter segment (torch.optim.Adam semantics, train.py:52-56):
 * m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * `grad_scale` multiplies g first (1/world_size after a SUM all-reduce).
 * ------------------------------------------------------------------------------------------ */
int b200np_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                     float beta2, float eps, float weight_decay, int step, float grad_scale,
                     void* stream);
/* Same, with the step counter in device memory (*step_dev is incremented, then used): no host value
 * changes between steps, so a captured CUDA graph of the whole meta-train step can be replayed. */
int b200np_adam_step_dev(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                         float beta2, float eps, float weight_decay, int* step_dev, float grad_scale,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * MMAML conv nets (SURVEY.md 8f-3): GatedConvModel (networks/gated_conv_net.py:167-212: 3x3 stride-2 conv ->
 * batch-statistics BatchNorm, training=True always -> FiLM x*(1+gamma)+beta (:154-159) -> ReLU) and
 * ConvEmbeddingModel (networks/conv_embedding_model.py:99-184, affine BatchNorm), any channel count.
 *
 * The convolution is im2col + b200np_gemm: col[m][ci*9 + r*3 + s] = x[n, 2oy+r-1, 2ox+s-1, ci] uses the flattening
 * of torch's [Cout, Cin, 3, 3] weight, so forward (col x W^T), weight gradient (dY^T x col) and data gradient
 * (dY x W, then col2im) read the parameter tensor as it is.  x NHWC [N,H,W,C], H and W even.
 * col2im gathers (deterministic); `mask` (nullable, dx geometry) gates the result with (mask > 0).
 *
 * bn_act: per channel over all `rows` = N*H*W rows of x [rows, C]: mean, biased variance (fp64 sums, two-level,
 * deterministic), y = relu?((x - mean) * rstd * (scale + plus_one) + shift); scale / shift nullable ([C]).  FiLM passes
 * scale = gamma, plus_one = 1, shift = beta; affine BatchNorm scale = weight, plus_one = 0, shift = bias.  mean / rstd
 * are saved for the backward; run_mean / run_var (nullable) get F.batch_norm's running update (unbiased variance).
 * The statistics are accumulated in fp64 and `mean` is an array of 2*C floats: mean[c] + mean[C + c] is the batch mean
 * as a (hi, lo) pair, and every kernel forms x - mean as (x - hi) - lo, so that the sign of a pre-activation near zero
 * -- the ReLU gate, which the backward and the second-order backward multiply by -- does not depend on the rounding of
 * the mean when |mean| >> std.
 * Backward: dshift = sum g, dscale = sum g * xhat (g = dy gated by y > 0 when relu), dx = the usual batch-norm data
 * gradient.  Workspace: b200np_bn_workspace(rows, C) bytes.
 * ------------------------------------------------------------------------------------------ */
/* im2col of an NCHW image with few channels for an R x R stride-2 convolution (the stems `nn.Conv2d(C,64,5,2,2)`,
 * networks/ResNet.py; `encoder_w0[0]`, CNPShapeNet1D.py:47): col [N*(H/2)*(W/2), ld], col[m][ci*R*R + r*R + s], columns
 * beyond Cin*R*R zero.  With b200np_gemm (forward: col x W^T + bias, ReLU; weight gradient: dY^T x col) it replaces the
 * CUDA-core direct convolution where the tcgen05 stem kernel (1 channel, 5x5, 64 outputs) does not apply. */
int b200np_im2col_small(const float* x, float* col, int N, int Cin, int H, int W, int R, int pad, int ld, void* stream);
/* tap-major <-> torch layout of a 3x3 conv weight: wt[co][tap*Cin + ci] = w[co][ci][tap] (to_tapmajor != 0) or the inverse */
int b200np_conv_weight_tapmajor(const float* src, float* dst, int Cout, int Cin, int to_tapmajor, void* stream);
/* col2im of a TAP-major column-gradient matrix [N*(H/2)*(W/2), 9*C] (k = tap*C + ci), C % 4 == 0: 16-byte gathers */
int b200np_col2im3x3s2_tapmajor(const float* dcol, const float* mask, float* dx, int N, int H, int W, int C, void* stream);
int b200np_im2col3x3s2(const float* x, float* col, int N, int H, int W, int C, void* stream);
int b200np_col2im3x3s2(const float* dcol, const float* mask, float* dx, int N, int H, int W, int C, void* stream);
size_t b200np_bn_workspace(long long rows, int C);
int b200np_bn_act_fwd(const float* x, const float* scale, const float* shift, float plus_one, float eps, float* y,
                      float* mean, float* rstd, float* run_mean, float* run_var, float momentum, long long rows, int C,
                      int relu, void* ws, size_t ws_bytes, void* stream);
int b200np_bn_act_bwd(const float* dy, const float* y, const float* x, const float* mean, const float* rstd,
                      const float* scale, float plus_one, float* dx, float* dscale, float* dshift, long long rows, int C,
                      int relu, void* ws, size_t ws_bytes, void* stream);
/* Second order (the reference's MMAML trainer differentiates through the inner-loop gradient,
 * trainer/meta_learner_reg.py:116-130, train.py:99 first_order=False): gradients of
 * <vx, dx> + <vs, dscale> + <vt, dshift> -- the three outputs of b200np_bn_act_bwd -- with respect to x (gx), dy (gdy)
 * and scale (gscale); vx / vs / vt and the outputs are nullable.  Workspace: b200np_bn_workspace2(rows, C). */
size_t b200np_bn_workspace2(long long rows, int C);
int b200np_bn_act_bwd2(const float* dy, const float* y, const float* x, const float* mean, const float* rstd,
                       const float* scale, float plus_one, const float* vx, const float* vs, const float* vt, float* gx,
                       float* gdy, float* gscale, long long rows, int C, int relu, void* ws, size_t ws_bytes,
                       void* stream);
/* out = alpha * a * b * c, elementwise (b, c nullable): second-order products (tanh, MSE loss) */
int b200np_mul3(const float* a, const float* b, const float* c, float alpha, float* out, long long n, void* stream);

/* ------------------------------------------------------------------------------------------
 * Bayes-by-backprop weight sampling + KL (SURVEY.md 8f-4; networks/bbb/BBBConv.py:83-105, BBBLinear.py):
 *   sigma = log1p(exp(rho)), w = mu + eps * sigma, kl = calculate_kl(prior_mu, prior_sigma, mu, sigma) (:32-34,:102-105)
 * eps [n] is drawn by the caller (the reference draws it on the host, :86).  kl_part receives b200np_bbb_kl_blocks(n)
 * partial sums (sum them in order with b200np_reduce: deterministic).  Backward: dw [n] (nullable) and the device
 * scalar dkl (nullable) -> dmu, drho.
 * ------------------------------------------------------------------------------------------ */
int b200np_bbb_kl_blocks(long long n);
int b200np_bbb_sample_kl_fwd(const float* mu, const float* rho, const float* eps, float prior_mu, float prior_sigma,
                             float* w, float* sigma, float* kl_part, long long n, void* stream);
int b200np_bbb_sample_kl_bwd(const float* dw, const float* dkl, const float* mu, const float* rho, const float* eps,
                             const float* sigma, float prior_mu, float prior_sigma, float* dmu, float* drho,
                             long long n, void* stream);

/* ------------------------------------------------------------------------------------------
 * Diagnostics (tools/ only; never called on the product path).  They switch global state of the
 * library and are NOT thread-safe.
 *   b200np_debug_set_wgrad_waves   pixel chunks per weight-gradient launch = waves * resident CTAs
 * ------------------------------------------------------------------------------------------ */
void b200np_debug_set_wgrad_waves(int waves);

/* ------------------------------------------------------------------------------------------
 * Multi-GPU.  SURVEY.md 8b sketched `b200np_comm_{init,allreduce_sum,allreduce_max,destroy}` wrappers over
 * NCCL.  They are deliberately NOT part of this ABI: the host side is Python/PyTorch (north_star), which already
 * owns the NCCL communicator (`torch.distributed`, backend "nccl", one process per GPU); the three exchanges of
 * the path -- the SUM all-reduce of the flat gradient and the FAVOR+ key-stabiliser MAX / its gradient SUM -- are
 * issued on that communicator from b200np/dist.py on the same stream as the kernels and are captured into the
 * step's CUDA graph with them.  A second communicator inside this library would duplicate NCCL's bootstrap for
 * no data-path benefit.
 * ------------------------------------------------------------------------------------------ */

#ifdef __cplusplus
}
#endif
#endif /* B200NP_H */
