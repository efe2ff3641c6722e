/*
 * libdeltakd_sm100 — C ABI of the B200-native DeltaKD distillation-loss hot path.
 *
 * The reference (serizard/DeltaKD) has no FFI: its boundary is the Python callable
 * `DistillationLoss.forward` (model/loss.py:29-242, called at tools/engine.py:48).  Each entry
 * point below replaces the eager ATen op chain of one piece of that callable; the reference
 * lines are cited per function.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (inputs const, outputs written, never
 *    retained past return); the library never allocates or frees;
 *  - all work is enqueued on `stream`; no host synchronisation, no device->host read-backs;
 *  - return value: DKD_OK or a negative DKD_E_* code; dkd_last_error() gives the message of the
 *    last failure on the calling thread; no C++ exception crosses the ABI;
 *  - `dtype` is the storage type of activations (DKD_F32 / DKD_BF16); accumulation is fp32;
 *  - scalars losses are fp32 on the device;
 *  - there is no CPU path: on a device that is not sm_100 every compute call returns DKD_E_ARCH.
 */
#ifndef DELTAKD_H_
#define DELTAKD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DKD_API __attribute__((visibility("default")))
#else
#define DKD_API
#endif

typedef struct CUstream_st* dkd_stream_t; /* == cudaStream_t */

enum { DKD_F32 = 0, DKD_BF16 = 1 };

enum {
  DKD_OK = 0,
  DKD_E_SHAPE = -1,
  DKD_E_DTYPE = -2,
  DKD_E_ALIGN = -3,
  DKD_E_ARCH = -4,
  DKD_E_LAUNCH = -5,
  DKD_E_WORKSPACE = -6,
  DKD_E_UNSUPPORTED = -7
};

/* tensor-core arithmetic of the dense contractions */
enum {
  DKD_PREC_BF16 = 0,  /* one bf16 tcgen05 pass, fp32 accumulate                                  */
  DKD_PREC_BF16X3 = 1, /* hi/lo bf16 split, 3 passes (hi*hi + hi*lo + lo*hi): ~2^-16 relative,  */
                       /* the mode that meets the fp32 parity gates                             */
  /* OR'ed into `precision` of the gradient-bearing feature entry points (align_mse, align_nmse, wass_l1,
   * wass_sinkhorn, masked_generation, lrkd: *_workspace_bytes, *_fwdbwd, and dkd_masked_generation_hidden_offset):
   * every gradient is bit-reproducible.  Split-K weight gradients and column sums store one fp32 partial per split
   * (per CTA) into the workspace and a fold kernel adds them in split order in fp64; split counts and grids depend on
   * the shapes only.  The workspace grows by those partial regions (appended after the others). */
  DKD_PREC_DETERMINISTIC = 0x100
};

DKD_API int dkd_version(void);
DKD_API const char* dkd_last_error(void);
/* DKD_OK when the current CUDA device is compute capability 10.x, else DKD_E_ARCH. */
DKD_API int dkd_check_device(void);
/* Number of CUDA kernels this library has enqueued since it was loaded (statistics for bench.py's
 * `gpu_launches`; under CUDA-graph capture it counts the captured launches once). */
DKD_API unsigned long long dkd_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Logit losses: base CE + soft / hard KD, forward and backward in one launch.
 * Replaces model/loss.py:35 (base criterion: timm SoftTargetCrossEntropy or
 * LabelSmoothingCrossEntropy, loss.py:244-249), :57-64 (soft KD), :66-67 (hard KD) and the mix
 * `base*(1-alpha) + kd*alpha` at :241, plus their autograd backward.
 *
 *   outputs, outputs_kd, teacher_logits : [B, C] `dtype`, row-major contiguous
 *                                         (outputs_kd / teacher_logits may be NULL when kd_kind==0)
 *   labels      : label_kind 0 -> soft targets [B, C] `dtype`; 1 -> int64 class ids [B];
 *                 -1 -> no base term (outputs/labels/g_outputs ignored; total = alpha * kd)
 *   mix_lam     : NULL, or (label_kind 1 only) a DEVICE fp32 scalar lam: the target of row r is then the Mixup / CutMix
 *                 soft label timm's Mixup would have built (tools/train.py:288-295, engine.py:16-18: mixup_target)
 *                     lam * smooth_onehot(labels[r]) + (1 - lam) * smooth_onehot(labels[B-1-r]),
 *                 smooth_onehot(k)[c] = smoothing/C + (1 - smoothing) * [c == k], generated inside the kernel: the
 *                 [B, C] soft-label tensor is neither written by the mixer nor read by the loss
 *   kd_kind     : 0 none (loss = base), 1 soft (temperature `tau`), 2 hard (teacher argmax, first max)
 *   g_outputs, g_outputs_kd : [B, C] `dtype` gradients of the returned loss (NULL -> not written)
 *   loss_out    : fp32[3] = { total, base, kd }
 *   workspace   : >= dkd_logit_kd_workspace_bytes(B) bytes, ZERO-INITIALISED ONCE by the caller
 *                 (holds per-row partials and a ticket counter that the kernel resets itself)
 */
DKD_API size_t dkd_logit_kd_workspace_bytes(int64_t B);
DKD_API int dkd_logit_kd_fwdbwd(const void* outputs, const void* outputs_kd, const void* teacher_logits,
                        const void* labels, int label_kind, int kd_kind, int64_t B, int64_t C, int dtype,
                        float smoothing, float alpha, float tau, const float* mix_lam, void* g_outputs,
                        void* g_outputs_kd, float* loss_out, void* workspace, size_t workspace_bytes,
                        dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Mask selection by rank (bit-exact integer work).  Replaces the double argsort of
 * model/misc.py:17-30 (random_masking) and :72-81, :118-128, :150-160 (saliency_masking):
 *   ids_restore[b,i] = rank of score[b,i] in ascending order, ties -> lower index first
 *   ids_shuffle[b,r] = index of the token with rank r            (NULL -> not written)
 *   mask[b,i]        = 1.0f if ids_restore[b,i] >= len_keep else 0.0f
 *   score : fp32 [B, L], L <= 1024.
 */
DKD_API int dkd_mask_rank(const float* score, int64_t B, int64_t L, int64_t len_keep, float* mask,
                  int64_t* ids_restore, int64_t* ids_shuffle, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * x[i] *= *scale for i < n (and x2[i] for i < n2; pass NULL/0 for one tensor), skipped entirely
 * (no memory traffic) when *scale == 1.0f.
 * Used by the autograd backward of the fused fwd+bwd losses: gradients are produced for
 * d(loss)=1 in the forward sweep and only rescaled when the incoming grad_output is not 1
 * (e.g. under an AMP GradScaler, tools/engine.py:60).  `scale` is a device fp32 scalar.
 */
DKD_API int dkd_scale_if_not_one(void* x, int64_t n, void* x2, int64_t n2, int dtype, const float* scale,
                                 dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Layer-wise hidden-state matching with a linear alignment head, forward + backward:
 *     y = s[:, s_off:s_off+n_tok, :] W^T + bias ;  d = y - t[:, t_off:t_off+n_tok, :]
 *     *loss += scale * sum(d^2)                      (accumulates: zero *loss before the first layer)
 *     g_s = 2*scale * d W  (written into [B,Ts,Ds]; the s_off special-token rows are zeroed)
 *     g_W = 2*scale * d^T s,   g_b = 2*scale * sum_rows d          (overwritten)
 * Replaces, per selected layer, `mse_loss(Linear(student[:,1:]), teacher[:,2:], reduction='sum')` and its
 * backward in curkd_loss early/mid (model/loss.py:376-393; scale = 4e-5/(nL*B)) and the ViTKD
 * mimicking term (loss.py:277-289; scale = alpha_vitkd/B).
 *   s [B,Ts,Ds], t [B,Tt,Dt] : `dtype`, contiguous, special tokens included (consumed in place)
 *   W [Dt,Ds], bias [Dt], g_W, g_b, loss : fp32 ;  g_s : `dtype`  (any g_* may be NULL)
 *   precision : DKD_PREC_BF16 | DKD_PREC_BF16X3 (tcgen05 bf16 passes, fp32 accumulate in TMEM), optionally
 *               | DKD_PREC_DETERMINISTIC (bit-reproducible g_W / g_b; pass the same value to the workspace query)
 *   workspace : >= dkd_align_mse_workspace_bytes(...) bytes, 1024-byte aligned, contents don't matter
 * Built for Ds = 192 with Dt = 384 (DeiT-Tiny -> DeiT-Small) or Dt = 768 (DeiT-Tiny -> DeiT-Base); any other pair
 * returns DKD_E_SHAPE.
 */
DKD_API size_t dkd_align_mse_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision);
DKD_API int dkd_align_mse_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts,
                                 int s_off, int Tt, int t_off, int n_tok, int Ds, int Dt, int dtype, int precision,
                                 float scale, void* g_s, float* g_W, float* g_b, float* loss, void* workspace,
                                 size_t workspace_bytes, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Normalised hidden-state matching (feature term of DiffKD), forward + backward:
 *     a = s[:, s_off:, :] W^T + bias ;  a_hat = a/|a|, t_hat = t[:, t_off:, :]/|t| (L2 over channels, per token)
 *     *loss += scale * sum (a_hat - t_hat)^2     (accumulates);  g_s, g_W, g_b as in dkd_align_mse_fwdbwd
 * Replaces, per layer of the diffkd branch (model/loss.py:112-116, 139-140, 149), the alignment Linear, the two
 * per-token L2 normalisations and `F.mse_loss(s_feat, t_feat)` with their backward; the caller folds 1/numel into
 * `scale` and applies the data-dependent weight w_t.mean() (a device scalar) through the autograd rescale.
 * Same argument conventions as dkd_align_mse_fwdbwd, but built for Ds = 192, Dt = 384 only.  The noise-prediction term of that branch
 * (`student.denoise_fn`, an nn.Module with Dropout) stays a module call.
 */
DKD_API size_t dkd_align_nmse_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision);
DKD_API int dkd_align_nmse_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts,
                                  int s_off, int Tt, int t_off, int n_tok, int Ds, int Dt, int dtype, int precision,
                                  float scale, void* g_s, float* g_W, float* g_b, float* loss, void* workspace,
                                  size_t workspace_bytes, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * WassKD 'l1' term of one layer, forward + backward:
 *     a = s[:, s_off:, :] W^T + bias ;  per (sample, channel): sort the n_tok values of a and of t[:, t_off:, :]
 *     *loss += scale * sum |sort(a) - sort(t)|                (accumulates)
 *     g_a[b, pi(r), d] = scale * sign(sorted_a - sorted_t)[b, r, d]  -> g_s, g_W, g_b   (overwritten)
 * Replaces model/loss.py:187-199 (torch.sort over dim=1 of both tensors, mean |diff|) and its backward;
 * the caller folds 5/(3*B*n_tok*Dt) into `scale`.  Same argument conventions as dkd_align_mse_fwdbwd;
 * n_tok <= 256.  Ties in the student sort are ordered by token index.
 * Built for Ds = 192 with Dt = 384 (DeiT-Tiny -> DeiT-Small) or Dt = 768 (DeiT-Tiny -> DeiT-Base); any other pair
 * returns DKD_E_SHAPE.
 */
DKD_API size_t dkd_wass_l1_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision);
DKD_API int dkd_wass_l1_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts, int s_off,
                               int Tt, int t_off, int n_tok, int Ds, int Dt, int dtype, int precision, float scale,
                               void* g_s, float* g_W, float* g_b, float* loss, void* workspace, size_t workspace_bytes,
                               dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * WassKD 'sinkhorn' term of one layer, forward + backward:
 *     a = s[:, s_off:, :] W^T + bias ;  per sample b: S_b = debiased Sinkhorn divergence (p = 2, blur = 0.05,
 *     scaling = 0.5, uniform weights) between the n_tok points a[b] and t[b, t_off:, :] in R^Dt
 *     *loss += scale * sum_b S_b        (accumulates);   g_a = scale * dS_b/da -> g_s, g_W, g_b   (overwritten)
 * Replaces the per-sample Python loop over geomloss.SamplesLoss("sinkhorn", blur=0.05) of model/loss.py:200-225
 * (one host read-back of the diameter and ~60 logsumexp launches per sample there) and its backward; the caller
 * folds 5/(3*B*n_tok) into `scale`.  geomloss is absent and unpinned in the reference: the arithmetic follows
 * upstream geomloss 0.2.x (tensorized sinkhorn_loop with symmetric updates, eps ladder from the bounding-box
 * diameter, last extrapolation step differentiated through the cost matrices only) — oracle/sinkhorn.py.
 * The eps ladder is built on the device (no synchronisation).  Same argument conventions as
 * dkd_align_mse_fwdbwd; n_tok must be 196, Ds = 192, Dt = 384.  The cost matrices always use fp32-exact
 * split operands (6 bf16 products), the plan contraction bf16x3; `precision` applies to the alignment head.
 */
DKD_API size_t dkd_wass_sinkhorn_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision);
DKD_API int dkd_wass_sinkhorn_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts,
                                     int s_off, int Tt, int t_off, int n_tok, int Ds, int Dt, int dtype, int precision,
                                     float scale, void* g_s, float* g_W, float* g_b, float* loss, void* workspace,
                                     size_t workspace_bytes, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Masked generative distillation core, forward + backward (Ds = 192, Dt = 384) on a square patch grid of
 * n_tok = Ts - s_off = Tt - t_off tokens: 196 (14x14, 224-px inputs, patch 16) or 576 (24x24, 384-px inputs); any
 * other count returns DKD_E_SHAPE:
 *     x   = s[:, s_off:, :] W_align^T + b_align
 *     x_m = where(mask, mask_token, x)
 *     g   = conv3x3(relu(conv3x3(x_m; conv1)); conv2)          (pad 1, NHWC = the token layout)
 *     *loss += scale * sum( mask * (g - t[:, t_off:, :])^2 )   (accumulates)
 * plus the gradients of every input that has a non-NULL g_* pointer (all overwritten).
 * Replaces mgd_loss (model/loss.py:422-451; scale = mgd_alpha/(B*n_tok*Dt)), saliency_mgd_loss (:335-360;
 * scale = 4/(B*n_tok*Dt)), the late phase of curkd_loss (:394-420; scale = 5e-5/B) and the ViTKD
 * generation term (:291-310), including `student.generation` = Conv2d-ReLU-Conv2d (models.py:148-151).
 *   mask : fp32 [B, n_tok], 1 = masked (from dkd_mask_rank) ;  mask_token : fp32 [Dt]
 *   conv*_w : fp32 [Dt, Dt, 3, 3] (PyTorch layout), conv*_b : fp32 [Dt]
 */
DKD_API size_t dkd_masked_generation_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision);
/* Byte offset, inside the workspace, of the generator's hidden activations h = relu(conv1(x_m)) as bf16 planes
 * [P][B*n_tok][Dt] (P = 2 hi/lo planes for DKD_PREC_BF16X3, else 1; DKD_PREC_DETERMINISTIC does not move them).  They
 * stay valid after dkd_masked_generation_fwdbwd
 * returns: verification code reads the ReLU gate the backward pass used from them (h != 0), because the gradient of
 * F.relu (models.py:150) is discontinuous at 0 and parity of the gradients is only defined given the same gate. */
DKD_API size_t dkd_masked_generation_hidden_offset(int64_t B, int n_tok, int Ds, int Dt, int precision);
DKD_API int dkd_masked_generation_fwdbwd(const void* s, const void* t, const float* mask, const float* W_align,
                                         const float* b_align, const float* mask_token, const float* conv1_w,
                                         const float* conv1_b, const float* conv2_w, const float* conv2_b, int64_t B,
                                         int Ts, int s_off, int Tt, int t_off, int Ds, int Dt, int dtype, int precision,
                                         float scale, void* g_s, float* g_W_align, float* g_b_align, float* g_mask_token,
                                         float* g_conv1_w, float* g_conv1_b, float* g_conv2_w, float* g_conv2_b,
                                         float* loss, void* workspace, size_t workspace_bytes, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Saliency scores for saliency-MGD (no gradient).  Replace SimpleAttention / SimpleCrossAttention
 * (model/models.py:14-56) as used by saliency_masking (model/misc.py:62-70, 88-116, 135-148); the
 * ascending order of the score picks the kept tokens (dkd_mask_rank).  8 heads x 48 (D = 384).
 *
 * dkd_saliency_selfdiag_score — method 1: score[b,i] = mean_h softmax_j(q_i.k_j / sqrt(48))[i] over the n_tok
 *   patch tokens x[b, off + i, :] of x [B, T, D] (`dtype`); qk_w [2D, D], qk_b [2D] fp32 (q = first D outputs).
 *   Built for n_tok = 196.  Both contractions run on tcgen05: the qk projection (`precision`) writes q (pre-scaled) and
 *   k as bf16 planes, and one 128 x 208 x 48 GEMM per (sample, head, query half) forms the logits in tensor memory,
 *   where the epilogue reduces each row to its softmax diagonal — the attention maps are never materialised.
 * dkd_saliency_cls_score — methods 2 and 3: one query token per sample (xq + b*xq_stride, strides in elements)
 *   against n_keys key tokens (xk + b*xk_stride + j*D); separate q / k projections Wq,bq / Wk,bk ([D,D],[D], fp32;
 *   biases may be NULL).  query_is_key != 0 also counts the query token as key 0 of the softmax and drops its
 *   column from the output (method 2: CLS row over [CLS]+patches).  score: fp32 [B, n_keys].
 */
DKD_API size_t dkd_saliency_selfdiag_workspace_bytes(int64_t B, int n_tok, int D, int precision);
DKD_API int dkd_saliency_selfdiag_score(const void* x, int64_t B, int T, int off, int n_tok, int D, int dtype,
                                        const float* qk_w, const float* qk_b, int num_heads, int precision, float* score,
                                        void* workspace, size_t workspace_bytes, dkd_stream_t stream);
DKD_API int dkd_saliency_cls_score(const void* xq, int64_t xq_stride, const void* xk, int64_t xk_stride, int n_keys,
                                   int64_t B, int D, int dtype, const float* Wq, const float* bq, const float* Wk,
                                   const float* bk, int num_heads, int query_is_key, float* score, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LRKD low-rank projection matching, all selected layers, forward + backward:
 *     T_l = t[l][:, t_off:, :].reshape(M, Dt) ;  V_k = top-`rank` right singular vectors of T_l ;  A = T_l V_k
 *     s'  = s[l][:, s_off:, :] W[l]^T + bias[l]            (W[l] : [rank, Ds])
 *     *loss += coef[l] / (M * rank) * sum((A - s')^2)      (accumulates; coef is a HOST array)
 * plus g_s[l], g_W[l], g_b[l] (overwritten; any may be NULL).  Replaces model/loss.py:80-103 and lrkd_loss
 * (:314-330): `U,S,_ = torch.linalg.svd(T); A = U[:, :k] diag(S[:k])` (= T V_k), `MSELoss(mean)` against the projected
 * student, weighted by lrkd_alpha/beta/gamma, and their backward.  The tall SVD is replaced by the fp64 Jacobi
 * eigen-decomposition of the Dt x Dt Gram matrix T^T T (tcgen05, fp32-exact split operands, fp64 reduction).
 * The sign of each singular vector is arbitrary in any SVD; here the largest-magnitude component of every v is
 * positive.  Vk_out[l] (fp32 [rank, Dt]) and S_out[l] (fp32 [rank], singular values) are optional outputs for
 * sign alignment and inspection; sweeps_out (int[n_layers], device) receives the Jacobi sweep counts.
 * s, t, W, bias, g_*, Vk_out, S_out are HOST arrays of n_layers device pointers (n_layers <= 8).
 * Built for Ds = 192, Dt = 384, rank <= 128.  The eigensolver (dkd_lrkd_eigensolve below) is one launch of n_layers
 * 16-CTA thread-block clusters; where such a cluster cannot be scheduled it falls back to one cooperative launch
 * (24*n_layers co-resident CTAs when that fits 148 SMs, else 12*n_layers).
 */
DKD_API size_t dkd_lrkd_workspace_bytes(int n_layers, int64_t B, int n_tok, int Ds, int Dt, int rank, int dtype,
                                        int precision);
DKD_API int dkd_lrkd_fwdbwd(int n_layers, const void* const* s, const void* const* t, const float* const* W,
                            const float* const* bias, const float* coef, int64_t B, int Ts, int s_off, int Tt, int t_off,
                            int n_tok, int Ds, int Dt, int rank, int dtype, int precision, void* const* g_s,
                            float* const* g_W, float* const* g_b, float* loss, float* const* Vk_out, float* const* S_out,
                            int* sweeps_out, void* workspace, size_t workspace_bytes, dkd_stream_t stream);

/* The eigensolver of dkd_lrkd_fwdbwd on its own (tests, and the eigensolve time bench.py reports beside the roofline):
 * W [n_layers][384][384] fp64, symmetric positive semi-definite, device memory; overwritten with the columns
 * lambda_j v_j of its eigen-decomposition in an unspecified column order (column norms = eigenvalues).  One-sided fp64
 * Jacobi; sweeps_out [n_layers] device ints or NULL.  k = number of leading eigenpairs the caller will read (1..384):
 * the cluster-resident version stops when the k columns of largest norm are orthogonal to every other column (all
 * columns are rotated in every sweep, but the trailing ones converge last and may be left unconverged); k = 384 asks
 * for the full decomposition.  algo: 0 = what dkd_lrkd_fwdbwd uses (cluster-resident: one
 * 16-CTA thread-block cluster per matrix, columns exchanged through distributed shared memory; falls back to the
 * cooperative-launch version when such a cluster cannot be scheduled), 1 = cluster-resident or DKD_E_LAUNCH,
 * 2 = cooperative launch.  Replaces the torch.linalg.svd of model/loss.py:318-324 (V of T = U S V^T). */
DKD_API size_t dkd_lrkd_eigensolve_workspace_bytes(void);
DKD_API int dkd_lrkd_eigensolve(double* W, int n_layers, int k, int* sweeps_out, int algo, void* workspace,
                                size_t workspace_bytes, dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Row operations of the token streams that feed the loss path (SURVEY 8f rank 1: the callers of the path).
 * The reference builds student and teacher with timm 0.9.12 (model/models.py:59-74): every block is
 * x + attn(LayerNorm(x)), x + mlp(LayerNorm(x)) with nn.LayerNorm(eps=1e-6); these replace ATen's
 * native_layer_norm / native_layer_norm_backward and the bias-gradient `sum(0)` of nn.Linear on [B*197, D] streams.
 *
 *   dkd_layernorm_fwd : y[m,:] = (x[m,:] - mean_m) * rstd_m * gamma + beta,  rstd = 1/sqrt(var + eps) (biased var);
 *                       x [M, D] x_dtype, gamma / beta [D] p_dtype (beta may be NULL), y [M, D] y_dtype,
 *                       mean / rstd fp32 [M] (both NULL for inference).  D % 4 == 0, D <= 1024.
 *   dkd_layernorm_bwd : dx (x_dtype, may be NULL), dgamma, dbeta (fp32 [D], may be NULL) from dy (dy_dtype), x, gamma,
 *                       mean, rstd; overwrites.  D % 4 == 0, D <= 512.  Deterministic (fixed-order column folds).
 *   dkd_colsum        : out[n] = sum_m a[m, n], a [M, N] dtype, out fp32 [N].  N % 8 == 0, N <= 2048.  Deterministic.
 */
DKD_API int dkd_layernorm_fwd(const void* x, const void* gamma, const void* beta, int64_t M, int D, int x_dtype, int p_dtype,
                              int y_dtype, float eps, void* y, float* mean, float* rstd, dkd_stream_t stream);
DKD_API size_t dkd_layernorm_bwd_workspace_bytes(int64_t M, int D);
DKD_API int dkd_layernorm_bwd(const void* dy, const void* x, const void* gamma, const float* mean, const float* rstd, int64_t M,
                              int D, int dy_dtype, int x_dtype, int p_dtype, void* dx, float* dgamma, float* dbeta,
                              void* workspace, size_t workspace_bytes, dkd_stream_t stream);
/*   dkd_head_copy     : dst[b,h,n,0:hd] = src[b,h,n,0:hd] with independent (b,h,n) ELEMENT strides per side, hd contiguous
 *                       (hd * elt_bytes and all strides multiples of 16 bytes): the [B,H,N,hd] <-> [B,N,H,hd] relayouts
 *                       around scaled-dot-product attention (head merge, packed-qkv gradient assembly).
 */
DKD_API int dkd_head_copy(const void* src, void* dst, int64_t B, int H, int N, int hd, int elt_bytes, int64_t src_b, int64_t src_h,
                          int64_t src_n, int64_t dst_b, int64_t dst_h, int64_t dst_n, dkd_stream_t stream);
DKD_API size_t dkd_colsum_workspace_bytes(int64_t M, int N);
DKD_API int dkd_colsum(const void* a, int64_t M, int N, int dtype, float* out, void* workspace, size_t workspace_bytes,
                       dkd_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Step epilogue (SURVEY 8f rank 3) and input-side helpers (rank 4): what tools/engine.py does around the criterion.
 *
 * dkd_step_epilogue — timm NativeScaler (torch GradScaler: unscale, inf/nan check, skipped step, scale update) +
 * gradient-norm clipping (`--clip-grad`: torch clip_grad_norm_) + AdamW (torch.optim.AdamW as built by timm
 * create_optimizer('adamw')) + timm ModelEma update, engine.py:58-69, in two launches over FLAT fp32 buffers of `n`
 * elements (parameters, gradients of the SCALED loss, exp_avg, exp_avg_sq, and the EMA copy or NULL).  Elements
 * [0, n_decay) receive decoupled weight decay, the rest (biases, norm scales: timm's no-decay group) do not.
 *   lr    : DEVICE fp32 scalar (a scheduler or a captured graph updates it in place)
 *   state : DEVICE fp32[8], owned by the caller, initialised to {loss_scale, 0, 0, 0, 0, 0, 0, 0}:
 *           [0] loss scale  [1] growth tracker  [2] optimizer step count  [3] 1 if the last step was skipped (non-finite
 *           gradients)  [4] total norm of the unscaled gradients  [5] clip coefficient applied.  Never read back by the host.
 *   beta1, beta2, ema_decay are doubles: 1 - x is formed in double (as the Python reference does) before rounding to fp32.
 *   clip_grad <= 0 disables clipping; dynamic_scale 0 keeps the loss scale fixed (use loss scale 1 for bf16 / fp32).
 *   zero_grad 1 clears the gradient buffer in the same pass (optimizer.zero_grad(), engine.py:58).
 *   workspace : >= dkd_step_workspace_bytes() bytes, zero-initialised once by the caller.
 */
DKD_API size_t dkd_step_workspace_bytes(void);
DKD_API int dkd_step_epilogue(float* params, float* grads, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n,
                              int64_t n_decay, const float* lr, double beta1, double beta2, float eps, float weight_decay,
                              float clip_grad, double ema_decay, int dynamic_scale, float growth_factor,
                              float backoff_factor, int growth_interval, int zero_grad, float* state, void* workspace,
                              size_t workspace_bytes, dkd_stream_t stream);
/* hits[0] = #rows whose target logit ranks < k0, hits[1] = ... < k1 (timm.utils.accuracy(output, target, topk=(k0, k1)),
 * engine.py:53-56: acc_k = 100 * hits / B); ties rank lower index first.  target int64 [B], hits fp32[2] (overwritten). */
DKD_API int dkd_topk_hits(const void* logits, const int64_t* target, int64_t B, int64_t C, int dtype, int k0, int k1,
                          float* hits, dkd_stream_t stream);
/* timm.data.Mixup (mode 'batch') image mixing, in place on x fp32 [B, CH, H, W] (train.py:288-295, engine.py:16-18):
 * use_cutmix 0: x[b] = lam * x[b] + (1 - lam) * x[B-1-b];  1: the box [y0,y1) x [x0,x1) of x[b] and x[B-1-b] is swapped.
 * lam is a DEVICE fp32 scalar (the same one dkd_logit_kd_fwdbwd takes as mix_lam). */
DKD_API int dkd_mix_batch(float* x, int64_t B, int64_t CH, int H, int W, const float* lam, int use_cutmix, int y0, int y1,
                          int x0, int x1, dkd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DELTAKD_H_ */
