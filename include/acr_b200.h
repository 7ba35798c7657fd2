/*
 * acr_b200.h -- C ABI of libacr_b200.so: the B200 (sm_100a) implementation of the ACR_WSSS
 * all-pairs attention-affinity hot path.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - return value: 0 = ok, <0 = invalid argument (ACR_E_*), >0 = a cudaError_t value;
 *     acr_last_error_string() describes the last failure on the calling thread;
 *   - no exceptions, no global state besides a lazily created per-device workspace cache;
 *   - there is no CPU fallback: with no usable sm_100 device every compute entry point fails.
 *
 * Each entry point cites the reference interface (file:line under the ACR_WSSS tree) it replaces.
 */
#ifndef ACR_B200_H_
#define ACR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACR_B200_ABI_VERSION 1

#define ACR_E_INVAL   (-1)  /* bad shape / null pointer / unsupported size          */
#define ACR_E_ALIGN   (-2)  /* pointer alignment requirement violated               */
#define ACR_E_NOSM100 (-3)  /* kernel needs an sm_100 device and none is current    */
#define ACR_E_NOMEM   (-4)  /* workspace too small                                  */

int acr_abi_version(void);
const char* acr_last_error_string(void);
/* 1 when the current device is compute capability 10.x (tcgen05/TMEM/TMA kernels usable). */
int acr_device_is_sm100(void);

/* Per-kernel device timing (bench.py's roofline): while enabled, the tensor-core attention kernels and the CAM finish kernel
 * are bracketed by CUDA event pairs on the launching stream.  acr_profile_read sums the elapsed time of every recorded launch
 * of `kernel` ("attn_fwd_kernel", "attn_mean_kernel", "attn_delta_kernel", "attn_bwd_kernel", "cam_finish_kernel") after
 * synchronising its events;
 * acr_profile_enable(0) drops the records.  Must be off during CUDA-graph capture. */
void acr_profile_enable(int on);
int acr_profile_read(const char* kernel, double* total_ms, long long* launches);

/* ------------------------------------------------------------------------------------------
 * (a1) Attention core.  Replaces models/vision_transformer.py:198-214 (Attention.forward, the part
 * between the qkv Linear and the proj Linear) together with the head mean of DPT/ACR.py:107-112.
 *
 * qkv is the output of the qkv Linear, UNPERMUTED: element (b,n,s,h,d) at ((b*N+n)*3+s)*H*D + h*D + d
 * (s=0 q, 1 k, 2 v) -- exactly the buffer the reference reshapes at vision_transformer.py:200.
 * out is [B,N,H*D] (the layout proj consumes, vision_transformer.py:211).
 * attn_mean points at slot l of the [B,L,N,N] fp32 stack: image b's N x N map starts at
 * attn_mean + b*mean_batch_stride (elements); rows are dense (stride N).  May be NULL.  mean_batch_stride must not be
 * negative and, for B > 1, at least N*N (the images' maps must not overlap); otherwise the call fails with ACR_E_INVAL.
 * p_row0 (nullable) receives the per-head softmax row of the cls token, [B,H,N] fp32 (GETAM, a8).
 * ------------------------------------------------------------------------------------------ */

/* Fused sm_100a path: bf16 operands, fp32 accumulate, tcgen05/TMEM/TMA.  D must be 64.
 * lse [B,H,N] fp32 receives log-sum-exp of the scaled scores (natural log) for the backward. */
int acr_attn_fwd_bf16(const void* qkv_bf16, int B, int N, int H, int D, float scale,
                      void* out_bf16, float* lse,
                      float* attn_mean, long long mean_batch_stride,
                      float* p_row0, void* stream);

/* Backward of the above with the dense affinity-gradient term (SURVEY section 9):
 *   dP_h = dO_h V_h^T + g_mean / H ;  dS_h = P_h * (dP_h - rowsum(P_h * dP_h)) ; dQ,dK,dV as usual.
 * g_mean (nullable) = dLoss/dA-bar for this block: element (b,i,j) at g_mean + b*g_batch_stride + i*g_row_stride + j
 * (row and batch strides that are multiples of 4 with a 16-byte aligned base enable 128-bit loads on full key tiles).
 * Alternatively (g_mean NULL) the gradient may be given as sign codes from acr_consistency_fwd_bwd: g_code with strides in
 * BYTES (row stride a multiple of 128 and >= the 128-padded N, base 16-byte aligned), the two weights, and an optional
 * DEVICE scalar g_scale multiplying them (NULL = 1; lets autograd's upstream gradient through without a host sync).
 * d_qkv_bf16 has the layout of qkv.  g_row0 (nullable, [B,H,N] fp32) receives row 0 of dP_h, which is
 * what the reference's save_attn_gradients hook keeps and getam consumes (DPT/ACR.py:182-213).
 * workspace: acr_attn_bwd_bf16_workspace() bytes, 256-byte aligned. */
size_t acr_attn_bwd_bf16_workspace(int B, int N, int H, int D);
int acr_attn_bwd_bf16(const void* qkv_bf16, const void* out_bf16, const float* lse,
                      const void* d_out_bf16, int B, int N, int H, int D, float scale,
                      const float* g_mean, long long g_batch_stride, long long g_row_stride,
                      const unsigned char* g_code, long long code_batch_stride, long long code_row_stride,
                      float w_cls, float w_aff, const float* g_scale,
                      void* d_qkv_bf16, float* g_row0,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Exact fp32 path (materialises P like the reference does; used for 1e-3 parity and for the
 * get_attn()/get_attn_gradients() accessor protocol, vision_transformer.py:186-196).
 * P [B,H,N,N] fp32 is written; out [B,N,H*D] fp32. */
int acr_attn_fwd_f32(const float* qkv, int B, int N, int H, int D, float scale,
                     float* P, float* out,
                     float* attn_mean, long long mean_batch_stride, void* stream);
/* dP [B,H,N,N] is a required output: on return it holds dP_h (= what the reference hook stores).
 * dS [B,H,N,N] is caller-provided scratch; d_qkv has the layout of qkv. */
int acr_attn_bwd_f32(const float* qkv, const float* P, const float* d_out,
                     int B, int N, int H, int D, float scale,
                     const float* g_mean, long long g_batch_stride,
                     float* dP, float* dS, float* d_qkv, void* stream);

/* ------------------------------------------------------------------------------------------
 * LayerNorm either side of the attention core (SURVEY section 8f rank 2).  Replaces the nn.LayerNorm(eps=1e-6) calls of
 * Block.forward, models/vision_transformer.py:230-233.  x [M,E] fp32 or bf16 (E a multiple of 128, <= 2048; dx has x's type); y [M,E] in fp32 or,
 * with y_is_bf16, directly in the bf16 operand type of the following Linear; mean/rstd [M] fp32 are kept for backward.
 * Backward: dy [M,E] fp32 or bf16 -> dx [M,E] fp32, dgamma/dbeta [E] fp32 (deterministic two-level reduction).
 * Residual fusion (Block.forward's `x = x + branch(x)` followed by the next norm): with `residual` (x's type) the kernel
 * normalises s = x + residual and also stores s in `sum_out`; in backward `d_residual` (dx's type, may be NULL) is the
 * gradient arriving over the skip connection and is added to dx before the single rounding; `dx_colsum` [E] (may be NULL)
 * receives the column sums of dx = the bias gradient of the Linear whose output was the residual branch.  With
 * `accumulate` != 0 all three [E] outputs (dgamma, dbeta, dx_colsum) are incremented instead of overwritten, so they can
 * point straight at fp32 .grad buffers.
 * ------------------------------------------------------------------------------------------ */
int acr_layernorm_fwd(const void* x, int x_is_bf16, const void* residual, void* sum_out, const float* gamma, const float* beta,
                      int M, int E, float eps, void* y, int y_is_bf16, float* mean, float* rstd, void* stream);
size_t acr_layernorm_bwd_workspace(int E);
int acr_layernorm_bwd(const void* dy, int dy_is_bf16, const void* d_residual, const void* x, int x_is_bf16, const float* mean, const float* rstd,
                      const float* gamma, int M, int E, void* dx, float* dgamma, float* dbeta, float* dx_colsum, int accumulate,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Column sums of a bf16 matrix: out[F] (+)= sum_m x[m,:]  (bias gradients of the Linear layers around the attention core;
 * deterministic two-stage reduction, fp32 accumulation).  workspace: acr_colsum_workspace(F) bytes. */
size_t acr_colsum_workspace(int F);
int acr_colsum_bf16(const void* x_bf16, int M, int F, float* out, int accumulate, void* workspace, size_t workspace_bytes,
                    void* stream);

/* Training-batch preparation on the GPU (SURVEY 8f rank 3).  Replaces the per-image body of get_data_from_chunk_v2,
 * myTool.py:1171-1196: RandomResizeLong (cv2.resize bilinear, :995-1008) -> flip (:895-899) -> ImageNet normalisation ->
 * RandomCrop into a zero-filled crop_size x crop_size container (:923-955).  src: the decoded uint8 RGB images, HWC, packed
 * back to back on the DEVICE; offsets[b]: byte offset of image b; params: 12 ints per image
 *   {h, w, resized_h, resized_w, flip, img_top, img_left, cont_top, cont_left, ch, cw, 0}
 * (the host draws them in the reference's RNG order: acr_wsss_b200/data.py).  out [B,3,crop,crop] fp32 normalised,
 * ori_out [B,3,crop,crop] uint8 (the de-normalised copy the reference also returns; may be NULL). */
int acr_augment_batch(const unsigned char* src, const long long* offsets, const int* params, int B, int crop_size,
                      float* out, unsigned char* ori_out, void* stream);

/* Optimiser update of the step on flat fp32 buffers (PolyOptimizer, tool/torchutils.py:10-31, as it really runs: SGD with
 * momentum = the weight-decay value, SURVEY Q2): buf = momentum*buf + grad ; param += (*neg_lr)*buf ; param_bf16 = bf16(param)
 * (param_bf16 may be NULL).  neg_lr is a DEVICE scalar (-lr_t), so the poly schedule works across CUDA-graph replays.
 * n a multiple of 4. */
int acr_sgd_momentum_step(float* param, const float* grad, float* momentum_buf, void* param_bf16, long long n,
                          float momentum, const float* neg_lr, void* stream);

/* Exact (erf) GELU of the ViT MLP (Mlp.act = nn.GELU, models/vision_transformer.py:148-164) on bf16 activations, fp32 math.
 * Forward: y[n] = gelu(x[n]).  Backward: dx[M,F] = dy * gelu'(x) and, when `colsum` is given, colsum[F] (+)= sum_m dx[m,:]
 * (the bias gradient of fc1) from the same pass.  F a multiple of 8; workspace: acr_gelu_bwd_workspace(F) bytes. */
int acr_gelu_fwd_bf16(const void* x_bf16, void* y_bf16, long long n, void* stream);
size_t acr_gelu_bwd_workspace(int F);
int acr_gelu_bwd_bf16(const void* x_bf16, const void* dy_bf16, void* dx_bf16, int M, int F, float* colsum, int accumulate,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a7) All-pairs consistency loss, forward and gradient in one pass.
 * Replaces train_acr.py:143-161 (= train_acr_coco.py:140-158): the slicing, the 3*p in-place
 * flips and the two F.l1_loss calls.  attn1/attn2 are the [B,L,N,N] fp32 stacks of the two views
 * (N = p*p+1), NOT modified.  loss2[0] = cls_align, loss2[1] = aff_align (means, before alpha).
 * g1/g2 (nullable together) receive alpha_cls*d(cls_align)/dA + alpha_aff*d(aff_align)/dA as [B,L,N] rows of
 * g_row_stride (>= N) floats; a stride that is a multiple of 4 lets the attention backward use 128-bit loads.
 * code1/code2 (nullable together; exclusive with g1/g2): the same gradients as one SIGN CODE byte per element, rows of
 * code_row_stride bytes: 0x00 = 0, 0x3F = +w, 0xBF = -w with w = alpha_cls/(B*L*(N-1)) on row 0 and
 * alpha_aff/(B*L*(N-1)^2) elsewhere (the code is the top byte of +-0.5f).  4x less HBM traffic than fp32 gradients;
 * acr_attn_bwd_bf16 consumes them directly.  The padding bytes [N, code_row_stride) of a row are written as 0x00; the
 * attention backward never reads them as gradient, so any row padding works there.
 * workspace: scratch of acr_consistency_workspace() bytes.
 * ------------------------------------------------------------------------------------------ */
size_t acr_consistency_workspace(int B, int L, int N);
int acr_consistency_fwd_bwd(const float* attn1, const float* attn2, int B, int L, int N, int p,
                            float alpha_cls, float alpha_aff,
                            float* loss2, float* g1, float* g2, long long g_row_stride,
                            unsigned char* code1, unsigned char* code2, long long code_row_stride,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a8) GETAM from row-0 quantities.  Replaces ACR.getam, DPT/ACR.py:177-215, for the part that
 * reaches the result (row 0 of each block's map).  p_row0/g_row0: [L,H,N] fp32 for ONE image
 * (per-block, per-head cls-token row of P and of dP).  func: 0 'grad', 1 'grad_s', 2 'cam_grad',
 * 3 'cam_grad_s'.  skip = 1 (2 for the distilled DeiT variant).  cam_out [N-skip] fp32.
 * cam_rows (nullable) [L,N] receives each block's c_l row 0.  The clamps keep NaN, as clamp(min=0) / relu do: a NaN in
 * g_row0, or in g*p for the cam_grad funcs (a NaN in p_row0, inf * 0), makes that token's c_l NaN, and its CAM too if
 * l >= start_layer.
 * ------------------------------------------------------------------------------------------ */
int acr_getam_row0(const float* p_row0, const float* g_row0, int L, int H, int N,
                   int start_layer, int func, int skip,
                   float* cam_out, float* cam_rows, void* stream);
/* The same for S (image, flip, class) samples at once (batched CAM inference, infer_cam.py:167-184 looped over images):
 * p_row0/g_row0 [L,S,H,N] (the per-block row-0 tensors of a batch of S samples stacked over the L used blocks),
 * cam_out [S,N-skip]. */
int acr_getam_row0_batch(const float* p_row0, const float* g_row0, int S, int L, int H, int N,
                         int start_layer, int func, int skip, float* cam_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a9) Affinity refinement.  Replaces infer_cam.py:164-165 (patch_aff = sum_l attn[:,l,1:,1:]) and
 * infer_cam.py:184 (matmul(patch_aff, cam)), batched over classes.
 * attn [B,L,N,N] fp32 -> A [B,Np,Np] with Np=N-1.  If normalize!=0 rows of A are divided by their sum.
 * cam [B,Np,C] -> out [B,Np,C] = A^t cam (t>=1).  tmp is [B,Np,C] scratch (only touched when t>1).
 * ------------------------------------------------------------------------------------------ */
int acr_affinity_sum(const float* attn, int B, int L, int N, int normalize, float* A, void* stream);
int acr_affinity_refine(const float* A, const float* cam, int B, int Np, int C, int t,
                        float* out, float* tmp, void* stream);

/* The same two steps fused and on the tensor cores (sm_100a, tcgen05 / TMEM; north star item 3):
 *   out [B,Np,C] = A^t cam with A = sum_l attn[:,l,1:,1:] summed while it is read (never materialised for t = 1);
 *   normalize != 0 divides every application by the row sums of A (= row-normalised affinity power).
 * fp32 operands are split into bf16 hi + lo parts (3 MMAs, fp32 accumulate): relative error ~2^-16.
 * C + (normalize ? 1 : 0) <= 128.  workspace: acr_affinity_refine_tc_workspace() bytes, 256-byte aligned, only for t > 1. */
size_t acr_affinity_refine_tc_workspace(int B, int N, int C, int t);
int acr_affinity_refine_tc(const float* attn, int B, int L, int N, const float* cam, int C, int t, int normalize,
                           float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Patch CAM on the tensor cores: out [B,M,C] = (relu)(tokens . weight^T + bias).  Replaces
 * F.relu(self.cls_head(x_patch)), DPT/ACR.py:133-134 (x_patch = layer_4[:,1:,:]).
 * tokens: fp32, element (b,i,k) at tokens + b*tok_batch_stride + i*tok_row_stride + k (pass the pointer to token 1);
 * weight [C,E] and bias [C] (nullable) as nn.Linear stores them; C <= 128.  Same bf16 hi/lo split as above. */
int acr_patch_cam_tc(const float* tokens, long long tok_batch_stride, long long tok_row_stride, int B, int M, int E,
                     const float* weight, const float* bias, int C, int relu, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Finish of batched CAM inference, one launch for a whole batch.  Replaces infer_cam.py:153-215 after the low-res maps
 * (the resizes to the original image size at :156-162 and :185-187, the flips, the sums over scales and views, and the
 * per-class min-max normalisation of :202,209) for M images whose original sizes may differ.
 *   scale s (num_scales in 1..8), HOST arrays: cams_host[s] -> cams_s [2M, ph_s*pw_s, n] (GETAM maps, channel-last),
 *   patch_host[s] -> patch_s [2M, ph_s*pw_s, C] (patch CAMs), grid_host[2s], grid_host[2s+1] = ph_s, pw_s.  Batch index
 *   v*M + m is view v of image m; view 0 is the horizontally flipped input.
 *   labels [M,C] (device): label values; a patch-CAM plane of class c of image m is multiplied by labels[m*C + c].
 *   planes_host: HOST table of num_planes planes (0..65535), 6 long long each {offset, image, channel, kind, rows, cols}:
 *     kind 0: GETAM plane of copy `channel` (< n) of cams_s, bilinear with align_corners=True, eps 1e-6;
 *     kind 1: patch-CAM plane of class `channel` (< C) of patch_s, align_corners=False, times the label, eps 1e-5.
 *   Each plane is written as rows x cols fp32 at out + offset (offset + rows*cols <= out_elems):
 *   norm(sum over scales, then views with view 0 first, of the bilinear resize to rows x cols, view 0 read at column
 *   cols-1-c), norm(x) = (x - min) / (max - min + eps) over the plane.  The resize is ATen's upsample_bilinear2d
 *   arithmetic for an explicit output size.  A plane whose sum holds a NaN is written as all NaN (amin / amax propagate
 *   it in the reference's normalisation).  Deterministic: no atomics.
 *   Low-res maps of all scales: 2 * sum_s ph_s*pw_s floats <= 200 KB.
 *   workspace: >= 48 * num_planes bytes, 8-byte aligned; receives a copy of the table on `stream`.
 * num_planes = 0 launches nothing (planes_host, out and workspace may then be NULL).
 * ------------------------------------------------------------------------------------------ */
int acr_cam_finish(const float* const* cams_host, const float* const* patch_host, const int* grid_host, int num_scales,
                   int M, int n, int C, const float* labels, const long long* planes_host, int num_planes,
                   float* out, long long out_elems, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pseudo-label evaluation.  Replaces evaluation.py:28-67 (pseudo_label's argmax over [tau, cam_1..cam_C], then label_iou's
 * per-class P, T, TP) for a whole sweep of background thresholds in one pass, for a batch of images of any sizes.
 * K = num_cls (1..255): labels 0 (background) .. K-1; a ground-truth pixel of 255 is ignored, one in [K, 255) is valid and
 * matches no label (label_iou's `cal = gt < 255`).
 *
 * acr_cam_label_counts:
 *   cams: packed fp32 planes (cam_elems floats); planes_host: HOST table of num_planes rows {offset, image, class}, the
 *   rows*cols plane of dict class `class` (0..K-2, label class+1) of image `image` at cams + offset.  Planes may come in any
 *   order; an image may have none; two planes of one image with the same class are rejected.
 *   gt: packed uint8 ground truth (gt_elems bytes); images_host: HOST table of num_images rows {gt_offset, rows, cols},
 *   1 <= rows*cols < 2^31.
 *   thresholds_host: HOST array of T = num_thresholds (1..4096) doubles, finite and non-descending after float32 rounding
 *   (equal neighbours are allowed); the comparison is made in float32, as pseudo_label's float32 tensor makes it.
 *   Per pixel with gt != 255: (c*, m) = the FIRST maximum over labels 1..K-1 in label order, a label without a plane reading
 *   0 (pseudo_label's zero planes; they decide when a threshold is negative or no plane is present); ties go to the lower
 *   label whatever the table order; a NaN in any plane makes c* the first NaN label (np.argmax).  The pseudo-label at
 *   threshold t is c* when m > float32(tau_t), else 0; j = #{t : float32(tau_t) < m} (a NaN m gives j = T).
 *   counts: caller-owned int64 DEVICE counters, ADDED TO (so a dataset streams through in batches), Tp = T + 1:
 *     [(K-1) * Tp] pixels with c* = c at row c-1, column j;   [(K-1) * Tp] the same with gt == c;
 *     [Tp] pixels with gt == 0 by j;   [K + 1] pixels with gt == g (g < K), then valid pixels with gt >= K.
 *   P, T, TP of label_iou at threshold t follow by suffix sums over j > t (cam.LabelEvaluator).
 *   Envelope: histograms of (2K-1)*(T+1)*4 + 4K bytes <= 200 KB (COCO K = 81 up to T = 316, VOC K = 21 up to T = 1247).
 *   workspace: >= acr_label_counts_workspace(num_images, num_planes, T) bytes, 8-byte aligned; receives the tables on
 *   `stream`.  Deterministic (integer atomics).  No image launches nothing.
 * acr_label_map_counts: label-map predictions (e.g. the argmax of crf_with_alpha's marginals).  pred and gt: packed uint8,
 *   elems bytes each, image i at the same offset in both; images_host rows {offset, rows, cols}.  counts [3][K] int64 DEVICE,
 *   added to: P[c] = #(pred == c), T[c] = #(gt == c), TP[c] = #(pred == gt == c) over pixels with gt != 255 (labels >= K count
 *   in no class).  workspace: >= acr_label_counts_workspace(num_images, 0, 0) bytes, 8-byte aligned.
 * Both reject null pointers, K out of range, a table row outside its buffer and a too-small workspace before any device work.
 * ------------------------------------------------------------------------------------------ */
size_t acr_label_counts_workspace(int num_images, int num_planes, int num_thresholds);
int acr_cam_label_counts(const float* cams, long long cam_elems, const long long* planes_host, int num_planes,
                         const unsigned char* gt, long long gt_elems, const long long* images_host, int num_images,
                         const double* thresholds_host, int num_thresholds, int num_cls, long long* counts,
                         void* workspace, size_t workspace_bytes, void* stream);
int acr_label_map_counts(const unsigned char* pred, const unsigned char* gt, long long elems, const long long* images_host,
                         int num_images, int num_cls, long long* counts, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Head of the dense-CRF regulariser (BASELINE configs[3]; call shape myTool.py:825-857, loop train_acr_coco.py:137-165):
 * the probabilities the bilateral filter sees, straight from the patch-token logits.
 *   logits [B,P*P,C] fp32 channel-last (cls_head(layer_4[:,1:]), DPT/ACR.py:133-134)
 *   seg    [B,C+1,S/2,S/2] = bilinear_down_0.5( softmax_k([0, bilinear_up(logits -> SxS)]) ), both align_corners=False
 * Backward: g_seg [B,C+1,S/2,S/2] -> d_up [B,C,S,S] = gradient with respect to the up-sampled logits (fold it to patch
 * resolution with the bilinear backward).  S even, 1 <= P <= S (the model up-samples; P > S is rejected, so the backward
 * never meets a shape the bilinear backward below does not take).
 * ------------------------------------------------------------------------------------------ */
int acr_crf_head_fwd(const float* logits, int B, int P, int C, int S, float* seg, void* stream);
int acr_crf_head_bwd(const float* logits, const float* g_seg, int B, int P, int C, int S, float* d_up, void* stream);
/* Backward of F.interpolate(x [planes,P,P] -> [planes,S,S], mode='bilinear', align_corners=False) without atomics:
 * d_patch [planes,P,P] = sum over the up-sampled pixels of their two-by-two tap weights times d_up [planes,S,S].  P <= S <= 512. */
int acr_bilinear_up_bwd(const float* d_up, int planes, int P, int S, float* d_patch, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a10) PAMR.  Replaces PAMR.forward, pamr.py:125-144, including the bilinear (align_corners=True)
 * up-sampling of the mask (pamr.py:126): x [B,K,H,W] image, mask [B,C,mh,mw], dilations_host[nd] on
 * the HOST (1 <= nd <= 8).  out [B,C,H,W].  workspace: acr_pamr_workspace() bytes (affinity planes +
 * ping-pong mask).
 * ------------------------------------------------------------------------------------------ */
size_t acr_pamr_workspace(int B, int K, int C, int H, int W, int nd);
int acr_pamr_fwd(const float* x, const float* mask, int B, int K, int C, int H, int W, int mh, int mw,
                 const int* dilations_host, int nd, int num_iter,
                 float* out, void* workspace, size_t workspace_bytes, void* stream);
/* Backward of PAMR.forward with respect to the mask and the image (first order, fp32).
 * acr_pamr_fwd_save: the forward with its state kept for the backward.  out is bitwise equal to acr_pamr_fwd's.  saved:
 *   caller-owned, acr_pamr_save_workspace() bytes (the affinity weights and the num_iter padded iterates M_0 .. M_{T-1}),
 *   256-byte aligned; it must stay untouched until acr_pamr_bwd has run.
 * acr_pamr_bwd: g_out [B,C,H,W] = dL/dout -> d_mask [B,C,mh,mw] and d_x [B,K,H,W] (either may be NULL, not both; with
 *   d_x NULL the image-side kernels do not run; num_iter = 0 writes d_x as zeros).  Same shapes, dilations and num_iter as
 *   the acr_pamr_fwd_save call that filled `saved`.  workspace: acr_pamr_bwd_workspace() bytes, 256-byte aligned.
 *   Deterministic (gathers, no atomics); no host synchronisation and no allocation, so it can be captured in a CUDA graph.
 * Both reject null pointers, shapes <= 0, nd outside 1..8, a dilation < 1, num_iter < 0, short buffers and grids beyond
 * H <= 65535, B*C <= 65535 before any device work. */
size_t acr_pamr_save_workspace(int B, int K, int C, int H, int W, int nd, int num_iter);
int acr_pamr_fwd_save(const float* x, const float* mask, int B, int K, int C, int H, int W, int mh, int mw,
                      const int* dilations_host, int nd, int num_iter,
                      float* out, void* saved, size_t saved_bytes, void* stream);
size_t acr_pamr_bwd_workspace(int B, int K, int C, int H, int W, int nd);
int acr_pamr_bwd(const float* x, const void* saved, size_t saved_bytes, const float* g_out, int B, int K, int C, int H, int W,
                 int mh, int mw, const int* dilations_host, int nd, int num_iter, float* d_x, float* d_mask,
                 void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a11) Permutohedral bilateral filter.  Replaces bilateralfilter_batch,
 * wrapper/bilateralfilter/bilateralfilter.cpp:42-55 (and Permutohedral::init/compute,
 * permutohedral.cpp:115-440,507-631).  Same argument meaning and order as the SWIG export
 * (bilateralfilter.hpp:12); images [N,3,H,W] in 0..255, ins/outs [N,K,H,W], fp32.
 *   acr_bilateral_batch       : DEVICE buffers + workspace (acr_bilateral_workspace() bytes).
 *   bilateralfilter_batch_b200: HOST buffers, the literal drop-in for the SWIG symbol (copies
 *                               host->device, runs the kernels, copies back; returns void like the
 *                               reference; on failure `outs` is left untouched and the error is
 *                               readable through acr_last_error_string()).
 * lattice_size_host (nullable) receives M (number of lattice vertices) per image, for reporting.
 * ------------------------------------------------------------------------------------------ */
size_t acr_bilateral_workspace(int N, int K, int H, int W);
int acr_bilateral_batch(const float* images, const float* ins, float* outs,
                        int N, int K, int H, int W, float sigmargb, float sigmaxy,
                        void* workspace, size_t workspace_bytes, int* lattice_size_host, void* stream);
void bilateralfilter_batch_b200(const float* images_host, int len_images, const float* ins_host, int len_ins,
                                float* outs_host, int len_outs,
                                int N, int K, int H, int W, float sigmargb, float sigmaxy);

/* ------------------------------------------------------------------------------------------
 * Dense-CRF mean-field inference: densecrf 2.x as tool/imutils.py crf_inference drives it (a Potts model over a Gaussian
 * kernel on (x/sxy_g, y/sxy_g) and a bilateral kernel on (x/sxy_b, y/sxy_b, r/srgb, g/srgb, b/srgb), both permutohedral,
 * DIAG_KERNEL + NORMALIZE_SYMMETRIC).  DEVICE buffers: images [N,3,H,W] in 0..255, probs [N,C,H,W] scores (need not sum
 * to 1; unary = -log(max(P, clip))), q_out [N,C,H,W] the marginals after n_iter iterations (n_iter = 0: softmax of the
 * clipped log-scores).  PSA defaults: sxy_g = 3, compat_g = 3, sxy_b = 80, srgb = 13, compat_b = 10, clip = 1e-5.
 * 1 <= C <= 96, 6*H*W < 2^28, sigmas finite and > 0 (small enough sigmas for the image size are rejected: lattice keys are
 * int16), compat finite, clip in (0, 1].  workspace: acr_dense_crf_workspace() bytes, 256-byte aligned.
 * Deterministic (two calls, or an image alone and inside a batch, give the same bits); no host synchronisation and no
 * allocation, so the call can be captured in a CUDA graph.  A splat value outside the fixed-point range makes that image's
 * q_out NaN.
 * ------------------------------------------------------------------------------------------ */
size_t acr_dense_crf_workspace(int N, int C, int H, int W);
int acr_dense_crf(const float* images, const float* probs, float* q_out, int N, int C, int H, int W, int n_iter,
                  float sxy_g, float compat_g, float sxy_b, float srgb, float compat_b, float clip,
                  void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ACR_B200_H_ */
