/*
 * vidar_b200.h -- C ABI of libvidar_b200.so: the B200 (sm_100a) kernels that sit
 * under ViDAR's two hot-path operator boundaries.
 *
 *   (i)  multi-scale deformable attention   (mmcv `_ext.ms_deform_attn_{forward,backward}`,
 *        bound at projects/mmdet3d_plugin/bevformer/modules/multi_scale_deformable_attn_function.py:10-12,
 *        called at :42-48, :74-84, :118-124, :150-160)
 *   (ii) the voxel ray-caster family        (third_lib/dvr/dvr.cpp:65-69, third_lib/dvxlr/dvxlr.cpp:61-65,
 *        third_lib/dvxlr/dvxlr_v2.cpp:67-70) and the in-model renderers built on the same
 *        volume (latent_rendering.py:79-162, vidar_head_base.py:420-509,586-592,662-752).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to a dense, contiguous, 16-byte aligned buffer
 *     unless the parameter name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     no entry point synchronises the device or allocates memory;
 *   - return value 0 = success, non-zero = VIDAR_E_* ; vidar_last_error() gives the
 *     message of the last failure on the calling thread (the Python layer turns it
 *     into RuntimeError/ValueError, the reference raises through TORCH_CHECK);
 *   - all floating-point I/O is fp32 (the reference casts to fp32 with
 *     custom_fwd(cast_inputs=torch.float32), multi_scale_deformable_attn_function.py:93;
 *     the ray-casters are dispatched on float tensors, dvr.cu:367).
 *
 * No torch types appear here: the library links only against libcudart.
 */
#ifndef VIDAR_B200_H_
#define VIDAR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  VIDAR_OK = 0,
  VIDAR_E_INVALID = 1,   /* bad argument (shape, null pointer, unknown enum) */
  VIDAR_E_CUDA = 2,      /* a CUDA runtime call or launch failed */
  VIDAR_E_UNSUPPORTED = 3
};

/* Message of the last error raised on this thread ("" if none). */
const char* vidar_last_error(void);
/* Library / build identification, e.g. "vidar_b200 0.1 sm_100a". */
const char* vidar_version(void);
/* Number of kernels this library has launched since load (all threads).  bench.py
 * reports the delta across the timed region as `gpu_launches`. */
int64_t vidar_launch_count(void);

/* ------------------------------------------------------------------------------------
 * (i) Multi-scale deformable attention
 * ---------------------------------------------------------------------------------- */

/* Replaces ext_module.ms_deform_attn_forward
 *   (multi_scale_deformable_attn_function.py:118-124).
 *   value            [B, K, H, C]        K = sum_l Hl*Wl
 *   spatial_shapes   [L, 2] int64 (h, w) (device)
 *   level_start      [L]    int64        (device)
 *   sampling_loc     [B, Q, H, L, P, 2]  (x, y) normalised to [0,1]
 *   attn_weight      [B, Q, H, L, P]
 *   out              [B, Q, H*C]         fully overwritten
 * im2col_step is validated like mmcv (B % min(B, im2col_step) == 0) and otherwise unused. */
int vidar_msda_forward(const float* value, const int64_t* spatial_shapes,
                       const int64_t* level_start, const float* sampling_loc,
                       const float* attn_weight, float* out,
                       int B, int K, int H, int C, int L, int Q, int P,
                       int im2col_step, void* stream);

/* Replaces ext_module.ms_deform_attn_backward
 *   (multi_scale_deformable_attn_function.py:150-160).
 *   grad_out          [B, Q, H*C]
 *   grad_value        [B, K, H, C]        accumulated with atomics: caller zeroes it
 *                                         (torch.zeros_like, :146)
 *   grad_sampling_loc [B, Q, H, L, P, 2]  fully overwritten
 *   grad_attn_weight  [B, Q, H, L, P]     fully overwritten                              */
int vidar_msda_backward(const float* value, const int64_t* spatial_shapes,
                        const int64_t* level_start, const float* sampling_loc,
                        const float* attn_weight, const float* grad_out,
                        float* grad_value, float* grad_sampling_loc,
                        float* grad_attn_weight,
                        int B, int K, int H, int C, int L, int Q, int P,
                        int im2col_step, void* stream);

/* MSDeformableAttention3D's sampling with its elementwise prologue folded in
 *   (spatial_cross_attention.py:339-371 + the two calls above):
 *     attn = softmax_{L*P}(logits)                       (:339-342)
 *     loc  = offsets / (W_l, H_l) + ref_points[b, q, p % D]   (:356-371, point p = j*D + z)
 *   ref_points  [B, Q, D, 2]        projected Z-anchors (reference_points_cam), normalised
 *   offsets     [B, Q, H, L, P, 2]  raw output of the sampling_offsets Linear (pixels of level l)
 *   logits      [B, Q, H, L*P]      raw output of the attention_weights Linear
 * Requires L*P == 32 and head dim 16/32/64 (the shipped SCA configuration: 4 levels x 8 points).
 * Backward: grad_value accumulated (caller zeroes), grad_offsets / grad_logits overwritten; the
 * reference points carry no gradient (they come from the camera geometry). */
int vidar_msda_sca_forward(const float* value, const int64_t* spatial_shapes,
                           const int64_t* level_start, const float* ref_points,
                           const float* offsets, const float* logits, float* out,
                           int B, int K, int H, int C, int L, int Q, int P, int D, void* stream);
int vidar_msda_sca_backward(const float* value, const int64_t* spatial_shapes,
                            const int64_t* level_start, const float* ref_points,
                            const float* offsets, const float* logits, const float* grad_out,
                            float* grad_value, float* grad_offsets, float* grad_logits,
                            int B, int K, int H, int C, int L, int Q, int P, int D, void* stream);

/* Row-indirect variants: SpatialCrossAttention's rebatch / scatter-add (spatial_cross_attention.py:135-172)
 * folded into the op (SURVEY.md 8f-1).  A row is entry j of camera c's visible-pillar list:
 *   idx        [cams, Qd] int32   pillar of row j (ascending; entries >= count[c] unused), NULL: row j = pillar j
 *   count      [cams]     int32   live rows per camera, on the DEVICE (no host sync), NULL: all Qrows rows live
 *   inv_count  [bs, Qd]           1 / clamp(#cameras seeing the pillar, 1)  (:168-171), NULL: 1
 *   value      [bs*ncl, K, H, C]  the launch's cameras cam0 .. cam0+ncl-1, batch-major (n = b*ncl + camera)
 *   slots      [bs, Qd, H*C]      caller-zeroed; every live row adds inv_count * (its head vectors) to the slot
 *                                 of its pillar with red.global.add.v4.f32 (the reference's `slots[j, idx] += ...`
 *                                 followed by `slots / count`)
 * The launch covers rows j with (j / 64) % S in [s_lo, s_hi): interleaved sub-slices of a camera's list, the
 * unit of work when cameras are sharded over ranks (SURVEY.md 8e); S = 1, [0, 1) = every row.
 * `rows`: sampling locations / weights given per row, [bs*ncl, Qrows, H, L, P(, 2)] -- the plain op's inputs.
 * `sca_rows`: the fused MSDeformableAttention3D prologue of vidar_msda_sca_*, with
 *   ref_cam [cams, bs, Qd, D, 2] (reference_points_cam as point_sampling lays it out) and offsets / logits
 *   DENSE per pillar, [bs, Qd, H, L, P, 2] / [bs, Qd, H, L*P]: they are Linear(query) rows, equal for every
 *   camera that sees the pillar, so they are computed once per pillar and read through idx.
 * Backward: grad_slots [bs, Qd, H*C] is read through the same map; grad_value accumulated (caller zeroes);
 *   rows:     grad_sampling_loc / grad_attn_weight written for the rows of this launch (caller zeroes the rest);
 *   sca_rows: grad_offsets / grad_logits ACCUMULATED over cameras with red.global.add (caller zeroes). */
int vidar_sca_compact(const unsigned char* bev_mask, int32_t* idx, int32_t* count, float* inv_count,
                      int cams, int bs, int Q, int D, void* stream);
int vidar_msda_rows_forward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start,
                            const float* sampling_loc, const float* attn_weight, const int32_t* idx,
                            const int32_t* count, const float* inv_count, float* slots, int bs, int ncl,
                            int cam0, int K, int H, int C, int L, int Qrows, int Qd, int P, int S, int s_lo,
                            int s_hi, void* stream);
int vidar_msda_rows_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start,
                             const float* sampling_loc, const float* attn_weight, const int32_t* idx,
                             const int32_t* count, const float* inv_count, const float* grad_slots,
                             float* grad_value, float* grad_sampling_loc, float* grad_attn_weight, int bs,
                             int ncl, int cam0, int K, int H, int C, int L, int Qrows, int Qd, int P, int S,
                             int s_lo, int s_hi, void* stream);
int vidar_msda_sca_rows_forward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start,
                                const float* ref_cam, const float* offsets, const float* logits,
                                const int32_t* idx, const int32_t* count, const float* inv_count, float* slots,
                                int bs, int ncl, int cam0, int K, int H, int C, int L, int Qrows, int Qd, int P,
                                int D, int S, int s_lo, int s_hi, void* stream);
int vidar_msda_sca_rows_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start,
                                 const float* ref_cam, const float* offsets, const float* logits,
                                 const int32_t* idx, const int32_t* count, const float* inv_count,
                                 const float* grad_slots, float* grad_value, float* grad_offsets,
                                 float* grad_logits, int bs, int ncl, int cam0, int K, int H, int C, int L,
                                 int Qrows, int Qd, int P, int D, int S, int s_lo, int s_hi, void* stream);

/* (i-c) The Linear layer in front of the sampling (SURVEY.md 8f-4): value_proj of MSDeformableAttention3D
 * (spatial_cross_attention.py:333) over the flattened camera features (modules/transformer.py:159-179),
 * y [M, N] = x [M, K] w[N, K]^T + bias[N], fp32 in / out.  tcgen05 tensor cores with a 3xTF32 split (fp32
 * accuracy, ~1e-6 relative: a plain TF32 GEMM would miss the 1e-4 parity bar), operands by TMA, accumulator in
 * TMEM.  K % 32 == 0, N % 128 == 0; bias may be NULL.  w_split: 2*N*K floats of caller-owned scratch. */
int vidar_linear_tf32x3(const float* x, const float* w, const float* bias, float* y, float* w_split,
                        int M, int N, int K, void* stream);

/* ------------------------------------------------------------------------------------
 * (ii-a) dvr / dvxlr / dvxlr_v2 voxel ray-casters
 *   sigma   [N, T, Z, Y, X]   (reference names the dims H, L, W)
 *   origin  [N, T, 3]         voxel units (x, y, z)
 *   points  [N, M, 3]         voxel units (x, y, z), NaN for padded rays
 *   tindex  [N, M]            FLOAT frame index, < 0 = padded ray (skipped)
 *   T  = sigma frames, To = origin frames (origin is indexed by t, sigma by
 *        ts = (T == 1) ? 0 : t, dvr.cu:97,109)
 * ---------------------------------------------------------------------------------- */

/* dvr.init / dvxlr.init (dvr.cu:14-63,705-738; dvxlr.cu:12-61,528-561).
 *   occupancy [N, T, Z, Y, X]  caller zeroes it; set to 1 at every ray end point. */
int vidar_dvr_init(const float* points, const float* tindex, float* occupancy,
                   int N, int M, int T, int Z, int Y, int X, void* stream);

/* dvr.render_forward (dvr.cu:65-317,327-383).  train_phase: 0 = "test", 1 = "train".
 *   pred_dist, gt_dist [N, M]  caller fills with -1 (dvr.cu:354-355); rays that never
 *   enter the grid keep it. */
int vidar_dvr_render_forward(const float* sigma, const float* origin, const float* points,
                             const float* tindex, float* pred_dist, float* gt_dist,
                             int N, int M, int T, int To, int Z, int Y, int X,
                             int train_phase, void* stream);

/* dvr.render (dvr.cu:385-627,639-694): forward + loss gradient in one call.
 *   loss_type: 0 = "l1" (also "bce", dvr.cu:667-668), 1 = "l2", 2 = "absrel".
 *   grad_sigma [N, T, Z, Y, X]  caller zeroes it; accumulated atomically (the
 *   reference's `+=` at dvr.cu:622 is a documented race; this is the race-free sum). */
int vidar_dvr_render(const float* sigma, const float* origin, const float* points,
                     const float* tindex, float* pred_dist, float* gt_dist,
                     float* grad_sigma, int N, int M, int T, int To, int Z, int Y, int X,
                     int loss_type, void* stream);

/* dvxlr.render (dvxlr.cu:160-517) and dvxlr_v2.render_v2 (dvxlr_v2.cu:119-493).
 *   max_d                  third dim of the list outputs (reference: 1026, dvxlr.cu:10)
 *   dd_dsigma [N, M, max_d]      caller zeroes            (dvxlr.cu:492)
 *   indices   [N, M, max_d, 3]   caller zeroes; (z, y, x) stored as float (dvxlr.cu:450-452)
 *   (dd_dsigma and indices may both be NULL: the lists are then not written -- used by
 *    the fused autograd path, which never needs them)
 *   v2 only (pass NULL for v1):
 *   sigma_regul [N, T, Z, Y, X]
 *   ray_pred  [N, M, max_d]      caller zeroes            (dvxlr_v2.cu:467)
 *   indicator [N, M, max_d]      caller fills with -1     (dvxlr_v2.cu:468)               */
int vidar_dvxlr_render(const float* sigma, const float* origin, const float* points,
                       const float* tindex, const float* sigma_regul,
                       float* pred_dist, float* gt_dist, float* dd_dsigma, float* indices,
                       float* ray_pred, float* indicator,
                       int N, int M, int T, int To, int Z, int Y, int X, int max_d,
                       void* stream);

/* Forward half of DifferentiableVoxelRendering without the lists: pred_dist / gt_dist
 * only (both caller-filled with -1), same traversal as dvxlr.render. */
int vidar_dvxlr_forward(const float* sigma, const float* origin, const float* points,
                        const float* tindex, float* pred_dist, float* gt_dist,
                        int N, int M, int T, int To, int Z, int Y, int X, void* stream);

/* dvxlr.get_grad_sigma (dvxlr.cu:63-156) and dvxlr_v2.get_grad_sigma_v2 (dvxlr_v2.cu:12-115).
 *   elementwise_mult [N, M, max_d]; indices [N, M, max_d, 3]
 *   grad_sigma [N, T, Z, Y, X] caller zeroes.
 *   v2 only (NULL for v1): indicator, grad_ray_pred [N, M, max_d]; grad_sigma_regul like
 *   grad_sigma, caller zeroes. */
int vidar_dvxlr_get_grad_sigma(const float* elementwise_mult, const float* indices,
                               const float* tindex, const float* indicator,
                               const float* grad_ray_pred, float* grad_sigma,
                               float* grad_sigma_regul,
                               int N, int M, int T, int Z, int Y, int X, int max_d,
                               void* stream);

/* Fused backward of DifferentiableVoxelRendering[V2] (e2e_predictor_utils.py:91-143):
 * re-walks every ray and scatters grad_pred[n,m] * d pred/d sigma straight into
 * grad_sigma -- the [N,M,1026(,3)] lists are never materialised.  Same result as
 * dvxlr.render + `gradpred[...,None]*dd_dsigma` (NaN -> 0, :104-108) + get_grad_sigma.
 *   grad_pred [N, M];  grad_sigma caller-zeroed.
 *   v2 only (NULL otherwise): grad_ray_pred [N, M, max_d] -> grad_sigma_regul. */
int vidar_dvxlr_backward_fused(const float* sigma, const float* origin, const float* points,
                               const float* tindex, const float* grad_pred,
                               const float* grad_ray_pred, float* grad_sigma,
                               float* grad_sigma_regul,
                               int N, int M, int T, int To, int Z, int Y, int X, int max_d,
                               void* stream);

/* ------------------------------------------------------------------------------------
 * (ii-b) ViDAR head: ray sampler, fused cross-entropy, arg-max decode
 *   (projects/mmdet3d_plugin/bevformer/dense_heads/vidar_head_base.py:420-509, 586-592, 706-738)
 *   sigma  [F, Z, Y, X]  the F frame volumes of one batch element
 *   origin [F, 3], points [R, 3] (voxel units), frame [R] int32 frame of each ray (NULL = 0)
 *   Per ray: sample 0 = the GT point (with_gt), then num_way waypoints at
 *   o + u*(k+0.5)*step; K = num_way + with_gt samples; logit = trilinear grid_sample
 *   (align_corners=False, zeros) or -inf where any normalised coordinate leaves (-1,1).
 * ---------------------------------------------------------------------------------- */

/* Materialising sampler = the per-(batch,frame) body of _get_grid_features (:433-500).
 *   logits [R, K] (NULL = skip), length [R, K] |x-o| (NULL = skip),
 *   valid [R] 1/0: GT point strictly inside the volume (:464) (NULL = skip). */
int vidar_ray_sample(const float* sigma, const float* origin, const float* points,
                     const int32_t* frame, float* logits, float* length, float* valid,
                     int R, int F, int Z, int Y, int X, int num_way, float step, int with_gt,
                     void* stream);

/* Its backward: grad_sigma [F,Z,Y,X] (caller-zeroed) += trilinear scatter of grad_logits. */
int vidar_ray_sample_backward(const float* origin, const float* points, const int32_t* frame,
                              const float* grad_logits, float* grad_sigma,
                              int R, int F, int Z, int Y, int X, int num_way, float step,
                              int with_gt, void* stream);

/* Fused sampler + F.cross_entropy(label 0) (:586-588): ce[r] = logsumexp(logits) - logit_0.
 *   ce, lse, valid [R]; rays whose GT point is outside get ce = 0, valid = 0. */
int vidar_ray_ce_forward(const float* sigma, const float* origin, const float* points,
                         const int32_t* frame, float* ce, float* lse, float* valid,
                         int R, int F, int Z, int Y, int X, int num_way, float step,
                         void* stream);

/* Backward of the fused CE: grad_sigma (caller-zeroed) += sum_r grad_ce[r] * d ce[r]/d sigma.
 *   lse from the forward; grad_ce NULL = all ones. */
int vidar_ray_ce_backward(const float* sigma, const float* origin, const float* points,
                          const int32_t* frame, const float* lse, const float* grad_ce,
                          float* grad_sigma, int R, int F, int Z, int Y, int X, int num_way,
                          float step, void* stream);

/* Inference decode (:706-732): exact zeros -> -inf, first arg-max over the num_way
 * waypoints; depth [R] = its |x-o| (voxel units), index [R] (float, NULL = skip). */
int vidar_ray_argmax(const float* sigma, const float* origin, const float* points,
                     const int32_t* frame, float* depth, float* index,
                     int R, int F, int Z, int Y, int X, int num_way, float step, void* stream);

/* Fused gumbel decode of the dense loss term: ViDARHeadBase._custom_gumbel_softmax_distance
 * (vidar_head_base.py:754-773) applied to the sampler's logits without the GT slot (:631-636).
 *   noise [R, num_way]  Gumbel(0,1) noise, drawn by the host like F.gumbel_softmax draws it
 *   dist  [R]           length of the sampled waypoint (0 for rays whose end point is outside)
 *   lse, p_next [R]     saved for the backward (log-sum-exp of the logits, softmax mass beyond dist)
 * Backward: grad_sigma (caller-zeroed) += grad_dist[r] * dist[r] * softmax_k * ([len_k > dist[r]] - p_next[r]). */
int vidar_ray_gumbel_forward(const float* sigma, const float* origin, const float* points,
                             const int32_t* frame, const float* noise, float* dist, float* lse,
                             float* p_next, int R, int F, int Z, int Y, int X, int num_way,
                             float step, void* stream);
int vidar_ray_gumbel_backward(const float* sigma, const float* origin, const float* points,
                              const int32_t* frame, const float* dist, const float* lse,
                              const float* p_next, const float* grad_dist, float* grad_sigma,
                              int R, int F, int Z, int Y, int X, int num_way, float step,
                              void* stream);

/* ------------------------------------------------------------------------------------
 * (ii-c) LatentRendering core
 *   (projects/mmdet3d_plugin/bevformer/modules/ray_operations/latent_rendering.py:98-161:
 *   everything between the three Linear layers).  act: 0 = 'exp' (1-exp(-relu x)), 1 = 'sigmoid'.
 *   CHANNEL-LAST maps, as the Linear layers emit them:
 *   occ    [bs, Hb, Wb, D]     output of unsup_raymarching_head (:94), D = pred_height
 *   feat   [bs, Hb, Wb, D*G]   output of lora_a (:134); channel = d*G + j
 *   prob   [bs, Hb, Wb, D]     out: occ_path_prob (:127-128)
 *   pooled [bs, Hb*Wb, D*G]    out: ray-pooled feature that feeds lora_b (:148-153)
 *   grid_num waypoints of step grid_step / (min(Hb,Wb)//2) (:101-104); eps (:80,147).
 *   Supported: D a power of two <= 32, G in {1, 2, 4, 8, 16} (the reference default
 *   pred_height=1, reduction=16, embed_dims=256 is D=1, G=16).
 * ---------------------------------------------------------------------------------- */
int vidar_latent_render_forward(const float* occ, const float* feat, float* prob, float* pooled,
                                float* aux, int bs, int D, int G, int Hb, int Wb, int grid_num,
                                float grid_step, float eps, int act, void* stream);

/* aux (may be NULL everywhere): [3, bs, Hb, Wb, D] floats the forward fills (product of the
 * non-zero transmittance factors, count of zero factors, sum of sampled probabilities) so the
 * backward does not have to march the rays again to recompute them.
 *
 * Backward.  grad_prob [bs,Hb,Wb,D] = gradient reaching `prob` from outside the core (the
 * final product, :158-160); grad_pooled [bs,Hb*Wb,D*G]; pooled = forward output (needed with aux).
 * grad_prob_total [bs,Hb,Wb,D] is scratch (fully overwritten).  grad_occ, grad_feat:
 * caller-zeroed, shaped like occ, feat. */
int vidar_latent_render_backward(const float* occ, const float* feat, const float* prob,
                                 const float* pooled, const float* aux, const float* grad_prob,
                                 const float* grad_pooled, float* grad_prob_total, float* grad_occ,
                                 float* grad_feat, int bs, int D, int G, int Hb, int Wb,
                                 int grid_num, float grid_step, float eps, int act, void* stream);

/* The same four kernels, one phase per call, on a range [cell0, cell0+ncells) of the
 * bs*Hb*Wb BEV cells (row-major): when the cells are sharded over GPUs the host places a
 * collective on the small maps between the phases (vidar_b200/modules/latent_rendering.py).
 * Outputs are indexed by GLOBAL cell; scatter targets (grad_*) are caller-zeroed full maps
 * that receive this range's contributions. */
int vidar_latent_prob_forward(const float* occ, float* prob, float* aux, int bs, int D, int Hb,
                              int Wb, int grid_num, float grid_step, int act,
                              long long cell0, long long ncells, void* stream);
int vidar_latent_pool_forward(const float* prob, const float* feat, float* pooled, float* aux,
                              int bs, int D, int G, int Hb, int Wb, int grid_num,
                              float grid_step, float eps,
                              long long cell0, long long ncells, void* stream);
int vidar_latent_pool_backward(const float* prob, const float* feat, const float* pooled,
                               const float* aux, const float* grad_pooled,
                               float* grad_prob_map, float* grad_feat,
                               int bs, int D, int G, int Hb, int Wb, int grid_num,
                               float grid_step, float eps,
                               long long cell0, long long ncells, void* stream);
int vidar_latent_prob_backward(const float* occ, const float* aux, const float* grad_prob_total,
                               float* grad_occ, int bs, int D, int Hb, int Wb, int grid_num,
                               float grid_step, int act, long long cell0, long long ncells,
                               void* stream);

/* LatentRendering's projections around the ray-marching core, fused (one kernel per direction
 * on each side; replaces 3 + 6 skinny cuBLAS GEMMs and the elementwise kernels between them):
 *   latent_rendering.py:94   occ  = unsup_raymarching_head(embed)   (single Linear, num_pred_fcs == 0)
 *   latent_rendering.py:134  feat = lora_a(embed)
 *   latent_rendering.py:153-155  out = lora_b(pooled).view(.., D, E/D) * prob.view(.., D, 1)
 * rows = bs*Hb*Wb (or any contiguous row range of it: pass offset pointers); E = embed_dims
 * (128 or 256), D = pred_height, A = embed_dims / reduction; D + A <= 32.
 * Weights in nn.Linear layout [out, in].  Backward entry points ADD into grad_w and grad_b
 * (caller zero-fills) and overwrite the per-row gradients. */
int vidar_latent_proj_in_forward(const float* embed, const float* w_occ, const float* b_occ,
                                 const float* w_feat, const float* b_feat, float* occ, float* feat,
                                 long long rows, int E, int D, int A, void* stream);
int vidar_latent_proj_in_backward(const float* embed, const float* w_occ, const float* w_feat,
                                  const float* grad_occ, const float* grad_feat, float* grad_embed,
                                  float* grad_w_occ, float* grad_b_occ, float* grad_w_feat,
                                  float* grad_b_feat, long long rows, int E, int D, int A,
                                  void* stream);
int vidar_latent_proj_out_forward(const float* pooled, const float* prob, const float* w,
                                  const float* b, float* out, long long rows, int E, int D, int A,
                                  void* stream);
int vidar_latent_proj_out_backward(const float* grad_out, const float* pooled, const float* prob,
                                   const float* w, const float* b, float* grad_pooled,
                                   float* grad_prob, float* grad_w, float* grad_b,
                                   long long rows, int E, int D, int A, void* stream);

/* ------------------------------------------------------------------------------------
 * (i-b) BEV pillar -> camera projection, BEVFormerEncoder.point_sampling
 *   (projects/mmdet3d_plugin/bevformer/modules/encoder.py:94-156)
 *   ref3d [B, D, Q, 3] normalised pillar points; lidar2img [B, cams, 4, 4];
 *   pc_range_host: 6 floats in HOST memory (x0,y0,z0,x1,y1,z1); img_h/img_w = img_shape
 *   out: ref_cam [cams, B, Q, D, 2], bev_mask [cams, B, Q, D] (uint8 0/1).
 * ---------------------------------------------------------------------------------- */
int vidar_point_sampling(const float* ref3d, const float* lidar2img, const float* pc_range_host,
                         float* ref_cam, unsigned char* bev_mask, int B, int D, int Q, int cams,
                         float img_h, float img_w, void* stream);

/* ------------------------------------------------------------------------------------
 * (iii) nearest neighbour (K = 1) for the Chamfer distance -- SURVEY.md 8(f) item 2
 *   (third_lib/chamfer_dist/chamferdist/chamferdist/knn.cu:21-260, knn_cpu.cpp:7-106,
 *   chamfer.py:20-133; used by bevformer/utils/e2e_predictor_utils.py:163-183)
 *   p1 [N, P1, D], p2 [N, P2, D] (D = 2, 3 or 4); lengths1/2 [N] int64 (NULL = full)
 *   dists [N, P1] squared distance to the nearest p2 point, idx [N, P1] int64; zero padded
 *   beyond lengths1.  scratch: N*P1 uint64 (fully overwritten).
 * ---------------------------------------------------------------------------------- */
int vidar_nn_forward(const float* p1, const float* p2, const int64_t* lengths1,
                     const int64_t* lengths2, float* dists, int64_t* idx,
                     unsigned long long* scratch, int N, int P1, int P2, int D, void* stream);

/* knn_points_backward (knn_cpu.cpp:64-106): grad_p1 [N,P1,D] and grad_p2 [N,P2,D], both
 * caller-zeroed. */
int vidar_nn_backward(const float* p1, const float* p2, const int64_t* lengths1,
                      const int64_t* lengths2, const int64_t* idx, const float* grad_dists,
                      float* grad_p1, float* grad_p2, int N, int P1, int P2, int D, void* stream);

/* ------------------------------------------------------------------------------------
 * (iv) point-cloud forecasting metrics, one segment = one (batch element, frame), N = bs * F
 *   (ViDAR.forward_test, bevformer/detectors/vidar.py:389-502; get_rendered_pcds,
 *   dense_heads/vidar_head_base.py:344-389; compute_chamfer_distance_inner,
 *   utils/e2e_predictor_utils.py:146-184; clamp / _clamp / compute_ray_errors, utils/eval_utils.py:21-225)
 *
 * vidar_eval_gather: origin [bs, F, 3], points [bs, M, 3] (NaN padding), tindex [bs, M] (-1 padding),
 *   gt_dist / pred_dist [bs, M] (metres; both NULL: the points themselves are the cloud of every
 *   frame, pred = GT), pc_range_host: 6 host floats.  Rays of segment (b, t): tindex == t, gt_dist > 0,
 *   and inside pc_range if within_grid.  Writes stably ordered (ray order) lists, padded to M:
 *     pred_in, gt_in [N, M, 3]   predicted / GT points inside pc_range       counts[0*N + s], counts[1*N + s]
 *     pred_sph [N, M, 3], pred_dhat [N, M]  (atan2(x,y), atan2(z,y), 1) of pred - origin with d_hat > 1e-2,
 *                                            and d_hat                        counts[2*N + s]
 *     gt_sph, gt_pts [N, M, 3]   the same for GT with d > 1e-2, and the GT point     counts[3*N + s]
 *   counts [4, N] int64.  One block per segment.
 *
 * vidar_eval_ray_errors: nn_idx [N, Mg] = nearest pred_sph of every gt_sph (vidar_nn_forward);
 *   cham_fwd [N, Mp] / cham_bwd [N, Mg] = squared NN distances pred_in -> gt_in and gt_in -> pred_in
 *   (both NULL: Chamfer column 0).  pred_dhat is read with row stride Mp, gt_pts / nn_idx with Mg.
 *   out [N, 4] fp64 = (chamfer-inner, l1, absrel, count of GT rays with d > 1e-2); count is -1 where
 *   a clamped ray is degenerate (the reference raises RuntimeError) and -2 where a ray that meets the
 *   eval box cannot be clamped into it (the reference's assert(touches_volume)).  Deterministic: one
 *   block per segment, fixed-order fp64 sums, no atomics.
 * ---------------------------------------------------------------------------------- */
int vidar_eval_gather(const float* origin, const float* points, const float* tindex, const float* gt_dist,
                      const float* pred_dist, const float* pc_range_host, int within_grid, float* pred_in,
                      float* gt_in, float* pred_sph, float* pred_dhat, float* gt_sph, float* gt_pts,
                      int64_t* counts, int bs, int M, int F, void* stream);

int vidar_eval_ray_errors(const float* origin, const float* pred_dhat, const float* gt_pts,
                          const int64_t* nn_idx, const float* cham_fwd, const float* cham_bwd,
                          const int64_t* counts, double* out, int N, int Mp, int Mg, void* stream);

/* ------------------------------------------------------------------------------------
 * (v) ego motion (csrc/ego.cu)
 *
 * vidar_bev_rotate_forward: the previous BEV rotated like PerceptionTransformer.get_bev_features
 *   (bevformer/modules/transformer.py:136-149): torchvision.transforms.functional.rotate(img[C,H,W],
 *   angle, center) with nearest sampling, expand=False and zero fill, per sample.
 *   src, dst [bs, H*W, C] channel-last (must not alias); theta_host [bs, 3, 2] host floats = the
 *   rescaled affine matrix θᵀ / [W/2, H/2] of torchvision's _gen_affine_grid (rows x, y, 1).
 *   One warp per output cell; forward only.
 *
 * vidar_ego_align_points: ViDARHeadV1._get_reference_gt_points (dense_heads/vidar_head_v1.py:94-148)
 *   without its masks.  points [N, 4] (x, y, z, frame) packed over the batch, offsets_host [bs + 1]
 *   (N = offsets_host[bs]); slot_of_frame_host [num_frames] = the slot s of frame f, or -1;
 *   src_to_tgt_host [bs, S, 4, 4] host floats (row-vector convention p' = p @ M).
 *   out_points [N, 4] = ([x y z 1] @ M[b, s], s) for points of a frame with a slot, else
 *   (NaN, NaN, NaN, -1), in input order; origins [bs, S, 3] = [0 0 0 1] @ M[b, s].
 *   One thread per point; points and out_points may be NULL when N == 0.
 * ---------------------------------------------------------------------------------- */
int vidar_bev_rotate_forward(const float* src, const float* theta_host, float* dst, int bs, int H, int W, int C,
                             void* stream);

int vidar_ego_align_points(const float* points, const int64_t* offsets_host, const int32_t* slot_of_frame_host,
                           int num_frames, const float* src_to_tgt_host, float* out_points, float* origins, int bs,
                           int S, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VIDAR_B200_H_ */
