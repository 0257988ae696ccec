/*
 * presight_b200 — C-ABI of the B200-native NeRF inner loop (libpresight_b200.so).
 *
 * Drop-in boundary for the reference's `implementation` switch: where the reference calls
 * `self.tcnn_encoding(x)` (field_components/encodings.py:386-389, mlp.py:176-179) or the torch
 * fallbacks, a binding calls these entry points instead.  All paths below are relative to
 * /root/reference/nerfstudio-0.3.3/nerfstudio.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - buffers are allocated and owned by the caller (torch); kernels never allocate;
 *   - gradients of parameters are ACCUMULATED into caller-zeroed fp32 buffers;
 *   - `stream` is a cudaStream_t passed as void*; launches are stream-ordered and re-entrant;
 *   - return value: 0 = ok, non-zero = error (message: ps_last_error(), thread-local);
 *   - nothing throws across the ABI, no torch types in any signature.
 */
#ifndef PRESIGHT_B200_H
#define PRESIGHT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PS_MAX_LEVELS 32
#define PS_MAX_MLP_LAYERS 6
#define PS_MAX_FIELDS 32

/* activation codes for MLP outputs */
#define PS_ACT_NONE 0
#define PS_ACT_RELU 1
#define PS_ACT_SIGMOID 2

const char* ps_last_error(void);
int ps_abi_version(void);
/* number of kernels launched by this library in the calling process (for bench `gpu_launches`) */
int64_t ps_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * Kernel #1 — multiresolution hash encoding.
 * Replaces HashEncoding.pytorch_fwd (+ its autograd), field_components/encodings.py:343-384;
 * hash of encodings.py:324-341 evaluated in uint32 wrap-around arithmetic (bit-exact for T=2^k).
 *   x01      [P,3]   fp32 positions (normally in [0,1]; any value is hashed like the reference)
 *   table    [L*T,F] fp32, T = 1<<log2_T, F in {1,2,4,8}
 *   scalings_host[L] fp32 per-level scales (encodings.py:282-284), HOST pointer
 *   out      [P,L*F] fp32, level-major channels (encodings.py:384)
 */
int ps_hash_fwd(const float* x01, int64_t P, const float* table, const float* scalings_host, int L, int F,
                int log2_T, float* out, void* stream);
/* dtable [L*T,F] += scatter of dout [P,L*F];  dx [P,3] (nullable, caller-zeroed) += d/dx01.  */
int ps_hash_bwd(const float* x01, int64_t P, const float* table, const float* scalings_host, int L, int F,
                int log2_T, const float* dout, float* dtable, float* dx, void* stream);
/* Same kernels with the features / feature gradients stored level-major, [L][P][F] instead of [P][L*F]: every level's
 * F-vector of consecutive points is contiguous, so the per-level passes read and write full sectors.  Used by the
 * level-fused path together with ps_row_segment.feat_per_level. */
int ps_hash_fwd_lm(const float* x01, int64_t P, const float* table, const float* scalings_host, int L, int F,
                   int log2_T, float* out, void* stream);
int ps_hash_bwd_lm(const float* x01, int64_t P, const float* table, const float* scalings_host, int L, int F,
                   int log2_T, const float* dout, float* dtable, float* dx, void* stream);
/* Levels handled per thread for this grid shape (level groups are chosen so that the live tables stay L2-resident). */
int ps_hash_levels_per_thread(int L, int F, int log2_T);
/* Parity probe: the 8 corner rows (incl. level*T) in the reference's corner order h0..h7
 * (encodings.py:354-361) and the fractional offsets.  idx [P,L,8] int64, offset [P,L,3] fp32 (nullable). */
int ps_hash_indices(const float* x01, int64_t P, const float* scalings_host, int L, int log2_T, int64_t* idx,
                    float* offset, void* stream);

/* ---------------------------------------------------------------------------------------
 * Position prologue: aabb normalisation, L-inf scene contraction, selector.
 * Replaces fields/PreSight/utils.py:6-10, field_components/spatial_distortions.py:66-69 (order=inf),
 * fields/PreSight/ingp_field.py:169-177 (= prop_density_field.py:130-138).
 *   pos [P,3] world -> x01 [P,3] (masked points moved to the origin), selector [P] uint8
 *   aabb_host[6] = {min xyz, max xyz}; contract!=0 applies the contraction, else plain SceneBox normalisation.
 */
int ps_normalize_positions(const float* pos, int64_t P, const float* aabb_host, int contract, float* x01,
                           uint8_t* selector, void* stream);
/* Frustums.get_positions (cameras/rays.py:49-58): pos[n,s,:] = o[n] + d[n]*(bins[n,s]+bins[n,s+1])/2 */
int ps_sample_positions(const float* origins, const float* dirs, const float* eu_bins, int64_t N, int S,
                        float* pos, void* stream);
/* ps_sample_positions + ps_normalize_positions in one pass: bin edges -> unit-cube sample positions + selector. */
int ps_ray_points(const float* origins, const float* dirs, const float* eu_bins, int64_t N, int S,
                  const float* aabb_host, int contract, float* x01, uint8_t* selector, void* stream);
/* SHEncoding(levels=4).pytorch_fwd on (d+1)/2 (utils/math.py:27-74, fields/base_field.py:136-142).
 * dirs [P,3]; mapped == 0: raw directions (the kernel applies (d+1)/2), mapped != 0: already (d+1)/2; out [P,16]. */
int ps_sh4(const float* dirs, int64_t P, int mapped, float* out, void* stream);
/* nearest-centroid routing (fields/PreSight/ingp_field_ms.py:97): assign[p] = argmin_j |pos_p - c_j| */
int ps_nearest_centroid(const float* pos, int64_t P, const float* centroids, int nf, int32_t* assign, void* stream);

/* Prior query epilogue (scripts/extract_priors.py:137-138): mean[i] = (1/k) sum_j densities_host[j][i];
 * feats_half[i,c] = half(clip(sem[i,c], 0, 1)).  densities_host: HOST array of k device pointers (k <= 8). */
int ps_prior_finalize(const float* const* densities_host, int k, const float* sem, int64_t M, int C, float* mean,
                      void* feats_half, void* stream);

/* ---------------------------------------------------------------------------------------
 * Kernel #2 — fused MLP (Linear+ReLU stack, optional output activation).
 * Replaces MLP.pytorch_fwd (field_components/mlp.py:157-174) and its autograd.
 *   x [P,dims[0]] -> y [P,dims[n_layers]];  W_host[i] -> device fp32 [dims[i+1], dims[i]] (nn.Linear layout),
 *   b_host[i] -> device fp32 [dims[i+1]].  W_host/b_host/dims_host are HOST arrays.
 *   Hidden activations are never written to HBM; backward recomputes them.
 *   precision: 0 = error-compensated 3xTF32 tensor-core MMA, fp32-grade (1e-3 parity class),
 *              1 = bf16 tensor-core MMA with fp32 accumulate (1e-2 parity class).
 *   Supported shapes (padded to multiples of 16) are listed in csrc/mlp_dispatch.cuh; others return status 3.
 */
int ps_mlp_fwd(const float* x, int64_t P, const float* const* W_host, const float* const* b_host,
               const int* dims_host, int n_layers, int out_act, int precision, float* y, void* stream);
/* dx [P,dims[0]] (nullable) written; dW_host[i]/db_host[i] device buffers accumulated. y = forward output
 * (needed for the sigmoid derivative; nullable when out_act == PS_ACT_NONE). */
int ps_mlp_bwd(const float* x, const float* y, const float* dy, int64_t P, const float* const* W_host,
               const float* const* b_host, const int* dims_host, int n_layers, int out_act, int precision,
               float* dx, float* const* dW_host, float* const* db_host, void* stream);
/* Segmented variant: the logical input row of point r is the concatenation of up to PS_MLP_MAX_SEGMENTS column
 * segments (replaces the torch.cat / torch.split copies of ingp_field.py:186, 204-228): segment s supplies `width`
 * columns from src[(r / group) * stride + col0 + c].  group > 1 = a per-ray vector shared by `group` consecutive
 * points (view direction SH, appearance embedding).  On backward `dst` (nullable) receives the input gradient with the
 * same addressing; for group > 1 the group's gradients are summed into dst (dst zero-filled by the caller).
 * Density epilogue (ingp_field.py:187-190, prop_density_field.py:148-152): if density_out != NULL,
 * density_out[r] = exp(y[r,0]) * sel[r] (sel nullable = 1); y may then be NULL.  On backward, d_density (nullable)
 * replaces the gradient of column 0 by d_density[r]*sel[r]*exp(clamp(y[r,0],-15,15)) (activations.py:38-41); dy nullable. */
#define PS_MLP_MAX_SEGMENTS 3
typedef struct {
    const float* src;
    float* dst;
    int64_t stride;
    int col0, width, group;
    int feat_per_level; /* 0: rows are contiguous (src[r*stride + col0 + c]).  F > 0 (single-segment inputs only): the
                           columns are hash features stored level-major [L][P][F], element (r, c) at
                           src[((c / F) * P + r) * F + c % F] — the layout of ps_hash_fwd_lm / ps_hash_bwd_lm. */
} ps_row_segment;
int ps_mlp_fwd_ex(const ps_row_segment* segs_host, int n_seg, int64_t P, const float* const* W_host,
                  const float* const* b_host, const int* dims_host, int n_layers, int out_act, int precision, float* y,
                  const uint8_t* sel, float* density_out, void* stream);
int ps_mlp_bwd_ex(const ps_row_segment* segs_host, int n_seg, const float* dy, int64_t P, const float* const* W_host,
                  const float* const* b_host, const int* dims_host, int n_layers, int out_act, int precision,
                  float* const* dW_host, float* const* db_host, const uint8_t* sel, const float* d_density, void* stream);
/* trunc_exp (field_components/activations.py:28-41) fused with the selector multiply
 * (ingp_field.py:189-190): y = exp(x)*sel ; dx = dy*sel*exp(clamp(x,-15,15)). sel nullable. */
int ps_trunc_exp_fwd(const float* x, const uint8_t* sel, int64_t P, int64_t x_stride, float* y, void* stream);
int ps_trunc_exp_bwd(const float* x, const uint8_t* sel, const float* dy, int64_t P, int64_t x_stride,
                     float* dx, int64_t dx_stride, void* stream);

/* ---------------------------------------------------------------------------------------
 * Kernel #3 — samplers.
 * ps_spaced_bins replaces SpacedSampler.generate_ray_samples (model_components/ray_samplers.py:98-128)
 * with PreSight's piecewise spacing (models/PreSight/nerfacto_nusc_ms.py:312-317).
 *   lin_bins [S+1] = torch.linspace(0,1,S+1) (device);  t_rand [N] single jitter, NULL in eval
 *   -> sp_bins [N,S+1] in [0,1], eu_bins [N,S+1] euclidean
 */
int ps_spaced_bins(const float* nears, const float* fars, const float* lin_bins, const float* t_rand, int64_t N,
                   int S, float thr, float* sp_bins, float* eu_bins, void* stream);
/* ps_pdf_resample replaces PDFSampler.generate_ray_samples (ray_samplers.py:305-362, include_original=False)
 * including the annealing pow of ProposalNetworkSampler (ray_samplers.py:597).
 *   weights [N,S_in]; sp_in [N,S_in+1]; u_base [S_out+1] = linspace(0,1-1/nb,nb) (device);
 *   rand [N] single jitter (train) or NULL (eval: u = u_base + 1/(2 nb));
 *   -> sp_out/eu_out [N,S_out+1]; optional probes inds [N,S_out+1] int64, cdf [N,S_in+1] fp32, u [N,S_out+1].
 *   S_in <= 1024.
 */
int ps_pdf_resample(const float* weights, const float* sp_in, const float* u_base, const float* rand,
                    const float* nears, const float* fars, int64_t N, int S_in, int S_out, float padding, float eps,
                    float anneal, float thr, float* sp_out, float* eu_out, int64_t* inds, float* cdf, float* u,
                    void* stream);
/* searchsorted(cdf, u, side="right") alone — the bit-exact bin-index probe (ray_samplers.py:345). */
int ps_searchsorted_right(const float* cdf, const float* u, int64_t N, int n_cdf, int n_u, int64_t* inds,
                          void* stream);

/* ---------------------------------------------------------------------------------------
 * Kernel #4 — volumetric compositing.
 * ps_weights_* replace RaySamples.get_weights (cameras/rays.py:128-150) and its autograd.
 *   deltas, density [N,S] -> weights [N,S].   S <= 1024.
 */
int ps_weights_fwd(const float* deltas, const float* density, int64_t N, int S, float* weights, void* stream);
int ps_weights_bwd(const float* deltas, const float* density, const float* dweights, int64_t N, int S,
                   float* ddensity, void* stream);
/* Weighted sum along the ray: out[n,c] = sum_s w[n,s] * v[n,s,c]  (v NULL => v=1, C=1).
 * Replaces RGBRenderer.combine_rgb (model_components/renderers.py:102-103), AccumulationRenderer
 * (:313), the numerator of DepthRenderer "expected" (:377) and the semantics sum
 * (models/PreSight/nerfacto_nusc_ms.py:530). */
int ps_render_fwd(const float* weights, const float* values, int64_t N, int S, int C, float* out, void* stream);
/* dweights [N,S] ACCUMULATED (+=), dvalues [N,S,C] written (nullable). */
int ps_render_bwd(const float* weights, const float* values, const float* dout, int64_t N, int S, int C,
                  float* dweights, float* dvalues, void* stream);
/* DepthRenderer "threshold" (renderers.py:352-362): first sample with cumsum(w) >= thr. */
int ps_depth_threshold(const float* weights, const float* eu_bins, int64_t N, int S, float threshold,
                       float* depth, int64_t* index, void* stream);
/* One-pass compositing used by the model fast path (nerfacto_nusc_ms.py:503-544):
 *   in : eu_bins [N,S+1], density [N,S], rgb [N,S,3] (nullable), sem [N,S,C] (nullable, C<=128)
 *   out: weights [N,S], rgb_out [N,3], acc [N] (unclamped), depth_exp [N] = sum w t/(sum w+1e-10) (unclipped),
 *        depth_thr [N], sem_out [N,C], tminmax [2] (global min/max of mid-points, caller-initialised +inf/-inf)
 */
int ps_composite_fwd(const float* eu_bins, const float* density, const float* rgb, const float* sem, int64_t N,
                     int S, int C, float threshold, float* weights, float* rgb_out, float* acc, float* depth_exp,
                     float* depth_thr, float* sem_out, float* tminmax, void* stream);
/* grads: d_weights_in [N,S] (nullable; direct seeds on the weights), d_rgb_out [N,3], d_acc [N], d_depth_exp [N],
 *        d_sem_out [N,C] (each nullable) -> d_density [N,S], d_rgb [N,S,3], d_sem [N,S,C] (nullable if input null) */
int ps_composite_bwd(const float* eu_bins, const float* density, const float* rgb, const float* sem,
                     const float* weights, const float* acc, const float* depth_exp, int64_t N, int S, int C,
                     const float* d_weights_in, const float* d_rgb_out, const float* d_acc, const float* d_depth_exp,
                     const float* d_sem_out, float* d_density, float* d_rgb, float* d_sem, void* stream);

/* ---------------------------------------------------------------------------------------
 * Loss stack (SURVEY 8f-1): proposal / interlevel loss of mip-NeRF 360 as one kernel.
 * Replaces outer + lossfun_outer + the per-level body of interlevel_loss (model_components/losses.py:48-126).
 *   c [N,S+1], w [N,S]        final level's spacing-domain bin edges and weights (treated as constants)
 *   t_env [N,Sp+1], w_env [N,Sp]  proposal level's bin edges and weights
 *   loss_sum [1]  += sum over rays and samples of max(w - w_outer, 0)^2 / (w + 1e-7)   (caller-zeroed)
 *   grad_w_env [N,Sp] (nullable) = d loss_sum / d w_env (written, not accumulated).  Sp <= 2048.
 */
int ps_interlevel_loss(const float* c, const float* w, const float* t_env, const float* w_env, int64_t N, int S,
                       int Sp, float* loss_sum, float* grad_w_env, void* stream);
/* z-anti-aliased (zip-NeRF) interlevel loss — the reference's DEFAULT proposal loss (enable_z_anti_aliasing,
 * models/PreSight/nerfacto_nusc_ms.py:129,293-295): blur_stepfun + sorted_interp_quad + the per-level body of
 * z_anti_anliasing_interlevel_loss (model_components/PreSight/losses.py:127-206), one launch per proposal level.
 *   c [N,S+1], w [N,S]            final level's spacing-domain bin edges and weights (constants), S <= 128
 *   t_env [N,Sp+1], w_env [N,Sp]  proposal level's bin edges and weights;  pulse_width = config.pulse_width[level]
 *   loss_sum [1] += sum over rays and proposal samples of max(w_s - w_env, 0)^2 / (w_env + 1e-5)  (caller-zeroed; the
 *   reference's value is loss_sum / (N * Sp));  grad_w_env [N,Sp] (nullable) = d loss_sum / d w_env (written). */
int ps_zaa_interlevel_loss(const float* c, const float* w, int64_t N, int S, const float* t_env, const float* w_env,
                           int Sp, double pulse_width, float* loss_sum, float* grad_w_env, void* stream);
/* Distortion loss of mip-NeRF 360 (lossfun_distortion / distortion_loss, model_components/losses.py:130-149).
 *   c [N,S+1] spacing-domain bin edges and w [N,S] weights of the final level
 *   loss_sum [1] += sum over rays of (sum_ij w_i w_j |u_i - u_j| + sum_i w_i^2 (c_{i+1} - c_i) / 3), u = bin mid-points
 *   (caller-zeroed; the reference's value is loss_sum / N);  grad_w [N,S] (nullable) = d loss_sum / d w (written).
 *   S <= 1024. */
int ps_distortion_loss(const float* c, const float* w, int64_t N, int S, float* loss_sum, float* grad_w, void* stream);

/* ---------------------------------------------------------------------------------------
 * Loss stack (SURVEY 8f-1), per-ray tail of the step: model epilogue and rendered-output loss terms, one kernel each.
 *
 * ps_sky_blend_fwd replaces models/PreSight/nerfacto_nusc_ms.py:512-532:
 *   acc = clamp(acc_raw, 0, 1); rgb = [clamp01 if clamp_rgb](rgb_f) + (1 - acc) * sky_rgb; sem = sem_f + (1 - acc) * sky_sem
 *   rgb_f [N,3], acc_raw [N], sem_f [N,C] (nullable with sem), sky_rgb [N,3] / sky_sem [N,C] nullable (no blending).
 * ps_sky_blend_bwd: upstream d_rgb [N,3] / d_acc [N] / d_sem [N,C] (each nullable = zero) ->
 *   d_acc_raw [N] (written), d_sky_rgb [N,3], d_sky_sem [N,C] (written, nullable), d_rgb_f [N,3] (nullable: only needed
 *   when clamp_rgb, otherwise it equals d_rgb; d_sem_f always equals d_sem).
 * ps_render_losses replaces nn.MSELoss (nerfacto_nusc_ms.py:314,560-567), sky_loss and semantic_loss
 *   (model_components/PreSight/losses.py:106-125): losses[3] += {mean (rgb-gt)^2, mean BCE(clip(acc,eps,1-eps), 1-sky),
 *   mean (sem - clip(gt_sem,0,1))^2} (caller-zeroed; a term whose inputs are NULL is skipped) and
 *   g_rgb [N,3], g_acc [N], g_sem [N,C] = d losses[i] / d input (written, nullable). */
int ps_sky_blend_fwd(const float* rgb_f, const float* acc_raw, const float* sem_f, const float* sky_rgb,
                     const float* sky_sem, int64_t N, int C, int clamp_rgb, float* rgb, float* acc, float* sem,
                     void* stream);
int ps_sky_blend_bwd(const float* rgb_f, const float* acc_raw, const float* sky_rgb, const float* sky_sem,
                     const float* d_rgb, const float* d_acc, const float* d_sem, int64_t N, int C, int clamp_rgb,
                     float* d_rgb_f, float* d_acc_raw, float* d_sky_rgb, float* d_sky_sem, void* stream);
int ps_render_losses(const float* rgb, const float* gt_rgb, const float* acc, const float* sky_mask, const float* sem,
                     const float* gt_sem, int64_t N, int C, float eps, float* losses, float* g_rgb, float* g_acc,
                     float* g_sem, void* stream);

/* ---------------------------------------------------------------------------------------
 * Loss stack (SURVEY 8f-1), depth supervision: expected-depth loss + line-of-sight loss, loss sums and gradients in one
 * kernel.  Replaces model_components/PreSight/losses.py:24-103 (normalize_depth, line_of_sight_loss,
 * expected_depth_loss, expected_monodepth_loss) as called from models/PreSight/nerfacto_nusc_ms.py:577-629.
 *   weights [N,S] final-level weights (nullable: no line-of-sight term); sample mid-points in metres either given as
 *   steps_m [N,S] or derived as (eu_bins[s] + eu_bins[s+1]) / 2 / pose_scale from eu_bins [N,S+1] (exactly one of the
 *   two); expected_depth [N] rendered expected depth in scene units (nullable: no expected-depth term), divided by
 *   pose_scale inside; target_depth_m [N] metres; sky_mask [N] (1 = sky; nullable = the LiDAR variants);
 *   pose_scale_dev (nullable): one device float that overrides pose_scale — the reference keeps the factor as a tensor
 *   element (ray_samples.metadata["pose_scale_factor"][0,0,0]); reading it on the device avoids a host sync per step;
 *   mode 0 = depths mapped by clip(d / upper_bound, 0, 1), 1 = by 1 / (d + 5) (monodepth_loss_inverse).
 *   sums[3] += {#rays with 1 < target < upper_bound [and sky == 0], sum of squared errors, sum of line-of-sight terms}
 *   over those rays (caller-zeroed); g_expected [N] = d sums[1] / d expected_depth, g_weights [N,S] = d sums[2] / d weights
 *   (written, nullable).  The reference's means are sums[1] / sums[0] and sums[2] / sums[0]. */
int ps_depth_losses(const float* weights, const float* eu_bins, const float* steps_m, const float* expected_depth,
                    const float* target_depth_m, const float* sky_mask, int64_t N, int S, float pose_scale,
                    const float* pose_scale_dev, float sigma, float upper_bound, int mode, float* sums, float* g_expected,
                    float* g_weights, void* stream);

/* ---------------------------------------------------------------------------------------
 * Prior post-processing (SURVEY 8f-4): voxel down-sampling of extracted hit points with per-voxel means, on the GPU.
 * Replaces scripts/extract_priors.py:156-165 (density > 1 filter), :216-245 (open3d voxel_down_sample_and_trace with
 * bounds min - 1 / max + 1) and :175-191 (per-voxel hit count, colour mean, fp64 feature mean -> fp16, hit quantile).
 *
 * ps_voxel_min_bound: min_out[3] (caller-preset to +inf) = per-axis min over the points with densities > 1
 *   (densities nullable = all points).  points [N,3] fp32 metres.
 * ps_voxel_accumulate: adds the selected points to an open-addressing hash table keyed by open3d's voxel index
 *   floor((p - ((min - 1) - voxel/2)) / voxel) (double arithmetic; min_point [3] on the device, as written by
 *   ps_voxel_min_bound): keys [capacity] int64 preset to -1, counts [capacity] u32, sum_xyz / sum_col [capacity,3] and
 *   sum_feat [capacity,C] fp64, all caller-zeroed; capacity a power of two.  features_f16 [N,C] / colors [N,3] nullable
 *   together with their accumulators.  May be called repeatedly (streaming) with the same min_point.
 *   status |= 1 table full, |= 2 voxel index outside 21 bits per axis (checked by the caller after a sync).
 * ps_voxel_finalize: occupied slots -> rows 0..*n_out-1 (caller-zeroed counter; row order arbitrary): out_keys (packed
 *   ix<<42 | iy<<21 | iz), out_xyz [.,3] = centre of mass, out_col [.,3], out_feat_f16 [.,C], out_hits.
 * ps_hits_quantile: out[0] = np.quantile(hits[0..M), q) (linear interpolation); hist [bins] u32 caller-zeroed scratch,
 *   bins > max(hits) (status |= 4 otherwise). */
int ps_voxel_min_bound(const float* points, const float* densities, int64_t N, float* min_out, void* stream);
int ps_voxel_accumulate(const float* points, const void* features_f16, const float* colors, const float* densities,
                        int64_t N, int C, const float* min_point, double voxel_size, int64_t* keys, int64_t capacity,
                        uint32_t* counts, double* sum_xyz, double* sum_col, double* sum_feat, int* status, void* stream);
int ps_voxel_finalize(const int64_t* keys, int64_t capacity, const uint32_t* counts, const double* sum_xyz,
                      const double* sum_col, const double* sum_feat, int C, uint64_t* n_out, int64_t* out_keys,
                      float* out_xyz, float* out_col, void* out_feat_f16, int64_t* out_hits, void* stream);
int ps_hits_quantile(const int64_t* hits, int64_t M, double q, uint32_t* hist, int64_t bins, double* out, int* status,
                     void* stream);

/* The tile voxelizer: the per-voxel means of ps_voxel_accumulate / ps_voxel_finalize in memory that follows the number of
 * voxels V, not of points.  Two passes over the points, with the same voxel key as ps_voxel_accumulate:
 * ps_voxel_insert: pass 1, keys only.  Inserts the key of every point into keys [capacity] int64 (preset to -1, capacity
 *   a power of two; the caller keeps capacity >= 2 * (V + N)) and adds the number of new voxels to *n_voxels.
 * ps_voxel_rehash: moves the occupied keys of old_keys [old_capacity] into keys [capacity] (preset to -1, capacity >=
 *   old_capacity, both powers of two).
 * ps_voxel_assign_rows: rows[slot of sorted_keys[r]] = r for r < V (sorted_keys: the occupied keys in ascending order;
 *   rows [capacity] int32 beside the table).
 * ps_voxel_accumulate_rows: pass 2.  Looks each point's row up (no insertion) and adds the point to the dense rows:
 *   counts [V] u32, sum_xyz / sum_col [V,3] and sum_feat [V,C] fp64, caller-zeroed.  features_f16 [N,C] / colors [N,3]
 *   nullable together with their sums.
 * ps_voxel_finalize_rows: row r's means -> out_xyz [V,3], out_col [V,3], out_feat_f16 [V,C], out_hits [V], as
 *   ps_voxel_finalize writes them; the rows stay in ascending key order.
 * status: |= 1 table full, |= 2 voxel index outside 21 bits per axis, |= 4 a point's voxel is not in the table (checked by
 *   the caller after a sync).  No kernel allocates. */
int ps_voxel_insert(const float* points, int64_t N, const float* min_point, double voxel_size, int64_t* keys,
                    int64_t capacity, uint64_t* n_voxels, int* status, void* stream);
int ps_voxel_rehash(const int64_t* old_keys, int64_t old_capacity, int64_t* keys, int64_t capacity, int* status,
                    void* stream);
int ps_voxel_assign_rows(const int64_t* sorted_keys, int64_t V, const int64_t* keys, int64_t capacity, int32_t* rows,
                         int* status, void* stream);
int ps_voxel_accumulate_rows(const float* points, const void* features_f16, const float* colors, int64_t N, int C,
                             const float* min_point, double voxel_size, const int64_t* keys, const int32_t* rows,
                             int64_t capacity, uint32_t* counts, double* sum_xyz, double* sum_col, double* sum_feat,
                             int* status, void* stream);
int ps_voxel_finalize_rows(const uint32_t* counts, const double* sum_xyz, const double* sum_col, const double* sum_feat,
                           int64_t V, int C, float* out_xyz, float* out_col, void* out_feat_f16, int64_t* out_hits,
                           void* stream);

/* ---------------------------------------------------------------------------------------
 * Ray generation (SURVEY 8f-3): RayGenerator.forward + Cameras.generate_rays for PERSPECTIVE cameras without distortion
 * (model_components/ray_generators.py:43-61, cameras/cameras.py:497-880).
 *   c2w [C,3,4], fx / fy / cx / cy [C] fp32; ray_indices [N,3] int64 = (camera, row, col); pixel_offset = 0.5
 *   -> origins [N,3], directions [N,3] (unit), pixel_area [N], directions_norm [N] (nullable). */
int ps_generate_rays(const float* c2w, const float* fx, const float* fy, const float* cx, const float* cy, int C,
                     const int64_t* ray_indices, int64_t N, float pixel_offset, float* origins, float* directions,
                     float* pixel_area, float* directions_norm, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused Adam step (SURVEY 8f-2): torch.optim.Adam without amsgrad as PreSight configures it
 * (configs/method_configs.py:115: lr 1e-2, eps 1e-15, weight_decay 1e-5; engine/optimizers.py:133-140), one pass.
 *   param / exp_avg / exp_avg_sq [n] fp32 updated in place, grad [n] read; step = 1 for the first update;
 *   16-byte aligned buffers take the float4 path, anything else an element-wise one; hyper-parameters as doubles (torch keeps them as Python floats and derives the
 *   bias corrections in double precision). */
int ps_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr, double beta1,
                 double beta2, double eps, double weight_decay, int64_t step, void* stream);

/* Self-test of the tcgen05 operand conventions used by the fused kernels (csrc/tc5.cuh): one CTA computes, from
 * X [128,64], Y [128,64], W [64,64] (fp32, rounded to bf16 on chip), C1 = X W^T (K-major operands), C2 = X W
 * (MN-major B: the input-gradient form) and C3 = 2 X^T Y (MN-major A and B, reduction over rows, accumulated over two
 * calls: the weight-gradient form; rows 64..127 of C3 are padding), all [128,64] fp32, and C4 [128,16] whose column 3
 * holds the column sums of X (bias-gradient form: one-hot B operand with a zero K stride). */
int ps_tc5_probe(const float* X, const float* Y, const float* W, float* C1, float* C2, float* C3, float* C4,
                 void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused field level on tcgen05 tensor cores (bf16 parity class).  One kernel evaluates, per 128-point tile,
 * iNGPField.get_density/get_outputs/semantic head (fields/PreSight/ingp_field.py:163-267) and the compositing of
 * nerfacto_nusc_ms.py:497-530 (weights, rgb, accumulation, expected / threshold depth, semantics); the backward
 * kernel recomputes the forward on chip and produces the hash-feature gradient, the appearance gradient and all
 * weight / bias gradients.  Only the architecture of the reference's field is supported: hidden width 64,
 * geo_feat_dim 15, semantic width 64, 3-layer heads, appearance dim <= 16, L*F <= 48 with F in {2,4},
 * samples per ray S in {32,64,96,128}.  Layer order in W/B/dW/dB: base0 [64,L*F], base1 [80,64], sem0..2 [64,64],
 * rgb0 [64,31+A], rgb1 [64,64], rgb2 [3,64] (nn.Linear layout, fp32, device pointers).
 */
typedef struct {
    const float* W[8];
    const float* B[8];
    float* dW[8]; /* backward only: accumulated into caller-zeroed buffers */
    float* dB[8];
    int app_dim;
} ps_field_net;
/* feat_lm: level-major hash features [L][P][F] (ps_hash_fwd_lm), sel [P] (nullable), eu_bins [N,S+1], dirs [N,3],
 * app [N,A] -> weights [N,S], rgb_out [N,3], acc [N] (unclamped), depth_exp [N] (unclipped), depth_thr [N],
 * sem_out [N,64], tminmax [2] (nullable; caller-initialised +inf/-inf). */
int ps_field_level_fwd(const ps_field_net* net, const float* feat_lm, int L, int F, const uint8_t* sel,
                       const float* eu_bins, const float* dirs, const float* app, int64_t N, int S, float threshold,
                       float* weights, float* rgb_out, float* acc, float* depth_exp, float* depth_thr, float* sem_out,
                       float* tminmax, void* stream);

/* Backward of ps_field_level_fwd (recomputes the forward on chip).  acc / depth_exp: the forward's outputs (needed only
 * with d_depth_exp).  Upstream gradients (each nullable): d_weights [N,S], d_rgb_out [N,3], d_acc [N], d_depth_exp [N],
 * d_sem_out [N,64].  Outputs: dfeat_lm [L][P][F] written; dapp [N,A] (nullable) and net->dW / net->dB accumulated into
 * caller-zeroed buffers. */
int ps_field_level_bwd(const ps_field_net* net, const float* feat_lm, int L, int F, const uint8_t* sel,
                       const float* eu_bins, const float* dirs, const float* app, int64_t N, int S, const float* acc,
                       const float* depth_exp, const float* d_weights, const float* d_rgb_out, const float* d_acc,
                       const float* d_depth_exp, const float* d_sem_out, float* dfeat_lm, float* dapp, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused proposal level (bf16 parity class).  One forward kernel replaces, per proposal level of
 * ProposalNetworkSampler.generate_ray_samples (model_components/ray_samplers.py:600-609),
 * Frustums.get_positions + PropNetDensityField.density_fn (fields/PreSight/prop_density_field.py:129-153: contraction,
 * selector, hash encoding, 2-layer MLP, trunc_exp) + RaySamples.get_weights (cameras/rays.py:128-150); one backward
 * kernel produces the hash-table and MLP gradients from d_weights.  Supported: 2-layer MLP with hidden width 16 or 64,
 * L*F <= 16 with F in {1,2}, S in {32,64,96,128}.
 */
typedef struct {
    const float* W0; /* [hidden, L*F] */
    const float* b0; /* [hidden] */
    const float* W1; /* [1, hidden] */
    const float* b1; /* [1] */
    float* dW0;      /* backward only: accumulated into caller-zeroed buffers */
    float* db0;
    float* dW1;
    float* db1;
    int hidden;
} ps_prop_net;
/* row stride (in bf16 elements) of the feature buffer exchanged between the two kernels: 8 or 16 */
int ps_prop_level_feat_stride(int L, int F);
/* origins/dirs [N,3], eu_bins [N,S+1], aabb_host[6], table [L*T,F] -> weights [N,S]; feat_bf16 (nullable)
 * [N*S, stride] bf16 hash features saved for the backward. */
int ps_prop_level_fwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins, int64_t N,
                      int S, const float* aabb_host, int contract, const float* table, const float* scalings_host,
                      int L, int F, int log2_T, float* weights, void* feat_bf16, void* stream);
/* d_weights [N,S] -> dtable [L*T,F] and net->dW0/db0/dW1/db1, all accumulated. */
int ps_prop_level_bwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins, int64_t N,
                      int S, const float* aabb_host, int contract, const float* scalings_host, int L, int F, int log2_T,
                      const void* feat_bf16, const float* d_weights, float* dtable, void* stream);

/* ---------------------------------------------------------------------------------------
 * Density level of the main field, forward only (bf16 parity class): the same kernels as the fused proposal level,
 * instantiated for the density head of iNGPField (fields/PreSight/ingp_field.py:168-191): base0 [64, L*F] + ReLU, then
 * row 0 of base1 [80, 64] plus base1.bias[0], trunc_exp, selector.  Pass net->W1 = &base1.weight[0][0] and
 * net->b1 = &base1.bias[0]; the backward members are ignored.  Supported: hidden 64, L*F <= 48 with F in {1,2,4},
 * S in {32,64,96,128} (ray mode).  Used to find the threshold depth of eval rays (prior extraction).
 *   ps_density_level_fwd     origins/dirs [N,3], eu_bins [N,S+1] -> weights [N,S], exactly as ps_prop_level_fwd
 *   ps_density_level_fwd_ms  routed rows (see the sub-field section below) -> density [P] at each point's own index,
 *                            exactly as ps_prop_level_fwd_ms
 */
int ps_density_level_fwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins, int64_t N,
                         int S, const float* aabb_host, int contract, const float* table, const float* scalings_host,
                         int L, int F, int log2_T, float* weights, void* stream);
struct ps_prop_net_dev;
int ps_density_level_fwd_ms(const struct ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted,
                            const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows,
                            const float* const* tables_dev, const float* scalings_host, int L, int F, int log2_T,
                            float* density, void* stream);

/* Surface hits of rays at their threshold depth (scripts/extract_priors.py:100-126), one thread per ray:
 *   points_scaled [N,3] = fmaf(d, depth, o) per component; points_m [N,3] = points_scaled / pose_scale (IEEE division);
 *   keep [N] u8 = depth / pose_scale <= max_range_m && z_min_m <= points_m.z <= z_max_m, a non-finite bound not applied.
 * origins / dirs [N,3], depth [N]; pose_scale > 0. */
int ps_surface_hits(const float* origins, const float* dirs, const float* depth, int64_t N, float pose_scale,
                    float max_range_m, float z_min_m, float z_max_m, float* points_scaled, float* points_m, uint8_t* keep,
                    void* stream);

/* The kept hits of a chunk into the extractor's hit store, in ray order: the rows with keep[i] != 0 && density[i] > 1
 * (extract_priors.py:157) are written to store_points / store_colors [capacity,3] from row *cursor on (colors nullable:
 * zeros are stored), *cursor advances by their number, and the per-axis minimum of their points_m is folded into
 * min_out[3] (preset to +inf, as ps_voxel_min_bound).  When they do not all fit below capacity, nothing is written,
 * *cursor stays and status |= 1.  points_scaled / points_m [N,3], keep [N] u8 and density [N] as ps_surface_hits and
 * query_priors give them.  workspace: device memory of ps_hits_append_workspace(N) bytes.  No host synchronisation. */
int ps_hits_append_workspace(int64_t N, int64_t* bytes);
int ps_hits_append(const float* points_scaled, const float* points_m, const uint8_t* keep, const float* density,
                   const float* colors, int64_t N, float* store_points, float* store_colors, int64_t capacity,
                   int64_t* cursor, float* min_out, int* status, void* workspace, void* stream);

/* Image metrics of rendered images: replace the torchmetrics calls of the reference model's `get_metrics_dict` and
 * `get_image_metrics_and_images` (models/PreSight/nerfacto_nusc_ms.py, as nerfstudio's models/nerfacto.py):
 * `PeakSignalNoiseRatio(data_range=1.0)` and `structural_similarity_index_measure` with its defaults, one image at a time.
 *   pred, gt [B,H,W,3] fp32 channels-last, per image:
 *   sse [B] f64 = sum (pred - gt)^2;  psnr [B] f32 = 10 log10(data_range_psnr^2 / (sse / 3HW)), +inf for equal images
 *   ssim [B] f64: 11-tap Gaussian window (sigma 1.5), data range max(max - min of pred, of gt) over the image, mean over
 *                 channels and the (H-10) x (W-10) windows inside the image (what torchmetrics keeps after its reflect pad
 *                 and crop); NaN for two constant images.  Definitions in presight_b200/csrc/metrics_core.h.
 * ssim == NULL computes sse / psnr only, for any H, W (a ray batch as B = 1, H = 1, W = N); else H, W >= 11 (status 1
 * otherwise).  sse may be NULL.  workspace: device memory of ps_image_metrics_workspace(B, H, W) bytes.  No host
 * synchronisation and no floating-point atomics: repeated calls give bit-identical results. */
int ps_image_metrics_workspace(int B, int H, int W, int64_t* bytes);
int ps_image_metrics(const float* pred, const float* gt, int B, int H, int W, float data_range_psnr, void* workspace,
                     double* sse, float* psnr, double* ssim, void* stream);

/* LPIPS of rendered images, the reference model's third evaluation metric: nerfacto's
 * `LearnedPerceptualImagePatchSimilarity(normalize=True)` (AlexNet, LPIPS v0.1, mean reduction), as torchmetrics
 * functional/image/lpips.py defines it after lpips 0.1 (`pretrained_networks.alexnet`, `normalize_tensor`).  Per pair:
 *   x = (2 x - 1 - shift_c) / scale_c, shift (-0.030, -0.088, -0.188), scale (0.458, 0.448, 0.450);
 *   AlexNet features cut after each ReLU (torchvision features.{0,3,6,8,10}, max-pool 3x3/2 floor before conv 2 and 3);
 *   per layer k: f / (sqrt(sum_c f_c^2) + 1e-10) for both images, d = sum_c lin_k[c] (f0_c - f1_c)^2, mean over pixels;
 *   out [B] f64 = sum of the five means, per_layer [B,5] f64 the means themselves (may be NULL).
 * Convolutions in TF32 (operands rounded to nearest, fp32 accumulation), as cuDNN runs them for torchmetrics under
 * PyTorch's default allow_tf32.  pred, gt [B,H,W,3] fp32 channels-last in [0,1] (not checked); H, W >= 31.
 * net: device pointers packed by presight_b200.metrics.LPIPS: conv_w[k] [C_out][K_pad] fp32 with K = kh kw C_in in
 * (ky, kx, ci) order, zero-padded to K_pad = a multiple of 32 and TF32-rounded (RNA); conv_b[k] [C_out]; lin[k] [C_k],
 * C = 64, 192, 384, 256, 256.  workspace: device memory of ps_lpips_workspace(B, H, W) bytes (about 140 MB per pair at
 * 1600 x 900).  Status 1 for B outside [1, 32767], H or W below 31, sizes whose per-image indices overflow 32 bits, or a
 * null pointer.  No allocation, no host synchronisation and no floating-point atomics: repeated calls are bit-identical,
 * and lpips(x, x) == 0 and lpips(a, b) == lpips(b, a) exactly. */
typedef struct ps_lpips_net {
    const float* conv_w[5];
    const float* conv_b[5];
    const float* lin[5];
} ps_lpips_net;
int ps_lpips_workspace(int B, int H, int W, int64_t* bytes);
int ps_lpips(const float* pred, const float* gt, int B, int H, int W, const ps_lpips_net* net, void* workspace,
             double* per_layer, double* out, void* stream);

/* Colormapped evaluation images, as the reference model's `get_image_metrics_and_images` (nerfstudio's
 * models/nerfacto.py) builds them with utils/colormaps.py and default ColormapOptions, for one image of HW pixels:
 *   out[0]     [HW,3] = lut[idx(acc)]                                         (apply_colormap(accumulation))
 *   out[1 + m] [HW,3] = lut[idx(clip((d - near) / (far - near + 1e-10), 0, 1))] * acc + (1 - acc), d = maps[m]
 *                                                                             (apply_depth_colormap(d, accumulation))
 *   idx(x) = long(nan_to_num(clip(x, 0, 1)) * 255); near / far = min / max of the map, NaN if it holds one.
 * Bit-identical to torch running that definition on the device (rounding of each step in csrc/colormap_core.h).
 *   maps [M][HW] fp32 (M depth-like maps: depth, prop_depth_0, ...), acc [HW] fp32, lut [256][3] fp32 (e.g. matplotlib's
 *   turbo colours), out [M+1][HW][3] fp32.  M in [0, 1024]; maps and workspace may be NULL when M == 0.
 * workspace: device memory of ps_colormap_workspace(M, HW) bytes.  Status 1 for M outside [0, 1024], HW <= 0 or a null
 * pointer.  No host synchronisation and no floating-point atomics: repeated calls are bit-identical. */
int ps_colormap_workspace(int M, int64_t HW, int64_t* bytes);
int ps_colormap(const float* maps, int M, int64_t HW, const float* acc, const float* lut, void* workspace, float* out,
                void* stream);

/* Depth metrics of rendered depth maps against LiDAR depth (Eigen et al. / Monodepth convention), for one image of HW
 * pixels and M in [1, 4] maps (e.g. the "depth" and "expected_depth" outputs):
 *   pred_m = pred / pose_scale (fp32 IEEE division); valid pixels: min_m < target_m < max_m (0 = no LiDAR);
 *   p = pred_m clamped to [min_m, max_m]; per map, over the valid pixels, terms in fp64 from the fp32 p and t:
 *   out [M][8] f64 = abs_rel mean |p-t|/t, sq_rel mean (p-t)^2/t, rmse sqrt mean (p-t)^2, rmse_log sqrt mean (ln p -
 *   ln t)^2, a1 / a2 / a3 the fraction with max(p/t, t/p) < 1.25^k, n_valid.  No valid pixel: NaN metrics, n_valid 0.
 *   Definitions in presight_b200/csrc/depth_metrics_core.h.  pred [M][HW] fp32 (scene units), target_m [HW] fp32 metres.
 *   pose_scale: host value, or pose_scale_dev (a device float, read on the device) when not NULL.
 * workspace: device memory of ps_depth_metrics_workspace(M, HW) bytes.  Status 1 for M outside [1, 4], HW <= 0, a null
 * pointer, pose_scale <= 0 (host value), or bounds outside 0 < min_m < max_m < inf.  No host synchronisation and no
 * floating-point atomics: repeated calls are bit-identical. */
int ps_depth_metrics_workspace(int M, int64_t HW, int64_t* bytes);
int ps_depth_metrics(const float* pred, int M, int64_t HW, const float* target_m, float pose_scale,
                     const float* pose_scale_dev, float min_m, float max_m, void* workspace, double* out, void* stream);

/* Nearest-neighbour distances within a radius between two point clouds (accuracy / completeness of extracted priors
 * against a LiDAR cloud), on a grid of cells of side r = `cell` over the reference set.  Build, per reference set
 * points [M,3] f32 (M >= 1):
 *   ps_nn_grid_bounds        bounds[6] (device; caller presets +inf x3, -inf x3) <- per-axis min, max
 *   ps_nn_grid_cells_per_axis  cells[3] (host) <- floor((max - min) / r) + 1 per axis from bounds_host[6]; status 1 with
 *                            a message when an axis needs more than 2^21 cells
 *   ps_nn_grid_keys          keys [M] i64 <- (cx << 42) | (cy << 21) | cz, c = floor(((double)p - (double)min) / r); the
 *                            same extent check
 *   (the caller sorts the keys, keeping the permutation perm [M] i64)
 *   ps_nn_grid_count_cells   *n_cells (device i64, caller presets 0) += the number of distinct sorted keys
 *   ps_nn_grid_cells         cell_keys [capacity] i64 (caller presets -1), cell_ranges [capacity][2] i32 <- [start, end)
 *                            of every cell in sorted order; points_sorted [M,3] <- points[perm]; capacity a power of two
 *                            (>= 2 n_cells keeps probes short); status |= 1 table full, |= 2 a cell was lost.
 * Query, for N query points [N,3] f32 (any N; chunks of one scoring run are consecutive calls):
 *   ps_nn_grid_query         d = min over the grid's points of sqrt(((qx-px)^2 + (qy-py)^2) + (qz-pz)^2), every step in
 *                            fp64 from the fp32 coordinates, or r when that is not < r; dist_out [N] f64 (nullable).  The
 *                            call scores queries as blocks of PS_NN_BLOCK_QUERIES consecutive points: block_sums[first_block
 *                            + b] f64 = sum of d, block_counts[(first_block + b) K + k] i64 = #(d < taus_host[k]),
 *                            0 < taus_host[k] <= r, K <= PS_NN_MAX_TAUS.  A chunk that is not the last must hold a
 *                            multiple of PS_NN_BLOCK_QUERIES points for the blocks to line up.
 *   ps_nn_grid_reduce        mean[0] = sum of block_sums / n, counts[k] = sum of block_counts[.][k], fixed order.
 * No floating-point atomics: repeated calls, and any chunking into whole blocks, give bit-identical results. */
#define PS_NN_BLOCK_QUERIES 1024
#define PS_NN_MAX_TAUS 8
typedef struct ps_nn_grid {
    const float* points;        /* [M,3] in cell order (points_sorted) */
    const int64_t* cell_keys;   /* [capacity] */
    const int32_t* cell_ranges; /* [capacity][2] */
    int64_t capacity;
    float origin[3];            /* the per-axis minimum the keys were computed from */
    double cell;                /* r */
} ps_nn_grid;
int ps_nn_grid_bounds(const float* points, int64_t M, float* bounds, void* stream);
int ps_nn_grid_cells_per_axis(const float* bounds_host, double cell, int64_t* cells);
int ps_nn_grid_keys(const float* points, int64_t M, const float* bounds_host, double cell, int64_t* keys, void* stream);
int ps_nn_grid_count_cells(const int64_t* sorted_keys, int64_t M, int64_t* n_cells, void* stream);
int ps_nn_grid_cells(const float* points, const int64_t* perm, const int64_t* sorted_keys, int64_t M, int64_t* cell_keys,
                     int32_t* cell_ranges, int64_t capacity, float* points_sorted, int* status, void* stream);
int ps_nn_grid_query(const ps_nn_grid* grid, const float* queries, int64_t N, int64_t first_block, const double* taus_host,
                     int K, double* dist_out, double* block_sums, int64_t* block_counts, void* stream);
int ps_nn_grid_reduce(const double* block_sums, const int64_t* block_counts, int64_t nblocks, int K, int64_t n,
                      double* mean, int64_t* counts, void* stream);

/* ---------------------------------------------------------------------------------------
 * Sub-field routing and the sub-field mode of the fused levels (SURVEY §8 a10).  Replace the nearest-centroid routers
 * fields/PreSight/ingp_field_ms.py:80-126, prop_density_field_ms.py:86-105 (cdist().argmin, then per sub-field a
 * boolean-mask gather, a field call, a masked scatter and a `torch.any` host sync) without any host synchronisation:
 *
 *   ps_ms_route    every point (positions [P,3], or ray sample mid-points from origins / dirs [N,3] + eu_bins [N,S+1] with
 *                  P = N*S) -> sf_out [P] = index of the nearest centroid (first minimum), block_hist [nf, ceil(P/256)] =
 *                  points per sub-field of every block of 256 consecutive points.  centroids [nf,3] on the device.
 *   ps_ms_plan     block_hist -> (in place) first row of every block relative to its sub-field's segment; seg_start
 *                  [2*nf+1] = nf+1 segment starts (segments padded to multiples of `pad` rows) followed by the nf
 *                  sub-field totals; tile_sf [max_rows / tile_rows] = sub-field of every tile of `tile_rows` rows,
 *                  255 past the last segment.
 *   ps_ms_scatter  every point -> its row of its sub-field's segment (a STABLE counting sort: the original order is kept
 *                  inside a segment, the result is deterministic): perm[row] = point (caller presets perm to -1 = padding), x01_sorted [max_rows,3] = unit-cube position
 *                  normalised by THAT sub-field's aabb (aabbs [nf,6] on the device: min xyz, max xyz;
 *                  fields/PreSight/utils.py:6-10 + the L-inf contraction), sel_sorted [max_rows] = inside-the-cube flag.
 *   max_rows >= P + nf * pad is a static bound, so nothing has to be read back.
 *
 *   ps_hash_fwd_ms / ps_hash_bwd_ms    the hash encoding over those rows (level-major features [L][rows][F]); tables /
 *                  dtables = device arrays of one table pointer per sub-field.
 *   ps_prop_level_fwd_ms / _bwd_ms     PropNetDensityField.density_fn per row with the row's sub-field's table and MLP
 *                  (nets_dev: device array of ps_prop_net_dev): density [P] written at the point's own index /
 *                  d_density [P] -> dtables and the sub-fields' dW0 / db0 / dW1 / db1 (accumulated).
 *   ps_field_level_fwd_ms / _bwd_ms    iNGPField (density, colour head, semantic head) per row from the sorted hash features
 *                  (nets_dev: device array of ps_field_net_dev): density [P], rgb [P,3], sem [P,64] at the point's own
 *                  index / their gradients -> dfeat (sorted), dapp [N,A] and the sub-fields' dW / dB (accumulated).
 *   Weights along the rays and their backward then run in ps_composite_fwd / ps_composite_bwd.  rows: multiple of 128
 *   (proposal) / 256 (field) — use pad = 256. */
typedef struct ps_prop_net_dev {
    const float* W0; const float* b0; const float* W1; const float* b1;
    float* dW0; float* db0; float* dW1; float* db1;
} ps_prop_net_dev;
typedef struct ps_field_net_dev {
    const float* W[8]; const float* B[8];
    float* dW[8]; float* dB[8];
    int in_dim;   /* L * F */
    int app_dim;
} ps_field_net_dev;
int ps_ms_route(const float* positions, const float* origins, const float* dirs, const float* eu_bins, int64_t P, int S,
                const float* centroids, int nf, uint8_t* sf_out, int32_t* block_hist, void* stream);
int ps_ms_plan(int32_t* block_hist, int64_t P, int nf, int pad, int tile_rows, int64_t max_rows, int32_t* seg_start,
               uint8_t* tile_sf, void* stream);
int ps_ms_scatter(const float* positions, const float* origins, const float* dirs, const float* eu_bins, int64_t P, int S,
                  const uint8_t* sf, const float* aabbs, int nf, int contract, const int32_t* block_off,
                  const int32_t* seg_start, int32_t* perm, float* x01_sorted, uint8_t* sel_sorted, void* stream);
int ps_hash_fwd_ms(const float* x01_sorted, int64_t rows, const float* const* tables, const uint8_t* tile_sf,
                   const float* scalings_host, int L, int F, int log2_T, float* out, void* stream);
int ps_hash_bwd_ms(const float* x01_sorted, int64_t rows, float* const* dtables, const uint8_t* tile_sf, const int32_t* perm,
                   const float* scalings_host, int L, int F, int log2_T, const float* dout, void* stream);
int ps_prop_level_fwd_ms(const ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted, const uint8_t* sel_sorted,
                         const int32_t* perm, const uint8_t* tile_sf, int64_t rows, const float* const* tables_dev,
                         const float* scalings_host, int L, int F, int log2_T, float* density, void* feat_bf16,
                         void* stream);
int ps_prop_level_bwd_ms(const ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted, const uint8_t* sel_sorted,
                         const int32_t* perm, const uint8_t* tile_sf, int64_t rows, float* const* dtables_dev,
                         const float* scalings_host, int L, int F, int log2_T, const void* feat_bf16,
                         const float* d_density, void* stream);
int ps_field_level_fwd_ms(const ps_field_net_dev* nets_dev, int app_dim, const float* feat_lm_sorted, int L, int F,
                          const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows, int S,
                          const float* dirs, const float* app, float* density, float* rgb, float* sem, void* stream);
int ps_field_level_bwd_ms(const ps_field_net_dev* nets_dev, int app_dim, const float* feat_lm_sorted, int L, int F,
                          const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows, int S,
                          const float* dirs, const float* app, const float* d_density, const float* d_rgb,
                          const float* d_sem, float* dfeat_lm_sorted, float* dapp, void* stream);

/* ---------------------------------------------------------------------------------------
 * Batch assembly on the device (SURVEY §8f-3).  Replaces ImageChunk.__getitem__ + the DataLoader's collate + the host->device
 * copies of next_train_image (data/PreSight/my_dataset.py:52-73, my_datamanager.py:257-285) for a chunk that is resident in
 * HBM: row idx[b] of every field -> row b of the batch, ray_index[b] = (image_index, pixel_index / width, pixel_index % width).
 *   chunk fields [n_chunk, ...]: rgbs [.,3] f32, segs u8 (nullable), skies f32, depths f32, features [.,C] f32 (nullable),
 *                pixel_indices / image_indices / video_ids / widths i64
 *   idx [B] i64 (the sampler's indices); bad_index_flag: set to 1 if an index falls outside the chunk
 */
int ps_assemble_batch(const float* rgbs, const uint8_t* segs, const float* skies, const float* depths, const float* features,
                      int C, const int64_t* pixel_indices, const int64_t* image_indices, const int64_t* video_ids,
                      const int64_t* widths, int64_t n_chunk, const int64_t* idx, int64_t B, float* rgb, uint8_t* seg,
                      float* sky, float* depth, float* feat, int64_t* image_index, int64_t* video_id, int64_t* ray_index,
                      int* bad_index_flag, void* stream);

/* ---------------------------------------------------------------------------------------
 * Data-parallel exchange step over peer memory (one node, NVLink / NVSwitch), copy engines instead of collective kernels.
 * Replaces the all-reduce DDP performs for the reference (pipelines/PreSight/my_pipeline.py:121-124) for the large
 * gradients; host protocol in presight_b200/peer_exchange.py.
 *   ps_peer_alloc / free     device buffer that can be exported to the other ranks of the node (plain cudaMalloc)
 *   ps_peer_export           handle64_host[64] <- cudaIpcMemHandle of the buffer
 *   ps_peer_open / close     map a buffer exported by another rank (peer access enabled lazily)
 *   ps_peer_copy             stream-ordered copy between any two (local or mapped) device buffers, on the copy engines
 *   ps_peer_wait_flags       block the stream until flags[i * stride] == value for all i < n (one polling warp)
 *   ps_peer_exchange_range   push + reduce + broadcast of one row range as two kernels (see below)
 *   ps_peer_reduce           dst[i] = scale * (dst[i] + sum_k srcs_host[k][i]), n a multiple of 4, n_src <= PS_MAX_FIELDS
 */
int ps_peer_alloc(size_t bytes, void** ptr);
int ps_peer_free(void* ptr);
int ps_peer_export(void* ptr, void* handle64_host);
int ps_peer_open(const void* handle64_host, void** ptr);
int ps_peer_close(void* ptr);
int ps_peer_copy(void* dst, const void* src, size_t bytes, void* stream);
int ps_peer_wait_flags(const uint32_t* flags, int n, int stride, uint32_t value, void* stream);
int ps_peer_reduce(float* dst, const float* const* srcs_host, int n_src, int64_t n, float scale, void* stream);
/* The same three phases for one row range with P2P stores from `ctas` small CTAs (push kernel, then wait + average +
 * broadcast kernel) — no per-copy latency.  peer_bases_host[world]: every rank's allocation as mapped in this process
 * (this rank's own included); offsets are bytes inside an allocation; flag*_off: [world] uint32 phase flags of the range;
 * counters: two zero-initialised uint32 in local device memory private to the range. */
int ps_peer_exchange_range(void* const* peer_bases_host, int world, int rank, size_t g_off, size_t s_off, size_t range_off,
                           size_t shard_bytes, size_t flag1_off, size_t flag2_off, uint32_t step, float scale,
                           unsigned int* counters, int ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PRESIGHT_B200_H */
