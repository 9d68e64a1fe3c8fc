/* irsgmcmc.h -- C ABI of libirsgmcmc.so: the B200-native SGLD registration step of dgrzech/ir-sgmcmc.
 *
 * The reference has no FFI: its hot path is Python calling PyTorch (SURVEY.md section 8b).  This header is the boundary a
 * maintainer would bind instead -- plain pointers and sizes, no torch types.  Each entry point names the reference
 * code it replaces (paths relative to the reference repository root).
 *
 * Common rules
 *   - every pointer is a DEVICE pointer to contiguous memory unless it is called a host pointer;
 *   - float = fp32.  Volumes are (D,H,W) row-major; vector fields are planar (C,3,D,H,W) with channel 0 = x (W axis),
 *     1 = y (H axis), 2 = z (D axis); C = number of chains (batch);
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous, nothing synchronises, nothing allocates;
 *   - the return value is 0 on success, a negative IRS_ERR_* for a rejected argument, a positive cudaError_t otherwise;
 *   - there is no CPU implementation behind any of these calls.
 */
#ifndef IRSGMCMC_H
#define IRSGMCMC_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRS_ABI_VERSION 4   /* 2: irs_svf_maxabs_floats() sizes the maxabs workspace; 3: cubic B-spline FFD entry points;
                               4: irs_sgld_config.hyper_mode (was reserved0), counters sized C + 8 with the ticket at [C] */

#define IRS_OK 0
#define IRS_ERR_BAD_ARG (-1)
#define IRS_ERR_UNSUPPORTED (-2)
#define IRS_ERR_WORKSPACE (-3)

int irs_abi_version(void);
/* human-readable text for a code returned by any function of this library */
const char* irs_error_string(int code);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Warping -- replaces RegistrationModule.forward, utils/registration.py:17-32 (F.grid_sample, border, align_corners)
 * and the uniform jitter add_noise_uniform_field, utils/util.py:44-45,52-53.
 *   T            (C,3,D,H,W) sampling grid in normalised [-1,1] units (the reference's `transformation`)
 *   img          (C or 1,1,D,H,W); img_chain_stride = D*H*W, or 0 to broadcast one image over all chains
 *   jitter_unit  optional (C,3,D,H,W) of U[0,1) numbers; the sample position becomes T + normalised(alpha - 2 alpha U)
 * ------------------------------------------------------------------------------------------------------------------ */
int irs_warp3d_fwd(const float* img, long long img_chain_stride, const float* T, const float* jitter_unit, float alpha,
                   float* out, int C, int D, int H, int W, void* stream);

/* gradient of the above w.r.t. T (the autograd of F.grid_sample w.r.t. its grid, reference utils/registration.py:29-30 inside
 * loss.backward(), trainer/trainer.py:349): g_T (C,3,D,H,W) */
int irs_warp3d_bwd_grid(const float* img, long long img_chain_stride, const float* T, const float* jitter_unit,
                        float alpha, const float* g_out, float* g_T, int C, int D, int H, int W, void* stream);

/* nearest-neighbour warp of int16 segmentations / bool masks, utils/registration.py:20-27.  Bit-exact with the
 * reference: fp32 unnormalise -> clip -> round-half-even in ATen's operation order. */
int irs_warp3d_nearest_i16(const short* seg, long long seg_chain_stride, const float* T, short* out,
                           int C, int D, int H, int W, void* stream);
int irs_warp3d_nearest_u8(const unsigned char* mask, long long mask_chain_stride, const float* T, unsigned char* out,
                          int C, int D, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Stationary velocity field -- replaces SVF_3D.forward, utils/transformation.py:63-76 (scaling and squaring) and its
 * autograd (n_steps x grid_sampler_3d_backward), in voxel units (SURVEY Appendix A.6).
 *   v        (C,3,D,H,W) velocity in voxels
 *   hist     workspace, n_steps*C*3*D*H*W floats: u_1 .. u_n (u_0 = v / 2^n is not stored); u_n is the displacement
 *   maxabs   workspace, irs_svf_maxabs_floats() floats: first the n_steps values max |u_k| of the input of step k (they
 *            size the adjoint's gather window), then per step the same maximum over cells of 32 x 8 x 8 voxels, which lets
 *            every tile of the adjoint pick its window from the displacements near it
 * Cubic volumes only (D == H == W, else IRS_ERR_UNSUPPORTED): the reference's own coordinate handling is consistent only
 * for cubes (utils/util.py:418-429 scales channel i by shape[2+i]; its data loader pads every image to a cube).
 * ------------------------------------------------------------------------------------------------------------------ */
size_t irs_svf_hist_floats(int C, int D, int H, int W, int n_steps);
size_t irs_svf_maxabs_floats(int C, int D, int H, int W, int n_steps);
int irs_svf_exp_fwd(const float* v, float* hist, float* maxabs, int n_steps, int C, int D, int H, int W, void* stream);

/* T = identity + normalised(u) and/or displacement copy.  lin_x/lin_y/lin_z: the fp32 torch.linspace(-1,1,n) tables of
 * utils/util.py:263-278 (W, H, D entries).  T or disp may be NULL. */
int irs_svf_outputs(const float* u, const float* lin_x, const float* lin_y, const float* lin_z, float* T, float* disp,
                    int C, int D, int H, int W, void* stream);

/* adjoint (what autograd does for reference utils/transformation.py:63-76 inside loss.backward(), trainer/trainer.py:349):
 * g_u (C,3,D,H,W) = dL/du_n  ->  g_v = dL/dv.  g_u is used as scratch and DESTROYED; g_work: C*3*D*H*W floats.
 * The interpolation transpose is computed as a GATHER over a window of radius floor(maxabs)+1 (no atomics); steps whose
 * radius exceeds gather_radius_max use an exact atomic scatter kernel instead. */
int irs_svf_exp_bwd(const float* v, const float* hist, const float* maxabs, float* g_u, float* g_work, float* g_v,
                    int n_steps, int gather_radius_max, int C, int D, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Cubic B-spline free-form deformation -- replaces Cubic_B_spline_FFD_3D.forward (utils/transformation.py:132-152: per
 * axis conv1D(transpose=True) = F.conv_transpose1d with stride s, the 4 s - 1 taps of B_spline_1D_kernel(s) :95-103 and
 * padding 2 s - 1, then the crop [s, s + n)) and its autograd.  SVFFD_3D (:155-164) is this followed by irs_svf_exp_fwd.
 *   cp      (C,3,gD,gH,gW) control-point velocities, g = get_control_grid_size(dims, cps) (utils/util.py:61-69) or any
 *           size whose un-cropped result (g-1) s + 1 covers the crop
 *   dense   (C,3,D,H,W)
 *   kernel_*_host  HOST arrays: the reference's B_spline_1D_kernel(s) for the D, H and W axis (4 s - 1 floats, s <= 8)
 *   work    irs_ffd_work_floats() floats
 * irs_bspline_axis is one axis of it on an (outer, len, inner) array -- conv1D(x, kernel, dim, stride, padding = 2 s - 1,
 * transpose=True) with crop_start = 0 and n = (g-1) s + 1; adjoint != 0 maps (outer, n, inner) back to (outer, g, inner).
 * ------------------------------------------------------------------------------------------------------------------ */
size_t irs_ffd_work_floats(int C, int gD, int gH, int gW, int D, int H, int W);
int irs_ffd_fwd(const float* cp, const float* kernel_d_host, const float* kernel_h_host, const float* kernel_w_host,
                int sD, int sH, int sW, float* work, float* dense, int C, int gD, int gH, int gW, int D, int H, int W,
                void* stream);
/* adjoint: g_dense (C,3,D,H,W) -> g_cp (C,3,gD,gH,gW); gathers over each control point's support, no atomics */
int irs_ffd_bwd(const float* g_dense, const float* kernel_d_host, const float* kernel_h_host,
                const float* kernel_w_host, int sD, int sH, int sW, float* work, float* g_cp, int C, int gD, int gH,
                int gW, int D, int H, int W, void* stream);
int irs_bspline_axis(const float* in, float* out, int adjoint, long long outer, int g, int n, long long inner,
                     const float* kernel_host, int stride, int crop_start, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Langevin proposal + Sobolev smoothing -- replaces SGLD.forward (utils/functions.py:76-80, utils/util.py:48-58) and
 * SobolevGrad.forward / separable_conv_3D (utils/functions.py:98-105, utils/util.py:394-404).
 *   out = S_x * S_y * S_z * replicate_pad( v + coef * sigma * eps ),  coef = sqrt(2 tau)
 *   eps: explicit N(0,1) numbers (C,3,D,H,W), or NULL to draw them with Philox4x32-10 keyed (seed, chain0 + c, iter);
 *   coef = 0 skips the noise exactly.  sigma may be NULL (= 1).  sigma_chain_stride = 3*D*H*W or 0 (shared).
 *   work: C*3*D*H*W floats.
 * ------------------------------------------------------------------------------------------------------------------ */
int irs_langevin_sobolev(const float* v, const float* sigma, long long sigma_chain_stride, float coef, const float* eps,
                         unsigned long long seed, unsigned long long iter, int chain0, const float* taps_host,
                         int n_taps, float* work, float* out, int C, int D, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Regulariser -- replaces GradientOperator.forward (utils/diff_op.py:78-96) and RegLoss.forward (model/loss.py:152-161)
 * ------------------------------------------------------------------------------------------------------------------ */
/* nabla (C,3,D,H,W,3): [c, j, ..., i] = d v_i / d x_j, forward differences, last one replicated; divided by the
 * spacing 2/(n-1) when transformation != 0 */
int irs_diff_fwd(const float* v, float* nabla, int transformation, int C, int D, int H, int W, void* stream);
/* adjoint of the above without spacing: g_v (C,3,D,H,W) from g_nabla */
int irs_diff_bwd(const float* g_nabla, float* g_v, int transformation, int C, int D, int H, int W, void* stream);
/* energy[c] = sum |D v_c|^2 (double).  partials: reduction scratch, irs_reduce_scratch_doubles(C,D,H,W) doubles;
 * counters: C zero-initialised unsigned ints (left zero on return) */
size_t irs_reduce_scratch_doubles(int C, int D, int H, int W);
int irs_reg_energy(const float* v, double* energy, double* partials, unsigned int* counters,
                   int C, int D, int H, int W, void* stream);
/* g_v[c] += coef[c] * d energy / d v  (coef: C doubles on the device; g_v accumulated in place) */
int irs_reg_energy_grad(const float* v, const double* coef, float* g_v, int C, int D, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Data term -- replaces GMM.map (LCC normalisation, model/loss.py:102-111), GMM.log_pdf / reduce
 * (model/loss.py:87-93,113-114), rescale_residuals + calc_VD_factor (utils/util.py:330-347,446-485).
 * ------------------------------------------------------------------------------------------------------------------ */
/* a = I - Box(I)/k^3 ;  rs = 1/sqrt(Box(a^2)/k^3 + 1e-10) ;  zn = a * rs     (k = 2 s + 1, replicate padding)
 * any of a / rs / zn may be NULL */
int irs_lcc_normalise(const float* im, int s, float* a, float* rs, float* zn, int C, int D, int H, int W, void* stream);
/* gradient of L w.r.t. im given g_zn = dL/d(zn);  work: C*D*H*W floats */
int irs_lcc_normalise_bwd(const float* g_zn, const float* a, const float* rs, int s, float* work, float* g_im,
                          int C, int D, int H, int W, void* stream);

/* per-voxel mixture log-density and its derivatives (reference GMM.log_pdf / forward, model/loss.py:87-93,113-114, with
 * log_proportions = log_softmax(logits + 1e-2), :67-69).  gmm_host: K log_std then K logits (host floats).
 *   logp[i] = log sum_k pi_k N(z_i; 0, sigma_k);  optional outputs: dz[i] = d logp_i / d z_i,
 *   g_params (2K doubles, device) = sum_i w_i d logp_i / d (log_std, logits), w = weights or 1 */
int irs_gmm_log_pdf(const float* z, long long n, const float* gmm_host, int K, float* logp, float* dz,
                    const float* weights, double* g_params, double* partials, unsigned int* counter, void* stream);

/* virtual decimation factor of one chain (reference rescale_residuals + calc_VD_factor, utils/util.py:330-347,446-485, called
 * from Trainer.__get_VD_factor, trainer/trainer.py:507-514): residual z (D,H,W), mask (D,H,W) bytes, mixture as above ->
 * alpha (1 double) */
int irs_vd_factor(const float* z, const unsigned char* mask, const float* gmm_host, int K, double* alpha,
                  double* partials, unsigned int* counter, int D, int H, int W, void* stream);

/* the same factor from an already rescaled residual field r (calc_VD_factor(residual, mask), utils/util.py:446-485) */
int irs_vd_factor_residual(const float* r, const unsigned char* mask, double* alpha, double* partials,
                           unsigned int* counter, int D, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Per-sample evaluation -- replaces calc_no_non_diffeomorphic_voxels + calc_det_J (utils/util.py:72-91,209-212),
 * calc_DSC_GPU (utils/util.py:123-148) and the average surface distance of calc_metrics (utils/util.py:171-176).
 *   log_det (C,D,H,W) optional: log det J of the transformation T (normalised units, spacing 2/(n-1));
 *   n_folded: C ints = number of voxels whose log det J is NaN (negative determinant)
 *   counts (C, n_labels, 3) unsigned: |A = l|, |B = l|, |A = l and B = l| for int16 label volumes; labels != 0
 * ------------------------------------------------------------------------------------------------------------------ */
int irs_log_det_jacobian(const float* T, float* log_det, int* n_folded, int C, int D, int H, int W, void* stream);
int irs_dice_counts(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                    int n_labels, unsigned int* counts, int C, long long V, void* stream);

/* Average surface distance -- replaces the LabelContour + HausdorffDistanceImageFilter.GetAverageHausdorffDistance() part of
 * calc_metrics (utils/util.py:171-176).  For sample c and label l, A = (seg_a[c] == l), B = (seg_b[c] == l); the contour of a
 * set is its voxels with a face neighbour outside it (outside the volume = outside); ASD = (mean over the contour of A of the
 * Euclidean distance to the contour of B + the same from B to A) / 2, inf when A or B is empty, spacing applied.
 *   irs_surface_boxes: boxes (C, n_labels, 8) ints = bounding box of A u B (z0, y0, x0, z1, y1, x1 inclusive), |A|, |B|.
 *   irs_average_surface_distance: for the pairs p = c * n_labels + l in [pair_begin, pair_end), asd[p] (asd is the whole
 *     (C, n_labels) double array).  boxes_host = the table above copied to the host; spacing_host = 3 floats (x, y, z), the W
 *     axis uses x; workspace >= 2 * (box voxels) floats summed over the non-empty pairs of the range, else IRS_ERR_WORKSPACE;
 *     partials IRS_ASD_PARTIALS_DOUBLES doubles; counters IRS_ASD_MAX_BOXES unsigned.  Deterministic (no float atomics).
 * seg_a / seg_b int16 as for irs_dice_counts; labels != 0 (IRS_ERR_UNSUPPORTED); spacing finite and > 0 (IRS_ERR_BAD_ARG). */
#define IRS_ASD_MAX_BOXES 48          /* (sample, label) boxes per launch group */
#define IRS_ASD_REDUCE_BLOCKS 64      /* blocks of the reduction per box, at most */
#define IRS_ASD_PARTIALS_DOUBLES (IRS_ASD_MAX_BOXES * 4 * IRS_ASD_REDUCE_BLOCKS)
int irs_surface_boxes(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                      int n_labels, int* boxes, int C, int D, int H, int W, void* stream);
int irs_average_surface_distance(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                                 int n_labels, const int* boxes_host, const float* spacing_host, int pair_begin,
                                 int pair_end, float* workspace, long long workspace_floats, double* partials,
                                 unsigned int* counters, double* asd, int C, int D, int H, int W, void* stream);

/* Hausdorff distance and its percentile, with the average surface distance of the same distance transform.  For the pair
 * (A, B) above, d_AB = the distances from the contour voxels of A to the contour of B (a multiset), d_BA the same from B to A:
 *   hd[p]   = max(max d_AB, max d_BA)                        (ITK HausdorffDistanceImageFilter on the contour images)
 *   hd_q[p] = max(P_q(d_AB), P_q(d_BA)), P_q = numpy.percentile(x, q), method 'linear': s sorted, h = (n - 1) (q / 100) in
 *             fp64, s[n - 1] when h >= n - 1, else s[i] + (s[i+1] - s[i]) g for g = h - i < 0.5 (i = floor(h)) and
 *             s[i+1] - (s[i+1] - s[i]) (1 - g) otherwise -- every element counts once, not weighted by surface area
 *   asd[p]  = bit-identical to irs_average_surface_distance
 * inf when A or B is empty, 0 when A == B.  The order statistics are selected on the fp32 squared distances (exact for unit and
 * dyadic spacings), then square-rooted and interpolated in fp64.  percentile in [0, 100] (else IRS_ERR_BAD_ARG, NaN included);
 * workspace >= 2 * (box voxels) + |A| + |B| floats (boxes[6], boxes[7]) summed over the non-empty pairs of the range, else
 * IRS_ERR_WORKSPACE; partials IRS_ASD_PARTIALS_DOUBLES doubles; counters IRS_SD_COUNTERS unsigned.  Deterministic: integer
 * atomics only, results independent of the batching of the pairs; no host synchronisation. */
#define IRS_SD_COUNTERS (3 * IRS_ASD_MAX_BOXES)
int irs_surface_distances(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                          int n_labels, const int* boxes_host, const float* spacing_host, double percentile, int pair_begin,
                          int pair_end, float* workspace, long long workspace_floats, double* partials,
                          unsigned int* counters, double* asd, double* hd, double* hd_q, int C, int D, int H, int W,
                          void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Posterior moments -- replaces calc_posterior_statistics (utils/util.py:114-120) without the host-side sample buffer:
 * Welford running (count, mean, M2) over samples; count is a host-side number.
 *   sample (n_new, n) : n_new new samples of n values each;  mean, m2: n floats updated in place
 * ------------------------------------------------------------------------------------------------------------------ */
int irs_welford_update(const float* sample, int n_new, long long n, double count_before, float* mean, float* m2,
                       void* stream);
/* std = sqrt(M2 / (count - 1))  (unbiased, torch.std default) */
int irs_welford_std(const float* m2, double count, float* std_out, long long n, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Convergence diagnostics -- voxel-wise split R-hat (Gelman et al., BDA3 section 11.4; the reference has no check).
 * The N kept samples of every chain are split into their first and last floor(N/2) (the middle one of an odd N is dropped):
 * M = 2 x (chains) sequences of n = floor(N/2) draws, each with its own Welford (mean, M2) in fp32.
 *   irs_split_welford_update: folds sample `count_before` + 1 of sequence (half, c) into mean / m2, for all C chains of this
 *     GPU in one launch.  disp (C,3,V), im (C,1,V); mean / m2 (2, C, 4, V): [half][c][0..2] displacement, [3] warped image.
 *     half in {0, 1}.
 *   irs_split_rhat_sums: over the n_seq sequences (n_seq, E) of mean / m2 in index order, in fp64:
 *     sums[0..E) = S1 = sum_j mean_j;  sums[E..2E) = SW = sum_j M2_j / (n - 1).  n >= 2.
 *   irs_split_rhat_between: sb[e] = SB = sum_j (mean_j - s1[e] / M)^2 over the same n_seq sequences; s1 and M (>= 2) are the
 *     totals over ALL sequences (all GPUs).
 *   irs_split_rhat_finish: rhat (n_comp, V) floats (n_comp <= IRS_RHAT_MAX_COMPONENTS, E = n_comp V) from the totals SW and SB:
 *     W = SW / M, var+ = (n - 1) / n W + SB / (M - 1), R-hat = sqrt(var+ / W); W = 0 gives 1 when SB = 0, else +inf.
 *     summary (n_comp, 3) doubles: per component over the voxels where mask (V bytes) != 0, max R-hat (0 for an empty mask), the
 *     number of voxels with R-hat > 1.01 and with R-hat > 1.1 -- block partials added in a fixed order, deterministic.
 *     partials: IRS_RHAT_PARTIALS_DOUBLES doubles; counters: IRS_RHAT_MAX_COMPONENTS unsigned ints (left zero).
 * With several GPUs: sums -> SUM all-reduce of (S1, SW) -> between -> SUM all-reduce of SB -> finish.
 * ------------------------------------------------------------------------------------------------------------------ */
#define IRS_RHAT_MAX_COMPONENTS 4
#define IRS_RHAT_REDUCE_BLOCKS 256
#define IRS_RHAT_PARTIALS_DOUBLES (IRS_RHAT_MAX_COMPONENTS * 3 * IRS_RHAT_REDUCE_BLOCKS)
int irs_split_welford_update(const float* disp, const float* im, int C, long long V, int half, double count_before,
                             float* mean, float* m2, void* stream);
int irs_split_rhat_sums(const float* mean, const float* m2, int n_seq, long long E, int n, double* sums, void* stream);
int irs_split_rhat_between(const float* mean, int n_seq, long long E, const double* s1, int M, double* sb, void* stream);
int irs_split_rhat_finish(const double* sw, const double* sb, int M, int n, const unsigned char* mask, int n_comp,
                          long long V, float* rhat, double* partials, unsigned int* counters, double* summary, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Posterior of the warped segmentation (the reference has none): a per-voxel histogram of labels over every accumulated
 * segmentation, kept in integers so that it is exact and independent of how samples are batched or split over GPUs.
 * labels_host: 1..32 distinct non-zero int16 values (0 in the list: IRS_ERR_UNSUPPORTED; duplicates: IRS_ERR_BAD_ARG); every
 * other voxel value is the class "other", which is never stored (its count is n - sum_l counts[l][v]).
 *   irs_label_counts_update: counts (n_labels, V) ints += [seg[c][v] == labels[l]] summed over the C segmentations (C, V).
 *     Zero counts before the first update.  No atomics: one thread owns each counts element.
 *   irs_label_posterior: from counts of n >= 1 segmentations,
 *     prob (n_labels, V) floats = (float)counts / (float)n;
 *     majority (V) shorts = the label of the largest count among the n_labels + 1 classes; ties go to "other" (written 0),
 *       then to the earlier entry of labels_host;
 *     entropy (V) floats = -sum_k p_k ln p_k over the n_labels + 1 classes in nats (0 ln 0 = 0);
 *     summary (n_labels, 3) long longs, exact: S = sum_v counts[l][v], O = the same over the voxels where seg_fixed == labels[l]
 *       (0 when seg_fixed is NULL), U = #{v : 0 < counts[l][v] < n}.  Integer atomics per block: deterministic.
 * Nothing synchronises with the host; both are graph-capturable.
 * ------------------------------------------------------------------------------------------------------------------ */
int irs_label_counts_update(const short* seg, int C, long long V, const int* labels_host, int n_labels, int* counts,
                            void* stream);
int irs_label_posterior(const int* counts, const int* labels_host, int n_labels, long long n, long long V,
                        const short* seg_fixed, float* prob, short* majority, float* entropy, long long* summary,
                        void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Posterior of the Jacobian determinant (the reference computes log det J per sample, utils/util.py:72-91,209-212, and
 * aggregates nothing).  ld(c, v) = what irs_log_det_jacobian writes for sample c at voxel v; the sample is finite at v when
 * ld is finite (det > 0) and folded otherwise: det < 0 (NaN, the reference's folding), det == 0 (-inf), NaN or inf input.
 * Without an exact zero or an overflow, "folded" is the reference's NaN count.  Accumulators per voxel (12 bytes, whatever
 * the number of samples): folds (V) ints = folded samples; mean, m2 (V) floats = Welford of ld over the n_v = n - folds
 * finite samples, the recurrence of irs_welford_update with the running count starting at count_before - folds.  Zero them
 * before the first update; with no fold anywhere mean / m2 equal irs_welford_update on the stacked log det volumes bit for bit.
 *   irs_jacobian_update: folds the C transformations T (C,3,D,H,W) into the accumulators (one launch); count_before = samples
 *     accumulated so far, count_before + C <= 2^24.  sample_stats (C,4) doubles per sample over the voxels where mask (V
 *     bytes) != 0: finite voxels, folded voxels, sum ld, sum ld^2 over the finite ones (counts by integer atomics, sums by
 *     block partials added in a fixed order).  partials: IRS_JACOBIAN_PARTIALS_DOUBLES(C) doubles; counters: C + 1 unsigned
 *     long longs, zero on the first call and left zero.
 *   irs_jacobian_posterior: from the accumulators of n (1..2^24) samples, p_fold = (float)folds / (float)n; mean_out = mean,
 *     NaN where n_v = 0; std_out = sqrt(m2 / (n_v - 1)), NaN where n_v < 2 (all (V) floats).  summary: IRS_JACOBIAN_SUMMARY_WORDS
 *     8-byte words over the mask voxels: [0] sum folds, [1] #{folds > 0}, [2] #{2 folds > n}, [3] #{n_v >= 1}, [4] #{n_v >= 2},
 *     [7] mask voxels as long longs (exact, integer atomics); [5] mean of mean_out over the voxels of [3], [6] mean of std_out
 *     over those of [4] as doubles (NaN for none; fixed-order block partials).  partials: IRS_JACOBIAN_PARTIALS_DOUBLES(1)
 *     doubles; counters: 1 unsigned long long.
 * Deterministic, no host synchronisation, graph-capturable.
 * ------------------------------------------------------------------------------------------------------------------ */
#define IRS_JACOBIAN_REDUCE_BLOCKS 1184
#define IRS_JACOBIAN_PARTIALS_DOUBLES(C) (2 * (size_t)(C) * IRS_JACOBIAN_REDUCE_BLOCKS)
#define IRS_JACOBIAN_SUMMARY_WORDS 8
int irs_jacobian_update(const float* T, const unsigned char* mask, int C, int D, int H, int W, double count_before,
                        int* folds, float* mean, float* m2, double* sample_stats, double* partials,
                        unsigned long long* counters, void* stream);
int irs_jacobian_posterior(const int* folds, const float* mean, const float* m2, long long n, long long V,
                           const unsigned char* mask, float* p_fold, float* mean_out, float* std_out, double* partials,
                           unsigned long long* counters, long long* summary, void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * Landmark registration error and landmark posterior (the reference has none).  Landmarks are (P,3) doubles in zero-based
 * voxel coordinates (x, y, z) = (W, H, D); row i of the fixed landmarks p corresponds to row i of the moving landmarks q.
 * spacing_host: 3 HOST doubles (x, y, z) in mm, finite and > 0 (both images share one grid).
 *   irs_landmark_map: for chain c of T (C,3,D,H,W) and landmark i, the predicted moving position pred (C,P,3) doubles: per
 *     axis i0 = min(floor(p_a), n_a - 2) clamped to [0, n_a - 2] (no coordinate, NaN included, reads outside T), f = p_a - i0;
 *     fp64 trilinear interpolation of the fp32 corners as lerps a + f (b - a) along x, then y, then z, every operation rounded
 *     on its own (no FMA); m_a = ((g_a + 1) (n_a - 1)) 0.5.  tre (C,P) doubles = sqrt of the sum over x, y, z of
 *     (s_a (m_a - q_a))^2.  p should lie in [0, n_a - 1] (the Python op checks it); outside, m extrapolates the edge cell.
 *   irs_landmark_update: folds pred / tre of C chains into acc (P, IRS_LANDMARK_ACC) doubles, chains in index order, sample
 *     count k = count_before + c + 1: delta = m - mean, mean += delta / k, M_ab += delta_a (m_b - mean_b) over (xx, xy, xz, yy,
 *     yz, zz), and the Welford mean / M2 of the TRE -- per landmark [0,3) mean, [3,9) M, [9] TRE mean, [10] TRE M2.  Zero acc
 *     before the first update; splitting the chains of a sample over several calls gives the same bits.  count_before: an
 *     integer >= 0 with count_before + C <= 2^53.  sample_stats (C,3) doubles per chain, landmarks in index order: sum TRE,
 *     sum TRE^2, max TRE.
 *   irs_landmark_posterior: from acc over n (1..2^53) samples, out (P, IRS_LANDMARK_COLS) doubles per landmark:
 *     [0,3) mean position (moving voxels), [3] TRE of the mean |s o (mean - q)|, [4] E[TRE],
 *     and for n >= 2 (NaN for n = 1): [5] unbiased std of TRE, [6,12) covariance s_a s_b M_ab / (n - 1) in mm^2 (xx, xy, xz, yy,
 *     yz, zz), [12,15) principal standard deviations sqrt(max(lambda, 0)) in descending order (closed-form symmetric 3x3),
 *     [15] squared Mahalanobis distance r^T Sigma^-1 r, r = s o (q - mean), by a Cholesky factorisation (+inf for a pivot <= 0).
 * C < 1, P < 1, n_a < 2, null pointers, bad spacing or counts: IRS_ERR_BAD_ARG before any CUDA call.  No atomics, no host
 * synchronisation, graph-capturable.
 * ------------------------------------------------------------------------------------------------------------------ */
#define IRS_LANDMARK_ACC 11
#define IRS_LANDMARK_COLS 16
int irs_landmark_map(const float* T, int C, int D, int H, int W, const double* p, const double* q, int P,
                     const double* spacing_host, double* pred, double* tre, void* stream);
int irs_landmark_update(const double* pred, const double* tre, int C, int P, double count_before, double* acc,
                        double* sample_stats, void* stream);
int irs_landmark_posterior(const double* acc, const double* q, int P, long long n, const double* spacing_host, double* out,
                           void* stream);

/* ------------------------------------------------------------------------------------------------------------------ *
 * The fused SGLD transition -- replaces Trainer._SGLD_transition, trainer/trainer.py:291-356, for all chains of this
 * GPU, including the sequential per-chain GMM Adam step (trainer.py:316-327, 68-77; optimizers/adam_rate_decay.py),
 * the regulariser's hyper-parameter Adam step (trainer.py:353-354) and the plain-SGD state update (trainer.py:351).
 * No host synchronisation; all scalars stay on the device.
 * ------------------------------------------------------------------------------------------------------------------ */
#define IRS_DATA_LCC 0
#define IRS_DATA_SSD 1
#define IRS_REG_L2 0
#define IRS_REG_LOGNORMAL 1

/* layout of the `hyper` device array of doubles */
#define IRS_HYPER_GMM_STEP 0     /* Adam step counter of the GMM optimiser */
#define IRS_HYPER_LOG_STD 1      /* 8 slots each */
#define IRS_HYPER_LOGITS 9
#define IRS_HYPER_M_LOG_STD 17
#define IRS_HYPER_V_LOG_STD 25
#define IRS_HYPER_M_LOGITS 33
#define IRS_HYPER_V_LOGITS 41
#define IRS_HYPER_REG_STEP 49
#define IRS_HYPER_REG_P 50       /* (loc, log_scale) or (log_w_reg, -) */
#define IRS_HYPER_REG_M 52
#define IRS_HYPER_REG_V 54
#define IRS_HYPER_ITER 56        /* iteration counter: the Philox offset */
#define IRS_HYPER_GMM_BETA_POW 57 /* beta1^t, beta2^t of the mixture optimiser (running products) */
#define IRS_HYPER_REG_BETA_POW 59 /* same for the regulariser optimiser */
#define IRS_HYPER_SCRATCH 64     /* 24 doubles of reduction scratch used inside a step */
#define IRS_HYPER_SIZE 96
#define IRS_HYPER_REFERENCE 0
#define IRS_HYPER_PER_CHAIN 1
#define IRS_HYPER_FROZEN 2

/* layout of one row of the per-chain `stats` output (doubles) */
#define IRS_STAT_ALPHA 0         /* virtual decimation factor */
#define IRS_STAT_DATA 1          /* alpha * NLL with the updated mixture  (loss_terms['data'][c]) */
#define IRS_STAT_REG 2           /* regularisation loss                   (loss_terms['reg'][c]) */
#define IRS_STAT_ENERGY 3        /* sum |D v|^2                           (aux['reg_energy'][c]) */
#define IRS_STAT_NLL_PRE 4       /* NLL before the mixture update */
#define IRS_STAT_REG_COEF 5      /* d reg / d energy used for the field gradient */
#define IRS_STAT_SIZE 8

typedef struct irs_sgld_config {
    int C, D, H, W;
    int chain_offset;            /* global index of chain 0: Philox key, makes results independent of the GPU count */
    int data_term;               /* IRS_DATA_* */
    int K;                       /* mixture components (1 for SSD) */
    int lcc_s;                   /* LCC half window */
    int reg_type;                /* IRS_REG_* */
    int reg_learnable;
    int n_taps;                  /* Sobolev kernel width 2 s + 1 (0 = smoothing disabled) */
    int svf_steps;
    int virtual_decimation;
    int use_jitter;
    int gather_radius_max;       /* adjoint gather window limit; larger displacements use the atomic kernel */
    int hyper_mode;              /* IRS_HYPER_REFERENCE (0): ONE mixture / regulariser parameter set shared by all chains,
                                  * stepped chain after chain in index order (trainer/trainer.py:316-327,353-354);
                                  * IRS_HYPER_PER_CHAIN: a parameter block per chain, i.e. every chain is an independent
                                  * reference run with no_chains = 1 (`hyper` holds C * IRS_HYPER_SIZE doubles);
                                  * IRS_HYPER_FROZEN: shared parameters, no Adam steps (the reference with all hyper learning
                                  * rates at zero) -- the last two have no dependency between chains */
    float taps[16];
    double tau;
    double jitter_alpha;
    double w_reg;
    double dof;                  /* 3 D H W */
    double lr_log_std, lr_logits, lr_reg0, lr_reg1, lr_decay, beta1, beta2, adam_eps;
    double gmm_scale_prior_loc, gmm_scale_prior_scale, dirichlet_alpha;
    double reg_scale_prior_loc, reg_scale_prior_scale;
    double w_reg_prior_shape, w_reg_prior_rate;
    double n_mask;               /* number of true voxels of the fixed mask */
    unsigned long long seed;
    /* SVFFD_3D as the transformation model (utils/transformation.py:155-164): ffd_cps[0] > 0 turns it on.  The chain
     * state v, sigma, eps, css and grad_v then live on the control grid (C,3,gD,gH,gW) = ffd_grid; Langevin proposal,
     * Sobolev smoothing, regulariser and update act there, the dense velocity field is ffd_dense.  dof stays 3 D H W
     * (model/loss.py:134 takes the image size). */
    int ffd_cps[3];              /* control point spacing along D, H, W (each <= 8); all 0 = plain SVF_3D */
    int ffd_grid[3];             /* gD, gH, gW */
    float ffd_kernel[3][32];     /* B_spline_1D_kernel(cps) per axis: 4 cps - 1 taps */
} irs_sgld_config;

typedef struct irs_sgld_buffers {
    float* v;                    /* (C,3,V) chain states, updated in place */
    const float* sigma;          /* preconditioner: (C,3,V), or (1,3,V) with sigma_chain_stride = 0, or NULL (= 1) */
    long long sigma_chain_stride;
    const float* fixed;          /* LCC: normalised fixed image (F-u_F)/sigma_F (1,V);  SSD: fixed image */
    const float* moving;         /* moving image (1,V) */
    const unsigned char* mask;   /* fixed mask (1,V) bytes */
    const float* eps;            /* optional explicit N(0,1) numbers (C,3,V) instead of Philox */
    const float* jitter_unit;    /* optional explicit U[0,1) numbers (C,3,V) instead of Philox */
    float* css;                  /* (C,3,V) smoothed noisy state            = output['curr_state'] */
    float* hist;                 /* irs_svf_hist_floats();  last block      = output['displacement'] */
    float* im_warped;            /* (C,1,V)                                 = output['im_moving_warped'] */
    float* z;                    /* (C,1,V) residuals                       = aux['residuals'] (unmasked) */
    float* lcc_a;                /* (C,1,V) scratch */
    float* lcc_rs;               /* (C,1,V) scratch */
    float* scratch1;             /* (C,1,V) scratch */
    float* scratch2;             /* (C,1,V) scratch */
    float* field_a;              /* (C,3,V) scratch */
    float* field_b;              /* (C,3,V) scratch */
    float* grad_v;               /* (C,3,V) sigma^2 dL/d css: what SGD applies */
    float* maxabs;               /* irs_svf_maxabs_floats() */
    double* hyper;               /* IRS_HYPER_SIZE doubles (parameters, optimiser state, scratch); C blocks of that size with
                                  * IRS_HYPER_PER_CHAIN (the iteration counter / Philox offset is block 0's) */
    double* stats;               /* C * IRS_STAT_SIZE doubles */
    float* gmm_table;            /* C * 16 floats: per chain (lw[8], prec[8]) after that chain's update */
    double* partials;            /* irs_sgld_partials_doubles() doubles */
    unsigned int* counters;      /* C + 8 zero-initialised unsigned ints (left zero on return) */
    /* only with cfg->ffd_cps[0] > 0 */
    float* ffd_dense;            /* (C,3,V) dense velocity field of the control points */
    float* ffd_grad;             /* (C,3,V) its gradient */
    float* ffd_scratch;          /* (C,3,gD gH gW) scratch of the smoothing passes */
    float* ffd_work;             /* irs_ffd_work_floats() floats */
} irs_sgld_buffers;

size_t irs_sgld_partials_doubles(const irs_sgld_config* cfg);

/* enqueue one transition of all chains on `stream` = Trainer._SGLD_transition (reference trainer/trainer.py:291-356):
 * irs_sgld_launches_per_step(cfg) kernel launches (41 at 128^3 with one chain; 7 more with the FFD), no host synchronisation,
 * capturable in a CUDA graph */
int irs_sgld_step(const irs_sgld_config* cfg, const irs_sgld_buffers* buf, void* stream);

/* Profiling aid: one eager transition with a CUDA event between stages; synchronises the stream and writes the
 * IRS_N_STAGES stage durations (milliseconds) to the HOST array ms_host.  Stage order:
 *   0 langevin+sobolev, 1 reg energy, 2 svf forward, 3 warp, 4 residual map, 5 per-chain mixture step, 6 dL/dz,
 *   7 residual-map + warp adjoint, 8 regulariser hyper step, 9 svf adjoint, 10 regulariser gradient + SGD update */
#define IRS_N_STAGES 11
int irs_sgld_step_profile(const irs_sgld_config* cfg, const irs_sgld_buffers* buf, void* stream, float* ms_host);

/* number of kernels irs_sgld_step launches for this configuration */
int irs_sgld_launches_per_step(const irs_sgld_config* cfg);

/* one-time initialisation of the shared mixture, replaces Trainer.__GMM_init (trainer/trainer.py:529-547): forward pass
 * of the velocity sample v_sample (1,3,D,H,W) without noise, sigma_hat = std of the residuals over the mask,
 * log_std = linspace(log sigma_hat/100, log 5 sigma_hat, K), virtual decimation factor, n_warmup Adam steps.
 * Uses the chain-0 part of the step buffers. */
int irs_sgld_gmm_init(const irs_sgld_config* cfg, const irs_sgld_buffers* buf, const float* v_sample, int n_warmup,
                      void* stream);

/* mean / std over a mask, replaces Trainer.__GMM_init's statistics (trainer/trainer.py:537-541):
 * writes mean, unbiased std and count of z over the mask to out[0..2] (device doubles) */
int irs_masked_mean_std(const float* z, const unsigned char* mask, long long n, double* out, double* partials,
                        unsigned int* counter, void* stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * VI warm start: one iteration of Trainer._run_VI (reference trainer/trainer.py:119-171) as a fused device sequence.
 * q(v) = N(mu, diag(exp(log_var)) + u u^T).  Per iteration (reference lines in brackets):
 *   delta = eps sigma + x u, samples mu + delta and mu - delta                       [utils/sampler.py:4-21, trainer.py:133]
 *   both samples through the SGLD step's operators (no Langevin noise, tau = 0) as two chains on the shared mixture, in
 *   order: Sobolev, integration, warp, residual map, VD factor, mixture Adam step, data / regulariser terms and their
 *   gradients with respect to the samples                                          [trainer.py:79-117, 135-136]
 *   entropy terms and their gradients in closed form (Sherman-Morrison)              [model/loss.py:350-372, trainer.py:153-154]
 *   loss = mean data + mean reg - entropy; Adam on mu, log_var, u (lr / (1 + step lr_decay)) and, with half the summed
 *   gradient (the mean over the two samples), on the regulariser's hyper-parameters  [trainer.py:157-171]
 * cfg must describe C = 2 chains with tau = 0 and hyper_mode = IRS_HYPER_REFERENCE; buf->sigma must be NULL; buf->v and
 * buf->grad_v receive the two samples and the gradients of (data + reg) with respect to them. */
#define IRS_VI_STATE_SIZE 16
#define IRS_VI_STEP 0        /* Adam step counter = iteration number (Philox offset of eps and x) */
#define IRS_VI_BETA_POW 1    /* beta1^t, beta2^t */
#define IRS_VI_X 3           /* the scalar N(0,1) of the rank-1 term used by the last iteration */
#define IRS_VI_SUMS 4        /* sum a^2, sum a u_n, sum u_n^2, sum log_var   (a = eps + x u_n, u_n = u / sigma) */
#define IRS_VI_ENTROPY 8     /* sample term (model/loss.py:360-372), then the log-determinant term (:350-358) */

typedef struct irs_vi_buffers {
    float* mu;                   /* (1,3,Vs) variational parameters on the state grid, updated in place */
    float* log_var;
    float* u;
    float* adam_m[3];            /* Adam first / second moments of mu, log_var, u (same shapes) */
    float* adam_v[3];
    float* eps_store;            /* (1,3,Vs): the N(0,1) field of this iteration (kept from sampling to the update) */
    double* vi_state;            /* IRS_VI_STATE_SIZE doubles, zero-initialised */
    double* partials;            /* reduction scratch: 4 * 592 doubles */
    unsigned int* counter;       /* one zero-initialised unsigned int */
    const float* eps;            /* optional explicit N(0,1) numbers (1,3,Vs) instead of Philox (parity tests) */
    const float* x;              /* optional explicit scalar N(0,1) (device pointer) */
    double lr_mu, lr_log_var, lr_u, lr_decay, beta1, beta2, adam_eps;
} irs_vi_buffers;

int irs_vi_step(const irs_sgld_config* cfg, const irs_sgld_buffers* buf, const irs_vi_buffers* vi, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IRSGMCMC_H */
