"""
Helpers of the SGLD hot path with the reference's names (reference utils/util.py).  Volume-sized work goes to the CUDA
kernels of libirsgmcmc.so; what is left in torch is scalar or book-keeping glue.  File / VTK / SimpleITK helpers of the
reference are out of scope (SURVEY.md section 2).
"""
import math

import numpy as np
import torch

from .. import ops


def get_noise_uniform(shape, device, alpha):
    """reference :52-53"""
    return -2.0 * alpha * torch.rand(shape, device=device) + alpha


def get_noise_Langevin(sigma, tau):
    """reference :56-58"""
    return math.sqrt(2.0 * tau) * sigma * torch.randn_like(sigma)


def add_noise_uniform_field(field, alpha):
    """reference :44-45"""
    return field + transform_coordinates(get_noise_uniform(field.shape, field.device, alpha))


def add_noise_Langevin(field, sigma, tau):
    """reference :48-49"""
    return field + get_noise_Langevin(sigma, tau)


def get_control_grid_size(dims, cps):
    """control grid size of a B-spline FFD with control point spacing cps (reference utils/util.py:61-69)"""
    return tuple([int(math.ceil((sz - 1) / c) + 1 + 2) for sz, c in zip(dims, cps)])


def transform_coordinates(field):
    """voxel units -> normalised units: channel i times 2 / (shape[2 + i] - 1)  (reference :418-429)"""
    scale = torch.tensor([2.0 / float(n - 1) for n in field.shape[2:]], device=field.device, dtype=field.dtype)
    return field * scale.view(1, -1, *([1] * (field.dim() - 2)))


def transform_coordinates_inv(field):
    """reference :432-443"""
    scale = torch.tensor([float(n - 1) / 2.0 for n in field.shape[2:]], device=field.device, dtype=field.dtype)
    return field * scale.view(1, -1, *([1] * (field.dim() - 2)))


def init_identity_grid_3D(dims):
    """(1, nz, ny, nx, 3) identity sampling grid, last dim (x, y, z), from fp32 torch.linspace (reference :263-278)"""
    nx, ny, nz = dims[0], dims[1], dims[2]
    x, y, z = (torch.linspace(-1, 1, steps=n) for n in (nx, ny, nz))
    gz, gy, gx = torch.meshgrid(z, y, x, indexing='ij')
    return torch.stack((gx, gy, gz), 3).unsqueeze(0)


def separable_conv_3D(field, *args):
    """
    separable smoothing of a vector field with replicate padding.  Two call forms like the reference (:350-406):
    (field, kernel_1d, padding_sz) with a (3,1,k) conv1d weight, or (field, S_x, S_y, S_z, padding6) with the three
    depthwise conv3d weights.  Same taps on every axis and channel are assumed (all the reference ever builds).
    """
    from .functions import langevin_sobolev
    kernel = args[0]
    taps = [float(t) for t in kernel[0].reshape(-1).tolist()]
    return langevin_sobolev(field.contiguous(), None, 0.0, taps)


def rescale_residuals(res, mask, data_loss):
    """
    precision-weighted squared residuals r = z^2 sum_k rho_k(z) / sigma_k^2 on the mask, 0 elsewhere -- the closed form
    of the reference's inner autograd pass (:330-347)
    """
    z = res.detach().contiguous()
    _, dz, _ = ops.gmm_log_pdf(z.reshape(-1), data_loss.log_std, data_loss.logits, want_dz=True)
    r = (-z.reshape(-1) * dz).view(res.shape)
    return torch.where(mask, r, torch.zeros_like(r))


@torch.no_grad()
def calc_VD_factor(residual, mask):
    """virtual decimation factor from the rescaled residual field (reference :446-485)"""
    return ops.vd_factor_from_residual(residual.contiguous(), mask.contiguous()).float()


def calc_det_J(nabla):
    """Jacobian determinant of field gradients (reference :72-91)"""
    a, b, c = nabla[..., 0], nabla[..., 1], nabla[..., 2]
    return a[:, 0] * b[:, 1] * c[:, 2] + b[:, 0] * c[:, 1] * a[:, 2] + c[:, 0] * a[:, 1] * b[:, 2] \
        - a[:, 2] * b[:, 1] * c[:, 0] - b[:, 2] * c[:, 1] * a[:, 0] - c[:, 2] * a[:, 1] * b[:, 0]


def calc_no_non_diffeomorphic_voxels(transformation, diff_op):
    """number of voxels with a NaN log det J per sample, and log det J (reference :209-212): one fused kernel over the
    forward-difference GradientOperator (no (N,3,D,H,W,3) gradient tensor is materialised).  There is no PyTorch path:
    another operator, a CPU tensor or another dtype raises."""
    from .diff_op import GradientOperator
    if type(diff_op) is not GradientOperator:
        raise NotImplementedError('calc_no_non_diffeomorphic_voxels: only GradientOperator has a CUDA kernel '
                                  '(the reference ships no other working operator, utils/diff_op.py)')
    if not transformation.is_cuda or transformation.dtype != torch.float32:
        raise NotImplementedError('calc_no_non_diffeomorphic_voxels needs a float32 CUDA tensor: irsgmcmc_b200 has no CPU path')
    counts, log_det_J = ops.log_det_jacobian(transformation.detach().contiguous())
    return counts.cpu().numpy(), log_det_J


def calc_norm(field):
    """voxel-wise Euclidean norm, (N,1,D,H,W) (reference :215-225)"""
    return torch.linalg.vector_norm(field, ord=2, dim=1, keepdim=True)


@torch.no_grad()
def calc_posterior_statistics(samples, device='cuda:0'):
    """mean and unbiased std over dim 0 through the Welford kernels (reference :114-120)"""
    samples = samples.to(device).contiguous()
    mean, m2 = torch.zeros_like(samples[0]), torch.zeros_like(samples[0])
    count = ops.welford_update(samples, 0, mean, m2)
    return mean, ops.welford_std(m2, count)


@torch.no_grad()
def calc_DSC_GPU(no_samples, seg_fixed, seg_moving, structures_dict):
    """Dice score per sample and structure (reference :123-148): one pass over the volumes for all samples and up to 32
    structures at a time (the reference loops samples x structures).  int16 CUDA segmentations only -- no PyTorch path."""
    labels = [int(x) for x in structures_dict.values()]
    a, b = seg_fixed[:no_samples], seg_moving[:no_samples].contiguous()
    if not (a.is_cuda and b.is_cuda) or a.dtype != torch.int16 or b.dtype != torch.int16:
        raise NotImplementedError('calc_DSC_GPU needs int16 CUDA segmentations: irsgmcmc_b200 has no CPU path')
    if 0 in labels:
        raise NotImplementedError('calc_DSC_GPU: label 0 is the background of the counting kernel')
    a = a[:1].contiguous() if a.stride(0) == 0 else a.contiguous()
    cnt = torch.cat([ops.dice_counts(a, b, labels[i:i + 32]) for i in range(0, len(labels), 32)], dim=1).double().cpu()
    return (2.0 * cnt[..., 2] / (cnt[..., 0] + cnt[..., 1])).float().numpy()


def _segmentations_for_surface_kernels(no_samples, seg_fixed, seg_moving, structures_dict, spacing, name):
    """(seg_a, seg_b, labels, spacing) as the surface kernels take them: the first no_samples volumes, a fixed volume
    expanded over the samples passed once; CPU tensors, other dtypes and label 0 are refused"""
    labels = [int(x) for x in structures_dict.values()]
    a, b = seg_fixed[:no_samples], seg_moving[:no_samples].contiguous()
    if not (a.is_cuda and b.is_cuda) or a.dtype != torch.int16 or b.dtype != torch.int16:
        raise NotImplementedError(f'{name} needs int16 CUDA segmentations: irsgmcmc_b200 has no CPU path')
    if 0 in labels:
        raise NotImplementedError(f'{name}: label 0 is the background of the surface kernels')
    a = a[:1].contiguous() if a.stride(0) == 0 else a.contiguous()
    sp = [float(x) for x in np.asarray(spacing.cpu() if hasattr(spacing, 'cpu') else spacing, dtype=np.float64).reshape(-1)[:3]]
    return a, b, labels, sp


@torch.no_grad()
def calc_ASD_GPU(no_samples, seg_fixed, seg_moving, structures_dict, spacing):
    """average surface distance per sample and structure (the reference's calc_metrics, utils/util.py:171-176), float64
    (no_samples, structures), inf where a structure is empty: the label-contour / exact Euclidean distance transform kernels,
    one host synchronisation per call and no volume copies.  Same definition as calc_ASD_host, which the tests compare it
    with.  int16 CUDA segmentations only -- no PyTorch path."""
    a, b, labels, sp = _segmentations_for_surface_kernels(no_samples, seg_fixed, seg_moving, structures_dict, spacing,
                                                          'calc_ASD_GPU')
    return ops.average_surface_distance(a, b, labels, sp).cpu().numpy()


@torch.no_grad()
def calc_surface_distances_GPU(no_samples, seg_fixed, seg_moving, structures_dict, spacing, percentile=95.0):
    """(ASD, HD, HD_q), each float64 (no_samples, structures), from one distance transform (ops.surface_distances): ASD is
    calc_ASD_GPU's to the bit, HD and HD_q are calc_HD_GPU's.  One host synchronisation per call."""
    a, b, labels, sp = _segmentations_for_surface_kernels(no_samples, seg_fixed, seg_moving, structures_dict, spacing,
                                                          'calc_surface_distances_GPU')
    return tuple(t.cpu().numpy() for t in ops.surface_distances(a, b, labels, sp, percentile))


@torch.no_grad()
def calc_HD_GPU(no_samples, seg_fixed, seg_moving, structures_dict, spacing, percentile=95.0):
    """(HD, HD_q) per sample and structure, float64 (no_samples, structures) each, inf where a structure is empty, 0 where the
    two coincide: HD = max(max d_AB, max d_BA), the Hausdorff distance of the two label contours (what ITK's
    HausdorffDistanceImageFilter returns on the contour images calc_ASD_host builds), and HD_q = max(P_q(d_AB), P_q(d_BA)) with
    P_q numpy's default np.percentile (method 'linear') -- HD95 for the default q = 95, the symmetric form MONAI's
    compute_hausdorff_distance(percentile=q) uses.  d_AB holds the distance from every contour voxel of A to the contour of B
    once: no surface-area weights, unlike the DeepMind surface-distance package.  The label-contour / exact Euclidean distance
    transform kernels of calc_ASD_GPU plus a radix select on the device; same definition as calc_HD_host, which the tests
    compare it with.  int16 CUDA segmentations only -- no PyTorch path."""
    a, b, labels, sp = _segmentations_for_surface_kernels(no_samples, seg_fixed, seg_moving, structures_dict, spacing,
                                                          'calc_HD_GPU')
    _, hd, hd_q = ops.surface_distances(a, b, labels, sp, percentile)
    return hd.cpu().numpy(), hd_q.cpu().numpy()


def _label_contour(mask):
    """ITK LabelContourImageFilter with its defaults on a binary image: a foreground voxel belongs to the contour when one of its
    six face neighbours is background (FullyConnectedOff); voxels on the image border count as touching background."""
    from scipy import ndimage
    return mask & ~ndimage.binary_erosion(mask, structure=ndimage.generate_binary_structure(3, 1), border_value=0)


def calc_ASD_host(seg_fixed_structure, seg_moving_structure, spacing=(1.0, 1.0, 1.0)):
    """
    Average surface distance of two binary structures the way the reference computes it (utils/util.py:171-176):
    sitk.LabelContour of both, then HausdorffDistanceImageFilter.GetAverageHausdorffDistance() = the mean of the two directed
    average distances, each the mean over the contour voxels of one image of the Euclidean distance (image spacing applied) to
    the nearest contour voxel of the other.  Host-side like the reference's (SimpleITK there, scipy's exact Euclidean distance
    transform here).  PARITY UNPINNED: SimpleITK is absent from the build image, so this restates ITK's documented algorithm and is
    checked against a brute-force evaluation of the same definition (tests/test_writers.py), not against SimpleITK itself.
    Returns inf when a structure is empty (the reference's `except: ASD = inf`).
    """
    from scipy import ndimage
    a, b = np.asarray(seg_fixed_structure).astype(bool), np.asarray(seg_moving_structure).astype(bool)
    if not a.any() or not b.any():
        return float('inf')
    # crop to the bounding box of both structures (+ 1 voxel so that the contour sees their background): every contour voxel of
    # either image lies inside it, so the distances are unchanged and the distance transforms stay small
    idx = np.argwhere(a | b)
    lo, hi = np.maximum(idx.min(0) - 1, 0), np.minimum(idx.max(0) + 2, a.shape)
    box = tuple(slice(int(l), int(h)) for l, h in zip(lo, hi))
    a, b = a[box], b[box]
    ca, cb = _label_contour(a), _label_contour(b)
    if not ca.any() or not cb.any():
        return float('inf')
    sp = [float(x) for x in np.asarray(spacing).reshape(-1)[:3]]
    # array axes are (z, y, x) of an image whose spacing is given as (x, y, z): sitk.GetImageFromArray reverses the axes
    sampling = sp[::-1]
    d_to_b = ndimage.distance_transform_edt(~cb, sampling=sampling)
    d_to_a = ndimage.distance_transform_edt(~ca, sampling=sampling)
    return 0.5 * (float(d_to_b[ca].mean()) + float(d_to_a[cb].mean()))


def calc_HD_host(seg_fixed_structure, seg_moving_structure, spacing=(1.0, 1.0, 1.0), percentile=95.0):
    """
    (HD, HD_q) of two binary structures on the host, the restatement calc_HD_GPU is tested against: the bounding-box crop,
    label contours and scipy distance transforms of calc_ASD_host, then HD = max of the two directed maxima and HD_q = max of
    np.percentile(d_AB, q) and np.percentile(d_BA, q) (method 'linear'), d_AB = the distances of the contour voxels of A to the
    contour of B.  (inf, inf) when a structure is empty.
    """
    from scipy import ndimage
    a, b = np.asarray(seg_fixed_structure).astype(bool), np.asarray(seg_moving_structure).astype(bool)
    if not a.any() or not b.any():
        return float('inf'), float('inf')
    idx = np.argwhere(a | b)
    lo, hi = np.maximum(idx.min(0) - 1, 0), np.minimum(idx.max(0) + 2, a.shape)
    box = tuple(slice(int(l), int(h)) for l, h in zip(lo, hi))
    a, b = a[box], b[box]
    ca, cb = _label_contour(a), _label_contour(b)
    sampling = [float(x) for x in np.asarray(spacing).reshape(-1)[:3]][::-1]
    d_ab = ndimage.distance_transform_edt(~cb, sampling=sampling)[ca]
    d_ba = ndimage.distance_transform_edt(~ca, sampling=sampling)[cb]
    hd = max(float(d_ab.max()), float(d_ba.max()))
    return hd, max(float(np.percentile(d_ab, percentile)), float(np.percentile(d_ba, percentile)))


@torch.no_grad()
def calc_metrics(seg_fixed, seg_moving, structures_dict, spacing, GPU=True, no_samples=1):
    """(ASD, DSC) per sample and structure like the reference's calc_metrics (:151-206), both from CUDA kernels: DSC from the
    counting kernel (calc_DSC_GPU), ASD from the label-contour / distance transform kernels (calc_ASD_GPU; same definition
    as the host restatement calc_ASD_host, parity with SimpleITK unpinned, see there).  `GPU=False` is not offered."""
    if not GPU:
        raise NotImplementedError('calc_metrics(GPU=False): the Dice scores come from the CUDA counting kernel only')
    DSC = calc_DSC_GPU(no_samples, seg_fixed, seg_moving, structures_dict)
    ASD = calc_ASD_GPU(no_samples, seg_fixed, seg_moving, structures_dict, spacing)
    return ASD, DSC


@torch.no_grad()
def calc_TRE_GPU(T, fixed_landmarks, moving_landmarks, spacing):
    """target registration error per transformation and landmark pair, float64 (C, P) in mm: T (C,3,D,H,W) fp32 normalised
    sampling grids (SGLDSampler.transformation()), landmarks (P,3) zero-based (x, y, z) voxel coordinates with row i of the
    fixed ones corresponding to row i of the moving ones, spacing (x, y, z) in mm.  The fixed landmark is carried to the moving
    image by trilinear interpolation of T (where the warp samples the moving image for it) and compared with the moving
    landmark.  CUDA kernel (ops.landmark_map), one host synchronisation; same definition as calc_TRE_host, which the tests
    compare it with bit for bit.  CUDA T only -- no PyTorch path."""
    if not T.is_cuda:
        raise NotImplementedError('calc_TRE_GPU needs a CUDA transformation: irsgmcmc_b200 has no CPU path')
    return ops.landmark_map(T.contiguous(), fixed_landmarks, moving_landmarks, spacing)[1].cpu().numpy()


def landmark_predict_host(T, fixed_landmarks):
    """(C, P, 3) float64 predicted moving positions of the fixed landmarks under T (C,3,D,H,W) on the host: the arithmetic of
    irs_landmark_predict restated in numpy, every operation rounded on its own (bit-equal to the kernel)"""
    T = np.asarray(T.detach().cpu() if hasattr(T, 'detach') else T, dtype=np.float32)
    p = np.asarray(fixed_landmarks.detach().cpu() if hasattr(fixed_landmarks, 'detach') else fixed_landmarks, dtype=np.float64)
    C, _, D, H, W = T.shape
    n = np.array([W, H, D])
    fl = np.floor(p)
    with np.errstate(invalid='ignore'):
        i0 = np.where(fl >= 0.0, np.where(fl <= n - 2, fl, n - 2), 0.0).astype(np.int64)   # NaN: 0
    f = p - i0
    x0, y0, z0 = i0[:, 0], i0[:, 1], i0[:, 2]
    fx, fy, fz = f[:, 0], f[:, 1], f[:, 2]

    def lerp(a, b, t):
        return a + t * (b - a)

    Td = T.astype(np.float64)
    out = np.empty((C, p.shape[0], 3))
    for ch in range(3):
        t = Td[:, ch]

        def at(dz, dy, dx):
            return t[:, z0 + dz, y0 + dy, x0 + dx]
        c00, c10 = lerp(at(0, 0, 0), at(0, 0, 1), fx), lerp(at(0, 1, 0), at(0, 1, 1), fx)
        c01, c11 = lerp(at(1, 0, 0), at(1, 0, 1), fx), lerp(at(1, 1, 0), at(1, 1, 1), fx)
        g = lerp(lerp(c00, c10, fy), lerp(c01, c11, fy), fz)
        out[:, :, ch] = ((g + 1.0) * float(n[ch] - 1)) * 0.5
    return out


def landmark_tre_host(pred, moving_landmarks, spacing):
    """(C, P) float64 |s o (pred - q)| with the squares summed in x, y, z order, as irs_landmark_tre"""
    q = np.asarray(moving_landmarks.detach().cpu() if hasattr(moving_landmarks, 'detach') else moving_landmarks, dtype=np.float64)
    s = [float(x) for x in np.asarray(spacing, dtype=np.float64).reshape(-1)[:3]]
    acc = np.zeros(pred.shape[:2])
    for a in range(3):
        d = s[a] * (pred[..., a] - q[:, a])
        acc = acc + d * d
    return np.sqrt(acc)


def calc_TRE_host(T, fixed_landmarks, moving_landmarks, spacing):
    """calc_TRE_GPU restated in numpy on the host, float64 (C, P) in mm, bit-equal to the kernel"""
    return landmark_tre_host(landmark_predict_host(T, fixed_landmarks), moving_landmarks, spacing)


# the columns of the per-landmark posterior table (ops.landmark_posterior)
LANDMARK_POSTERIOR_COLUMNS = {'mean_position': slice(0, 3), 'TRE_of_mean': 3, 'expected_TRE': 4, 'TRE_std': 5,
                              'covariance': slice(6, 12), 'principal_std': slice(12, 15), 'mahalanobis2': 15}


def landmark_posterior_summary(table, fixed_landmarks, moving_landmarks, spacing):
    """
    Host summaries of the (P, 16) landmark posterior table (ops.landmark_posterior) and the per-landmark arrays:
      the columns by name (LANDMARK_POSTERIOR_COLUMNS) as numpy arrays;
      'mean_TRE_of_mean', 'mean_expected_TRE'  means over the landmarks (mm);
      'initial_TRE' (P,) and 'mean_initial_TRE'  |s o (p - q)|, the TRE of the identity transformation;
      'coverage'  {50, 90, 95: fraction of landmarks whose squared Mahalanobis distance is <= the chi-square(3) quantile},
                  the share of true positions inside the posterior's credible ellipsoid (NaN with fewer than two samples);
      'uncertainty_error_spearman'  Spearman rank correlation of sqrt(trace covariance) with the TRE of the mean (NaN when
                  undefined).
    """
    from scipy import stats
    t = np.asarray(table.detach().cpu() if hasattr(table, 'detach') else table, dtype=np.float64)
    p = np.asarray(fixed_landmarks.detach().cpu() if hasattr(fixed_landmarks, 'detach') else fixed_landmarks, dtype=np.float64)
    q = np.asarray(moving_landmarks.detach().cpu() if hasattr(moving_landmarks, 'detach') else moving_landmarks, dtype=np.float64)
    out = {name: t[:, col] for name, col in LANDMARK_POSTERIOR_COLUMNS.items()}
    out['mean_TRE_of_mean'] = float(out['TRE_of_mean'].mean())
    out['mean_expected_TRE'] = float(out['expected_TRE'].mean())
    out['initial_TRE'] = landmark_tre_host(p[None], q, spacing)[0]
    out['mean_initial_TRE'] = float(out['initial_TRE'].mean())
    d2 = out['mahalanobis2']
    out['coverage'] = {level: float('nan') if np.isnan(d2).any() else float(np.mean(d2 <= stats.chi2.ppf(level / 100.0, 3)))
                       for level in (50, 90, 95)}
    cov = out['covariance']
    spread = np.sqrt(cov[:, 0] + cov[:, 3] + cov[:, 5])
    ok = np.isfinite(spread) & np.isfinite(out['TRE_of_mean'])
    rho = float('nan')
    if ok.sum() >= 2 and np.ptp(spread[ok]) > 0 and np.ptp(out['TRE_of_mean'][ok]) > 0:
        rho = float(stats.spearmanr(spread[ok], out['TRE_of_mean'][ok])[0])
    out['uncertainty_error_spearman'] = rho
    return out
