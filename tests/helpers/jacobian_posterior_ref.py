"""
numpy restatement of the Jacobian posterior (csrc/irs_jacobian.cu, ops.jacobian_update / ops.jacobian_posterior), the reference
the GPU tests compare the kernels with; itself checked against plain loops in tests/test_jacobian_posterior.py.
  ld         log det J of a transformation (C,3,D,H,W) in normalised units: forward differences with the last one replicated,
             times (n - 1) / 2, the six products in the reference's order, log (float64 here)
  folded     a sample whose ld is not finite at the voxel (det <= 0, NaN or inf input); the others are finite
  accumulate (N, V) log det volumes -> folds (V) int32, mean / m2 (V) float64 over the finite samples (two passes)
  posterior  p_fold = float32(folds) / float32(n); mean, NaN where n_v = n - folds = 0; std = sqrt(m2 / (n_v - 1)), NaN where
             n_v < 2; mask summaries
  sample_stats  per sample over the mask: finite voxels, folded voxels, sum ld, sum ld^2 over the finite voxels
"""
import numpy as np


def log_det_j(T):
    """T (C,3,D,H,W) -> ld (C,D,H,W) float64"""
    T = np.asarray(T, dtype=np.float64)
    C, _, D, H, W = T.shape
    J = np.empty((C, 3, 3, D, H, W))   # J[c, j, comp]: d T_comp / d x_j, x_j in (x = W, y = H, z = D)
    for j, (axis, n) in enumerate(((4, W), (3, H), (2, D))):
        d = np.diff(T, axis=axis)
        d = np.concatenate([d, np.take(d, [-1], axis=axis)], axis=axis) * ((n - 1) / 2.0)
        J[:, j] = d
    det = (J[:, 0, 0] * J[:, 1, 1] * J[:, 2, 2] + J[:, 0, 1] * J[:, 1, 2] * J[:, 2, 0] + J[:, 0, 2] * J[:, 1, 0] * J[:, 2, 1]
           - J[:, 2, 0] * J[:, 1, 1] * J[:, 0, 2] - J[:, 2, 1] * J[:, 1, 2] * J[:, 0, 0] - J[:, 2, 2] * J[:, 1, 0] * J[:, 0, 1])
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.log(det)


def accumulate(lds):
    """lds (N, ...) -> folds (V,) int32, mean (V,) float64 (0 where no sample is finite), m2 (V,) float64"""
    x = np.asarray(lds, dtype=np.float64).reshape(len(lds), -1)
    ok = np.isfinite(x)
    nv = ok.sum(0)
    xs = np.where(ok, x, 0.0)
    mean = np.where(nv > 0, xs.sum(0) / np.maximum(nv, 1), 0.0)
    m2 = np.where(ok, (x - mean) ** 2, 0.0).sum(0)
    return (len(x) - nv).astype(np.int32), mean, m2


def posterior(folds, mean, m2, n, mask):
    """-> (p_fold float32, mean float64, std float64, summary dict) with the keys of ops.jacobian_posterior"""
    folds = np.asarray(folds, dtype=np.int64).reshape(-1)
    mean, m2 = np.asarray(mean, np.float64).reshape(-1), np.asarray(m2, np.float64).reshape(-1)
    mask = np.asarray(mask).reshape(-1).astype(bool)
    nv = n - folds
    p_fold = folds.astype(np.float32) / np.float32(n)
    mean_out = np.where(nv >= 1, mean, np.nan)
    with np.errstate(divide='ignore', invalid='ignore'):
        std_out = np.where(nv >= 2, np.sqrt(m2 / (nv - 1)), np.nan)
    m1, m2_ = mask & (nv >= 1), mask & (nv >= 2)
    summary = {'sum_folds': int(folds[mask].sum()), 'voxels_ever_folded': int((folds[mask] > 0).sum()),
               'voxels_folded_in_majority': int((2 * folds[mask] > n).sum()), 'voxels_finite': int(m1.sum()),
               'voxels_finite_2': int(m2_.sum()), 'mask_voxels': int(mask.sum()),
               'mean_log_det_J': float(mean_out[m1].mean()) if m1.any() else float('nan'),
               'mean_std_log_det_J': float(std_out[m2_].mean()) if m2_.any() else float('nan')}
    return p_fold, mean_out, std_out, summary


def sample_stats(ld, mask):
    """ld (C, ...) of one sample -> (C, 4) float64: finite voxels, folded voxels, sum ld, sum ld^2 over the mask"""
    x = np.asarray(ld, dtype=np.float64).reshape(len(ld), -1)
    mask = np.asarray(mask).reshape(-1).astype(bool)
    ok = np.isfinite(x) & mask
    xs = np.where(ok, x, 0.0)
    return np.stack([ok.sum(1), (~np.isfinite(x) & mask).sum(1), xs.sum(1), (xs * xs).sum(1)], axis=1).astype(np.float64)


def sdlogj(stats):
    """population std of log det J over the finite mask voxels from sample_stats rows (..., 4)"""
    stats = np.asarray(stats, dtype=np.float64)
    m = stats[..., 2] / stats[..., 0]
    return np.sqrt(np.maximum(stats[..., 3] / stats[..., 0] - m * m, 0.0))
