"""
Functional wrappers over the C ABI (include/irsgmcmc.h): allocate outputs with torch, pass raw pointers, launch on
torch's current stream.  CUDA tensors only -- every function raises on CPU tensors (no fallback).
"""
import ctypes
import math

import torch

from . import _lib


def _dims(t):
    if t.dim() != 5:
        raise ValueError('expected a (C, channels, D, H, W) tensor')
    return t.shape[0], t.shape[2], t.shape[3], t.shape[4]


def _f32(*tensors):
    for t in tensors:
        if t is not None and t.dtype != torch.float32:
            raise NotImplementedError(f'fp32 only, got {t.dtype}')


def warp3d(img, T, jitter_unit=None, alpha=0.0):
    """trilinear warp, border padding, align_corners (reference utils/registration.py:29-30)"""
    lib = _lib.load()
    _lib.require_cuda(img, T, jitter_unit)
    _f32(img, T, jitter_unit)
    C, D, H, W = _dims(T)
    out = torch.empty(C, 1, D, H, W, device=T.device, dtype=torch.float32)
    stride = 0 if img.shape[0] == 1 else D * H * W
    _lib.check(lib.irs_warp3d_fwd(_lib.ptr(img), stride, _lib.ptr(T), _lib.ptr(jitter_unit), float(alpha), _lib.ptr(out),
                                  C, D, H, W, _lib.stream()))
    return out


def warp3d_bwd_grid(img, T, g_out, jitter_unit=None, alpha=0.0):
    lib = _lib.load()
    _lib.require_cuda(img, T, g_out, jitter_unit)
    _f32(img, T, g_out, jitter_unit)
    C, D, H, W = _dims(T)
    g_T = torch.empty_like(T)
    stride = 0 if img.shape[0] == 1 else D * H * W
    _lib.check(lib.irs_warp3d_bwd_grid(_lib.ptr(img), stride, _lib.ptr(T), _lib.ptr(jitter_unit), float(alpha),
                                       _lib.ptr(g_out), _lib.ptr(g_T), C, D, H, W, _lib.stream()))
    return g_T


def warp3d_nearest(seg, T):
    """nearest-neighbour warp of int16 / bool volumes, bit-exact with the reference (utils/registration.py:20-27)"""
    lib = _lib.load()
    _lib.require_cuda(seg, T)
    _f32(T)
    C, D, H, W = _dims(T)
    stride = 0 if seg.shape[0] == 1 else D * H * W
    out = torch.empty(C, 1, D, H, W, device=T.device, dtype=seg.dtype)
    if seg.dtype == torch.int16:
        _lib.check(lib.irs_warp3d_nearest_i16(_lib.ptr(seg), stride, _lib.ptr(T), _lib.ptr(out), C, D, H, W, _lib.stream()))
    elif seg.dtype in (torch.bool, torch.uint8):
        _lib.check(lib.irs_warp3d_nearest_u8(_lib.ptr(seg), stride, _lib.ptr(T), _lib.ptr(out), C, D, H, W, _lib.stream()))
    else:
        raise NotImplementedError
    return out


def svf_exp_fwd(v, n_steps=12):
    """returns (hist (n_steps,C,3,D,H,W) with hist[-1] = displacement in voxels, maxabs (n_steps,))"""
    lib = _lib.load()
    _lib.require_cuda(v)
    _f32(v)
    C, D, H, W = _dims(v)
    hist = torch.empty(n_steps, C, 3, D, H, W, device=v.device, dtype=torch.float32)
    # per-step max |u_k| followed by the per-cell maxima the adjoint reads (irs_svf_maxabs_floats); the returned tensor is
    # the first n_steps entries, a view that keeps the whole block alive
    mbuf = torch.zeros(int(lib.irs_svf_maxabs_floats(C, D, H, W, n_steps)), device=v.device, dtype=torch.float32)
    maxabs = mbuf[:n_steps]
    _lib.check(lib.irs_svf_exp_fwd(_lib.ptr(v), _lib.ptr(hist), _lib.ptr(maxabs), n_steps, C, D, H, W, _lib.stream()))
    return hist, maxabs


def svf_outputs(u, lin, want_T=True):
    lib = _lib.load()
    C, D, H, W = _dims(u)
    T = torch.empty_like(u) if want_T else None
    _lib.check(lib.irs_svf_outputs(_lib.ptr(u), _lib.ptr(lin[0]), _lib.ptr(lin[1]), _lib.ptr(lin[2]), _lib.ptr(T), None,
                                   C, D, H, W, _lib.stream()))
    return T


def svf_exp_bwd(v, hist, maxabs, g_u, gather_radius_max=2):
    """dL/dv from dL/du_n (g_u is left untouched: a copy is consumed)"""
    lib = _lib.load()
    _lib.require_cuda(v, hist, maxabs, g_u)
    C, D, H, W = _dims(v)
    g_in = g_u.clone()
    work, g_v = torch.empty_like(v), torch.empty_like(v)
    _lib.check(lib.irs_svf_exp_bwd(_lib.ptr(v), _lib.ptr(hist), _lib.ptr(maxabs), _lib.ptr(g_in), _lib.ptr(work),
                                   _lib.ptr(g_v), hist.shape[0], int(gather_radius_max), C, D, H, W, _lib.stream()))
    return g_v


def _ffd_args(cp, kernels, cps, dims):
    lib = _lib.load()
    _lib.require_cuda(cp)
    _f32(cp)
    if cp.dim() != 5 or cp.shape[1] != 3 or len(kernels) != 3 or len(cps) != 3 or len(dims) != 3:
        raise RuntimeError('cubic B-spline FFD: expected a (C,3,gD,gH,gW) field, three kernels, spacings and sizes')
    for k, s in zip(kernels, cps):
        if len(k) != 4 * int(s) - 1:
            raise RuntimeError('cubic B-spline FFD: a kernel of 4 * cps - 1 taps per axis is expected')
    return lib, [_lib.host_floats([float(x) for x in k]) for k in kernels], [int(s) for s in cps]


def ffd_fwd(cp, kernels, cps, dims):
    """dense (C,3,D,H,W) velocity field of control-point velocities cp (C,3,gD,gH,gW); kernels: the three
    B_spline_1D_kernel(s) as host sequences (reference utils/transformation.py:132-152)"""
    lib, hk, st = _ffd_args(cp, kernels, cps, dims)
    C, (gD, gH, gW), (D, H, W) = cp.shape[0], cp.shape[2:], [int(n) for n in dims]
    work = torch.empty(int(lib.irs_ffd_work_floats(C, gD, gH, gW, D, H, W)), device=cp.device, dtype=torch.float32)
    dense = torch.empty(C, 3, D, H, W, device=cp.device, dtype=torch.float32)
    _lib.check(lib.irs_ffd_fwd(_lib.ptr(cp), hk[0], hk[1], hk[2], st[0], st[1], st[2], _lib.ptr(work), _lib.ptr(dense),
                               C, gD, gH, gW, D, H, W, _lib.stream()))
    return dense


def ffd_bwd(g_dense, kernels, cps, grid_size):
    """adjoint of ffd_fwd: (C,3,D,H,W) -> (C,3,gD,gH,gW)"""
    lib, hk, st = _ffd_args(g_dense, kernels, cps, grid_size)
    C, (D, H, W), (gD, gH, gW) = g_dense.shape[0], g_dense.shape[2:], [int(n) for n in grid_size]
    work = torch.empty(int(lib.irs_ffd_work_floats(C, gD, gH, gW, D, H, W)), device=g_dense.device, dtype=torch.float32)
    g_cp = torch.empty(C, 3, gD, gH, gW, device=g_dense.device, dtype=torch.float32)
    _lib.check(lib.irs_ffd_bwd(_lib.ptr(g_dense), hk[0], hk[1], hk[2], st[0], st[1], st[2], _lib.ptr(work),
                               _lib.ptr(g_cp), C, gD, gH, gW, D, H, W, _lib.stream()))
    return g_cp


def bspline_axis(x, kernel, dim, stride, adjoint=False, crop_start=0, out_len=None):
    """one axis of the FFD on an arbitrary contiguous fp32 tensor: conv1D(x, kernel, dim, stride, padding=2 stride - 1,
    transpose=True) (reference utils/transformation.py:106-129) when adjoint is False, its transpose otherwise"""
    lib = _lib.load()
    _lib.require_cuda(x)
    _f32(x)
    stride = int(stride)
    if len(kernel) != 4 * stride - 1:
        raise RuntimeError('bspline_axis: a kernel of 4 * stride - 1 taps is expected')
    dim = dim % x.dim()
    outer = 1
    for n in x.shape[:dim]:
        outer *= int(n)
    inner = 1
    for n in x.shape[dim + 1:]:
        inner *= int(n)
    if adjoint:
        if out_len is None:
            raise ValueError('bspline_axis(adjoint=True) needs out_len = the number of control points along the axis')
        n, g = int(x.shape[dim]), int(out_len)
    else:
        g = int(x.shape[dim])
        n = (g - 1) * stride + 1 - int(crop_start) if out_len is None else int(out_len)
    shape = list(x.shape)
    shape[dim] = g if adjoint else n
    out = torch.empty(shape, device=x.device, dtype=torch.float32)
    _lib.check(lib.irs_bspline_axis(_lib.ptr(x), _lib.ptr(out), int(bool(adjoint)), outer, g, n, inner,
                                    _lib.host_floats([float(v) for v in kernel]), stride, int(crop_start), _lib.stream()))
    return out


def diff_fwd(v, transformation=False):
    lib = _lib.load()
    _lib.require_cuda(v)
    _f32(v)
    C, D, H, W = _dims(v)
    nabla = torch.empty(C, 3, D, H, W, 3, device=v.device, dtype=torch.float32)
    _lib.check(lib.irs_diff_fwd(_lib.ptr(v), _lib.ptr(nabla), int(bool(transformation)), C, D, H, W, _lib.stream()))
    return nabla


def diff_bwd(g_nabla, transformation=False):
    lib = _lib.load()
    _lib.require_cuda(g_nabla)
    C, _, D, H, W, _ = g_nabla.shape
    g_v = torch.empty(C, 3, D, H, W, device=g_nabla.device, dtype=torch.float32)
    _lib.check(lib.irs_diff_bwd(_lib.ptr(g_nabla), _lib.ptr(g_v), int(bool(transformation)), C, D, H, W, _lib.stream()))
    return g_v


def _scratch(C, D, H, W, device):
    n = _lib.load().irs_reduce_scratch_doubles(C, D, H, W)
    return torch.zeros(n, device=device, dtype=torch.float64), torch.zeros(C + 1, device=device, dtype=torch.int32)


def reg_energy(v):
    """sum of squared forward differences per chain, float64 (C,)"""
    lib = _lib.load()
    _lib.require_cuda(v)
    _f32(v)
    C, D, H, W = _dims(v)
    partials, counters = _scratch(C, D, H, W, v.device)
    energy = torch.empty(C, device=v.device, dtype=torch.float64)
    _lib.check(lib.irs_reg_energy(_lib.ptr(v), _lib.ptr(energy), _lib.ptr(partials), _lib.ptr(counters), C, D, H, W,
                                  _lib.stream()))
    return energy


def reg_energy_grad(v, coef):
    """coef[c] * d energy_c / d v"""
    lib = _lib.load()
    _lib.require_cuda(v, coef)
    C, D, H, W = _dims(v)
    g = torch.zeros_like(v)
    _lib.check(lib.irs_reg_energy_grad(_lib.ptr(v), _lib.ptr(coef.double().contiguous()), _lib.ptr(g), C, D, H, W,
                                       _lib.stream()))
    return g


def lcc_normalise(im, s):
    """returns (zn, a, rs): zn = (I - u)/sigma of reference model/loss.py:103-105"""
    lib = _lib.load()
    _lib.require_cuda(im)
    _f32(im)
    C, D, H, W = _dims(im)
    a, rs, zn = torch.empty_like(im), torch.empty_like(im), torch.empty_like(im)
    _lib.check(lib.irs_lcc_normalise(_lib.ptr(im), int(s), _lib.ptr(a), _lib.ptr(rs), _lib.ptr(zn), C, D, H, W,
                                     _lib.stream()))
    return zn, a, rs


def lcc_normalise_bwd(g_zn, a, rs, s):
    lib = _lib.load()
    _lib.require_cuda(g_zn, a, rs)
    C, D, H, W = _dims(a)
    work, g_im = torch.empty_like(a), torch.empty_like(a)
    _lib.check(lib.irs_lcc_normalise_bwd(_lib.ptr(g_zn), _lib.ptr(a), _lib.ptr(rs), int(s), _lib.ptr(work), _lib.ptr(g_im),
                                         C, D, H, W, _lib.stream()))
    return g_im


def gmm_log_pdf(z, log_std, logits, want_dz=False, weights=None, want_param_grads=False):
    """per-element mixture log-density of a flat residual tensor; optional d/dz and weighted parameter gradient sums"""
    lib = _lib.load()
    _lib.require_cuda(z, weights)
    _f32(z, weights)
    K = int(log_std.numel())
    n = z.numel()
    host = _lib.host_floats(list(log_std.detach().cpu().float().tolist()) + list(logits.detach().cpu().float().tolist()))
    logp = torch.empty(n, device=z.device, dtype=torch.float32)
    dz = torch.empty(n, device=z.device, dtype=torch.float32) if want_dz else None
    gp = partials = counter = None
    if want_param_grads:
        gp = torch.zeros(2 * _lib.MAX_K, device=z.device, dtype=torch.float64)
        partials = torch.zeros(1184 * 2 * _lib.MAX_K, device=z.device, dtype=torch.float64)
        counter = torch.zeros(1, device=z.device, dtype=torch.int32)
    _lib.check(lib.irs_gmm_log_pdf(_lib.ptr(z), n, host, K, _lib.ptr(logp), _lib.ptr(dz), _lib.ptr(weights), _lib.ptr(gp),
                                   _lib.ptr(partials), _lib.ptr(counter), _lib.stream()))
    return logp, dz, gp


def vd_factor(z, mask, log_std, logits):
    """virtual decimation factor of one chain (reference utils/util.py:330-347,446-485); float64 scalar tensor"""
    lib = _lib.load()
    _lib.require_cuda(z, mask)
    _f32(z)
    D, H, W = z.shape[-3:]
    K = int(log_std.numel())
    host = _lib.host_floats(list(log_std.detach().cpu().float().tolist()) + list(logits.detach().cpu().float().tolist()))
    alpha = torch.empty(1, device=z.device, dtype=torch.float64)
    partials = torch.zeros(1184 * 32, device=z.device, dtype=torch.float64)
    counter = torch.zeros(1, device=z.device, dtype=torch.int32)
    m8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    _lib.check(lib.irs_vd_factor(_lib.ptr(z), _lib.ptr(m8), host, K, _lib.ptr(alpha), _lib.ptr(partials),
                                 _lib.ptr(counter), D, H, W, _lib.stream()))
    return alpha[0]


def vd_factor_from_residual(r, mask):
    """calc_VD_factor of the reference: alpha from a rescaled residual field (1,1,D,H,W)"""
    lib = _lib.load()
    _lib.require_cuda(r, mask)
    _f32(r)
    D, H, W = r.shape[-3:]
    alpha = torch.empty(1, device=r.device, dtype=torch.float64)
    partials = torch.zeros(1184 * 5, device=r.device, dtype=torch.float64)
    counter = torch.zeros(1, device=r.device, dtype=torch.int32)
    m8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    _lib.check(lib.irs_vd_factor_residual(_lib.ptr(r), _lib.ptr(m8), _lib.ptr(alpha), _lib.ptr(partials), _lib.ptr(counter),
                                          D, H, W, _lib.stream()))
    return alpha[0]


def masked_mean_std(z, mask):
    lib = _lib.load()
    _lib.require_cuda(z, mask)
    out = torch.empty(3, device=z.device, dtype=torch.float64)
    partials = torch.zeros(1184 * 3, device=z.device, dtype=torch.float64)
    counter = torch.zeros(1, device=z.device, dtype=torch.int32)
    m8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    _lib.check(lib.irs_masked_mean_std(_lib.ptr(z), _lib.ptr(m8), z.numel(), _lib.ptr(out), _lib.ptr(partials),
                                       _lib.ptr(counter), _lib.stream()))
    return out


def welford_update(sample, count_before, mean, m2):
    lib = _lib.load()
    _lib.require_cuda(sample, mean, m2)
    n_new, n = sample.shape[0], mean.numel()
    _lib.check(lib.irs_welford_update(_lib.ptr(sample), n_new, n, float(count_before), _lib.ptr(mean), _lib.ptr(m2),
                                      _lib.stream()))
    return count_before + n_new


def welford_std(m2, count):
    lib = _lib.load()
    out = torch.empty_like(m2)
    _lib.check(lib.irs_welford_std(_lib.ptr(m2), float(count), _lib.ptr(out), m2.numel(), _lib.stream()))
    return out


def split_welford_update(disp, im, half, count_before, mean, m2):
    """fold the current sample of every chain into its split-R-hat sequence of half `half` (0: first floor(N/2) kept samples,
    1: last floor(N/2)), which already holds `count_before` draws.  disp (C,3,D,H,W), im (C,1,D,H,W); mean / m2 (2,C,4,D,H,W)
    fp32, updated in place."""
    lib = _lib.load()
    _lib.require_cuda(disp, im, mean, m2)
    C, V = disp.shape[0], disp[0, 0].numel()
    if disp.shape[:2] != (C, 3) or im.shape[:2] != (C, 1) or im[0, 0].numel() != V:
        raise ValueError('disp must be (C,3,D,H,W) and im (C,1,D,H,W)')
    if tuple(mean.shape[:3]) != (2, C, 4) or mean[0, 0, 0].numel() != V or m2.shape != mean.shape:
        raise ValueError(f'mean / m2 must be (2, {C}, 4, D, H, W)')
    for t in (disp, im, mean, m2):
        _f32(t)
    _lib.check(lib.irs_split_welford_update(_lib.ptr(disp), _lib.ptr(im), C, V, int(half), float(count_before),
                                            _lib.ptr(mean), _lib.ptr(m2), _lib.stream()))


def split_rhat(mean, m2, n, mask, group=None, distributed=True):
    """
    Split R-hat (BDA3 section 11.4) per element from per-sequence Welford moments: mean / m2 (n_seq, K, D, H, W) fp32, each
    sequence of n >= 2 draws; mask (D,H,W) bool / uint8.  With torch.distributed initialised (and `distributed`), the
    sequences of all ranks of `group` count (two SUM all-reduces of fp64 partial sums, parallel.split_rhat_totals).
    Returns (rhat (K,D,H,W) fp32, summary (K,3) fp64 = per component over the mask: max R-hat, voxels > 1.01, voxels > 1.1,
    M = total number of sequences).
    """
    from .parallel import split_rhat_totals
    lib = _lib.load()
    _lib.require_cuda(mean, m2, mask)
    _f32(mean)
    _f32(m2)
    if mean.dim() != 5 or m2.shape != mean.shape:
        raise ValueError('mean / m2 must be (n_seq, K, D, H, W)')
    n_seq, K, (D, H, W) = mean.shape[0], mean.shape[1], mean.shape[2:]
    if not 1 <= K <= _lib.RHAT_MAX_COMPONENTS or mask.numel() != D * H * W:
        raise ValueError(f'K must be 1..{_lib.RHAT_MAX_COMPONENTS} and mask (D,H,W)')
    if int(n) < 2:
        raise ValueError('split R-hat needs at least 2 draws per sequence')
    V = D * H * W
    E, dev, st = K * V, mean.device, _lib.stream()
    sums = torch.empty(2, E, device=dev, dtype=torch.float64)
    _lib.check(lib.irs_split_rhat_sums(_lib.ptr(mean), _lib.ptr(m2), n_seq, E, int(n), _lib.ptr(sums), st))

    def between(s1, M):
        sb = torch.empty(E, device=dev, dtype=torch.float64)
        _lib.check(lib.irs_split_rhat_between(_lib.ptr(mean), n_seq, E, _lib.ptr(s1), int(M), _lib.ptr(sb), _lib.stream()))
        return sb

    if distributed:
        M, sums, sb = split_rhat_totals(n_seq, sums, between, group)
    else:
        M, sb = n_seq, between(sums[0], n_seq)
    if M < 2:
        raise ValueError('split R-hat needs at least 2 sequences')
    rhat = torch.empty(K, D, H, W, device=dev, dtype=torch.float32)
    summary = torch.empty(K, 3, device=dev, dtype=torch.float64)
    partials = torch.empty(_lib.RHAT_PARTIALS_DOUBLES, device=dev, dtype=torch.float64)
    counters = torch.empty(_lib.RHAT_MAX_COMPONENTS, device=dev, dtype=torch.int32)
    m8 = mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.contiguous()
    _lib.check(lib.irs_split_rhat_finish(_lib.ptr(sums[1]), _lib.ptr(sb), int(M), int(n), _lib.ptr(m8), K, V, _lib.ptr(rhat),
                                         _lib.ptr(partials), _lib.ptr(counters), _lib.ptr(summary), _lib.stream()))
    return rhat, summary, M


def log_det_jacobian(T, want_log_det=True):
    """log det J of a transformation (C,3,D,H,W) and the per-sample count of folded (NaN) voxels"""
    lib = _lib.load()
    _lib.require_cuda(T)
    _f32(T)
    C, D, H, W = _dims(T)
    log_det = torch.empty(C, D, H, W, device=T.device, dtype=torch.float32) if want_log_det else None
    counts = torch.empty(C, device=T.device, dtype=torch.int32)
    _lib.check(lib.irs_log_det_jacobian(_lib.ptr(T), _lib.ptr(log_det), _lib.ptr(counts), C, D, H, W, _lib.stream()))
    return counts, log_det


def dice_counts(seg_a, seg_b, labels):
    """(C, n_labels, 3) counts |A = l|, |B = l|, |A = l and B = l| for int16 label volumes (seg_a may be shared by chains)"""
    import ctypes
    lib = _lib.load()
    _lib.require_cuda(seg_a, seg_b)
    if seg_a.dtype != torch.int16 or seg_b.dtype != torch.int16:
        raise NotImplementedError('int16 segmentations only')
    C = seg_b.shape[0]
    V = seg_b[0].numel()
    stride = 0 if seg_a.shape[0] == 1 else V
    lab = (ctypes.c_int * len(labels))(*[int(x) for x in labels])
    counts = torch.empty(C, len(labels), 3, device=seg_b.device, dtype=torch.int32)
    _lib.check(lib.irs_dice_counts(_lib.ptr(seg_a), stride, _lib.ptr(seg_b), lab, len(labels), _lib.ptr(counts), C, V,
                                   _lib.stream()))
    return counts


def _label_array(labels):
    import ctypes
    labels = [int(x) for x in labels]
    return (ctypes.c_int * len(labels))(*labels), len(labels)


def label_counts_update(seg, labels, counts):
    """add the C int16 segmentations seg (C, 1, D, H, W) into counts (L, D, H, W) int32 in place: counts[l][v] += number of
    chains whose voxel v carries labels[l] (1..32 distinct non-zero values; any other value is the class "other", not stored)"""
    lib = _lib.load()
    _lib.require_cuda(seg, counts)
    if seg.dtype != torch.int16:
        raise NotImplementedError('int16 segmentations only')
    if counts.dtype != torch.int32:
        raise NotImplementedError('int32 counts only')
    C, V = seg.shape[0], seg[0].numel()
    lab, L = _label_array(labels)
    if counts.shape[0] != L or counts[0].numel() != V:
        raise ValueError(f'counts must be ({L}, D, H, W) for {L} labels over the {V} voxels of a segmentation')
    _lib.check(lib.irs_label_counts_update(_lib.ptr(seg), C, V, lab, L, _lib.ptr(counts), _lib.stream()))


def label_posterior(counts, n, labels, seg_fixed=None):
    """
    The posterior of a segmentation from the label counts (L, D, H, W) int32 of n accumulated segmentations:
      prob     (L, D, H, W) fp32   (float)counts / (float)n
      majority (1, 1, D, H, W) int16  the most frequent of the L + 1 classes; ties go to "other" (0), then to the earlier label
      entropy  (1, D, H, W) fp32   -sum_k p_k ln p_k over the L + 1 classes (nats)
      summary  (L, 3) int64        per label: S = sum of the counts, O = the same inside seg_fixed == label (0 without
                                   seg_fixed), U = voxels with 0 < count < n
    S / n is the expected volume in voxels, 2 O / (S + n |F|) the soft Dice of the probability map.  seg_fixed: int16 volume of
    the same D, H, W, or None.
    """
    lib = _lib.load()
    _lib.require_cuda(counts, seg_fixed)
    if counts.dtype != torch.int32:
        raise NotImplementedError('int32 counts only')
    if seg_fixed is not None and seg_fixed.dtype != torch.int16:
        raise NotImplementedError('int16 segmentations only')
    if counts.dim() != 4:
        raise ValueError('counts must be (L, D, H, W)')
    lab, L = _label_array(labels)
    (D, H, W), V = counts.shape[1:], counts[0].numel()
    if counts.shape[0] != L:
        raise ValueError(f'counts has {counts.shape[0]} rows for {L} labels')
    if seg_fixed is not None and seg_fixed.numel() != V:
        raise ValueError(f'seg_fixed must hold the {V} voxels of the counts')
    dev = counts.device
    prob = torch.empty(L, D, H, W, device=dev, dtype=torch.float32)
    majority = torch.empty(1, 1, D, H, W, device=dev, dtype=torch.int16)
    entropy = torch.empty(1, D, H, W, device=dev, dtype=torch.float32)
    summary = torch.empty(L, 3, device=dev, dtype=torch.int64)
    _lib.check(lib.irs_label_posterior(_lib.ptr(counts), lab, L, int(n), V, _lib.ptr(seg_fixed), _lib.ptr(prob),
                                       _lib.ptr(majority), _lib.ptr(entropy), _lib.ptr(summary), _lib.stream()))
    return prob, majority, entropy, summary


def average_surface_distance(seg_a, seg_b, labels, spacing, workspace_bytes=512 << 20):
    """float64 (C, n_labels) average surface distance of the structures seg_a == l and seg_b[c] == l (the reference's
    LabelContour + average Hausdorff distance, utils/util.py:171-176): inf when either is empty.  int16 label volumes (C or
    1, 1, D, H, W); seg_a may be one volume shared by all samples; spacing (x, y, z).  The distance transforms run over the
    bounding box of each (sample, structure), 8 bytes per box voxel, in batches of pairs whose workspace fits
    `workspace_bytes` (a pair larger than that runs alone).  One host synchronisation per 32 labels (the box table)."""
    return _surface_distances(seg_a, seg_b, labels, spacing, workspace_bytes, None)[0]


def surface_distances(seg_a, seg_b, labels, spacing, percentile=95.0, workspace_bytes=512 << 20):
    """float64 (asd, hd, hd_q), each (C, n_labels), of the structures A = seg_a == l and B = seg_b[c] == l from one distance
    transform: asd is average_surface_distance's to the bit; hd = max(max d_AB, max d_BA) is the Hausdorff distance of the two
    label contours; hd_q = max(P_q(d_AB), P_q(d_BA)) with P_q numpy's default percentile (method 'linear') of the directed
    distances d_AB (every contour voxel of A to the contour of B) and d_BA, q = `percentile` in [0, 100] (95: HD95).  Each
    contour voxel counts once: no surface-area weights (those of the DeepMind surface-distance package).  inf when A or B is
    empty.  Arguments and batching as average_surface_distance, with |A| + |B| more workspace floats per pair for the
    distance lists."""
    q = float(percentile)
    if not 0.0 <= q <= 100.0:
        raise ValueError(f'percentile must lie in [0, 100], got {percentile}')
    return _surface_distances(seg_a, seg_b, labels, spacing, workspace_bytes, q)


def _surface_distances(seg_a, seg_b, labels, spacing, workspace_bytes, percentile):
    """(asd,) with percentile None (irs_average_surface_distance), else (asd, hd, hd_q) (irs_surface_distances)"""
    import ctypes
    lib = _lib.load()
    _lib.require_cuda(seg_a, seg_b)
    if seg_a.dtype != torch.int16 or seg_b.dtype != torch.int16:
        raise NotImplementedError('int16 segmentations only')
    if seg_b.dim() < 4 or seg_b[0].numel() != seg_b.shape[-3] * seg_b.shape[-2] * seg_b.shape[-1]:
        raise ValueError('expected (C, [1,] D, H, W) label volumes')
    C, (D, H, W) = seg_b.shape[0], seg_b.shape[-3:]
    if seg_a.shape[0] not in (1, C) or seg_a.shape[1:] != seg_b.shape[1:]:
        raise ValueError(f'seg_a {tuple(seg_a.shape)} does not match seg_b {tuple(seg_b.shape)}')
    stride = 0 if seg_a.shape[0] == 1 else D * H * W
    sp = _lib.host_floats([float(x) for x in spacing])
    if len(sp) != 3:
        raise ValueError('spacing: three values (x, y, z)')
    labels = [int(x) for x in labels]
    hausdorff = percentile is not None
    dev = seg_b.device
    outs = tuple(torch.empty(C, len(labels), device=dev, dtype=torch.float64) for _ in range(3 if hausdorff else 1))
    partials = torch.empty(_lib.ASD_PARTIALS_DOUBLES, device=dev, dtype=torch.float64)
    counters = torch.empty(_lib.SD_COUNTERS if hausdorff else _lib.ASD_MAX_BOXES, device=dev, dtype=torch.int32)
    budget = max(1, int(workspace_bytes) // 4)
    for l0 in range(0, len(labels), 32):
        chunk = labels[l0:l0 + 32]
        n = len(chunk)
        lab = (ctypes.c_int * n)(*chunk)
        boxes = torch.empty(C, n, 8, device=dev, dtype=torch.int32)
        _lib.check(lib.irs_surface_boxes(_lib.ptr(seg_a), stride, _lib.ptr(seg_b), lab, n, _lib.ptr(boxes), C, D, H, W,
                                         _lib.stream()))
        bh = boxes.cpu().view(-1, 8)
        ext = (bh[:, 3:6] - bh[:, 0:3] + 1).long()
        # workspace floats per pair: the two distance channels over the box, plus |A| + |B| for the Hausdorff lists
        per_pair = 2 * ext.prod(1) + (bh[:, 6].long() + bh[:, 7].long() if hausdorff else 0)
        need = torch.where((bh[:, 6] > 0) & (bh[:, 7] > 0), per_pair, torch.zeros_like(ext[:, 0])).tolist()
        batches, begin, acc = [], 0, 0   # consecutive pairs whose workspace fits the budget
        for p, f in enumerate(need):
            if acc + f > budget and p > begin:
                batches.append((begin, p, acc))
                begin, acc = p, 0
            acc += f
        batches.append((begin, len(need), acc))
        ws = torch.empty(max(1, max(b[2] for b in batches)), device=dev, dtype=torch.float32)
        res = tuple(torch.empty(C, n, device=dev, dtype=torch.float64) for _ in outs)
        host_boxes = bh.contiguous().numpy()
        for b, e, f in batches:
            common = (_lib.ptr(seg_a), stride, _lib.ptr(seg_b), lab, n, host_boxes.ctypes.data_as(ctypes.c_void_p), sp)
            scratch = (_lib.ptr(ws), ws.numel(), _lib.ptr(partials), _lib.ptr(counters))
            if hausdorff:
                _lib.check(lib.irs_surface_distances(*common, percentile, b, e, *scratch, *(_lib.ptr(r) for r in res),
                                                     C, D, H, W, _lib.stream()))
            else:
                _lib.check(lib.irs_average_surface_distance(*common, b, e, *scratch, _lib.ptr(res[0]), C, D, H, W,
                                                            _lib.stream()))
        for o, r in zip(outs, res):
            o[:, l0:l0 + n] = r
    return outs


def _mask_u8(mask, V):
    if mask.numel() != V:
        raise ValueError(f'mask must hold the {V} voxels of the volume')
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    if mask.dtype != torch.uint8:
        raise NotImplementedError('bool / uint8 masks only')
    return mask.contiguous()


def jacobian_scratch(C, device):
    """(partials, counters) of irs_jacobian_update for C chains (also enough for irs_jacobian_posterior); the counters start at
    zero and every call leaves them zero, so a caller may keep the pair for all its updates"""
    partials = torch.empty(2 * C * _lib.JACOBIAN_REDUCE_BLOCKS, device=device, dtype=torch.float64)
    return partials, torch.zeros(C + 1, device=device, dtype=torch.int64)


def jacobian_update(T, mask, count_before, folds, mean, m2, scratch=None):
    """
    Fold the log det J of the C transformations T (C,3,D,H,W) into the Jacobian-posterior accumulators of `count_before` earlier
    samples, in place: folds (D,H,W) int32 = folded samples (log det J not finite: det <= 0, NaN or inf), mean / m2 (D,H,W) fp32
    = Welford of log det J over the finite samples.  mask (D,H,W) bool / uint8.  Returns the (C,4) fp64 device tensor of this
    sample over the mask, per chain: finite voxels, folded voxels, sum of log det J and of its square over the finite voxels.
    scratch: jacobian_scratch(C, device), or None for a fresh pair.
    """
    lib = _lib.load()
    _lib.require_cuda(T, mask, folds, mean, m2)
    _f32(T, mean, m2)
    C, D, H, W = _dims(T)
    V = D * H * W
    if T.shape[1] != 3:
        raise ValueError('T must be (C,3,D,H,W)')
    if folds.dtype != torch.int32:
        raise NotImplementedError('int32 folds only')
    if folds.numel() != V or mean.numel() != V or m2.numel() != V:
        raise ValueError(f'folds, mean and m2 must hold the {V} voxels of T')
    m8 = _mask_u8(mask, V)
    partials, counters = jacobian_scratch(C, T.device) if scratch is None else scratch
    if partials.numel() < 2 * C * _lib.JACOBIAN_REDUCE_BLOCKS or counters.numel() < C + 1:
        raise ValueError(f'scratch too small for {C} chains')
    stats = torch.empty(C, 4, device=T.device, dtype=torch.float64)
    _lib.check(lib.irs_jacobian_update(_lib.ptr(T), _lib.ptr(m8), C, D, H, W, float(count_before), _lib.ptr(folds),
                                       _lib.ptr(mean), _lib.ptr(m2), _lib.ptr(stats), _lib.ptr(partials), _lib.ptr(counters),
                                       _lib.stream()))
    return stats


def jacobian_posterior(folds, mean, m2, n, mask):
    """
    The Jacobian posterior from the accumulators of n samples (ops.jacobian_update):
      p_fold   (D,H,W) fp32  (float)folds / (float)n
      mean     (D,H,W) fp32  mean of log det J over the n_v = n - folds finite samples, NaN where n_v = 0
      std      (D,H,W) fp32  sqrt(m2 / (n_v - 1)), unbiased like torch.std, NaN where n_v < 2
      summary  dict over the voxels of mask: 'sum_folds' (exact; / n = expected number of folded voxels), 'voxels_ever_folded'
               (folds > 0), 'voxels_folded_in_majority' (2 folds > n), 'voxels_finite' (n_v >= 1), 'voxels_finite_2'
               (n_v >= 2), 'mask_voxels', 'mean_log_det_J' (mean of the mean map over n_v >= 1), 'mean_std_log_det_J' (mean
               of the std map over n_v >= 2) -- one host read
    """
    lib = _lib.load()
    _lib.require_cuda(folds, mean, m2, mask)
    _f32(mean, m2)
    if folds.dtype != torch.int32:
        raise NotImplementedError('int32 folds only')
    V = folds.numel()
    if mean.numel() != V or m2.numel() != V:
        raise ValueError('folds, mean and m2 must have the same number of voxels')
    m8 = _mask_u8(mask, V)
    dev = folds.device
    p_fold, mean_out, std_out = (torch.empty(folds.shape, device=dev, dtype=torch.float32) for _ in range(3))
    partials, counters = jacobian_scratch(1, dev)
    summary = torch.empty(_lib.JACOBIAN_SUMMARY_WORDS, device=dev, dtype=torch.int64)
    _lib.check(lib.irs_jacobian_posterior(_lib.ptr(folds), _lib.ptr(mean), _lib.ptr(m2), int(n), V, _lib.ptr(m8),
                                          _lib.ptr(p_fold), _lib.ptr(mean_out), _lib.ptr(std_out), _lib.ptr(partials),
                                          _lib.ptr(counters), _lib.ptr(summary), _lib.stream()))
    s = summary.cpu()
    words = [int(x) for x in s]
    means = s[5:7].view(torch.float64).tolist()
    summ = {'sum_folds': words[0], 'voxels_ever_folded': words[1], 'voxels_folded_in_majority': words[2],
            'voxels_finite': words[3], 'voxels_finite_2': words[4], 'mask_voxels': words[7],
            'mean_log_det_J': means[0], 'mean_std_log_det_J': means[1]}
    return p_fold, mean_out, std_out, summ


def _landmarks_host(x, name):
    """(P, 3) float64 host copy of a landmark table"""
    x = torch.as_tensor(x).detach().to('cpu', torch.float64)
    if x.dim() != 2 or x.shape[1] != 3 or x.shape[0] < 1:
        raise ValueError(f'{name} must be a (P, 3) table of (x, y, z) voxel coordinates with P >= 1')
    return x.contiguous()


def landmark_spacing(spacing):
    """the three (x, y, z) spacings in mm as floats, each finite and > 0"""
    sp = [float(s) for s in torch.as_tensor(spacing, dtype=torch.float64).reshape(-1).tolist()]
    if len(sp) != 3 or not all(math.isfinite(s) and s > 0.0 for s in sp):
        raise ValueError(f'spacing must be three finite positive (x, y, z) values, got {sp}')
    return sp


def check_landmarks(fixed_landmarks, moving_landmarks, dims):
    """host checks of a pair of landmark tables for a (D, H, W) grid: (P, 3) each with the same P; every fixed coordinate
    finite and in [0, n_a - 1] of its axis (x = W, y = H, z = D); every moving coordinate finite.  Returns both as (P, 3)
    float64 host tensors."""
    p, q = _landmarks_host(fixed_landmarks, 'fixed_landmarks'), _landmarks_host(moving_landmarks, 'moving_landmarks')
    if p.shape != q.shape:
        raise ValueError(f'fixed and moving landmarks must correspond row by row: {tuple(p.shape)} vs {tuple(q.shape)}')
    D, H, W = dims
    hi = torch.tensor([W - 1, H - 1, D - 1], dtype=torch.float64)
    if not bool(torch.isfinite(p).all()) or bool((p < 0).any()) or bool((p > hi).any()):
        raise ValueError(f'fixed landmarks must be finite (x, y, z) voxel coordinates inside [0, {W - 1}] x [0, {H - 1}] x '
                         f'[0, {D - 1}]')
    if not bool(torch.isfinite(q).all()):
        raise ValueError('moving landmarks must be finite')
    return p, q


def landmark_map(T, fixed_landmarks, moving_landmarks, spacing):
    """
    Predicted moving positions and target registration errors of the P landmark pairs under the C transformations T
    (C,3,D,H,W) fp32 (normalised sampling grids, SGLDSampler.transformation()).  Landmarks are (P,3) (x, y, z) voxel
    coordinates, row i of the fixed ones corresponding to row i of the moving ones; spacing (x, y, z) in mm.  The ranges are
    checked here on the host (check_landmarks).  Returns pred (C,P,3) fp64 (moving voxel units: where the warp samples the
    moving image for the fixed landmark) and tre (C,P) fp64 in mm, device tensors (irs_landmark_map).
    """
    lib = _lib.load()
    _lib.require_cuda(T)
    _f32(T)
    C, D, H, W = _dims(T)
    if T.shape[1] != 3:
        raise ValueError('T must be (C,3,D,H,W)')
    p, q = check_landmarks(fixed_landmarks, moving_landmarks, (D, H, W))
    sp = landmark_spacing(spacing)
    P = p.shape[0]
    pd, qd = p.to(T.device), q.to(T.device)
    pred = torch.empty(C, P, 3, device=T.device, dtype=torch.float64)
    tre = torch.empty(C, P, device=T.device, dtype=torch.float64)
    _lib.check(lib.irs_landmark_map(_lib.ptr(T), C, D, H, W, _lib.ptr(pd), _lib.ptr(qd), P, (ctypes.c_double * 3)(*sp),
                                    _lib.ptr(pred), _lib.ptr(tre), _lib.stream()))
    return pred, tre


def landmark_update(pred, tre, count_before, acc):
    """
    Fold the C samples pred (C,P,3) / tre (C,P) fp64 (landmark_map) into the landmark accumulators acc (P,11) fp64 of
    `count_before` earlier samples, in place, chains in index order: per landmark the Welford mean (3) and co-moments
    (xx, xy, xz, yy, yz, zz) of the predicted position and the Welford mean / M2 of the TRE.  Returns the (C,3) fp64 device
    rows of this sample per chain, landmarks in index order: sum TRE, sum TRE^2, max TRE (irs_landmark_update).
    """
    lib = _lib.load()
    _lib.require_cuda(pred, tre, acc)
    if pred.dtype != torch.float64 or tre.dtype != torch.float64 or acc.dtype != torch.float64:
        raise NotImplementedError('fp64 landmark tensors only')
    if pred.dim() != 3 or pred.shape[2] != 3:
        raise ValueError('pred must be (C,P,3)')
    C, P = pred.shape[:2]
    if tuple(tre.shape) != (C, P) or tuple(acc.shape) != (P, _lib.LANDMARK_ACC):
        raise ValueError(f'tre must be ({C}, {P}) and acc ({P}, {_lib.LANDMARK_ACC})')
    stats = torch.empty(C, 3, device=pred.device, dtype=torch.float64)
    _lib.check(lib.irs_landmark_update(_lib.ptr(pred), _lib.ptr(tre), C, P, float(count_before), _lib.ptr(acc),
                                       _lib.ptr(stats), _lib.stream()))
    return stats


def landmark_posterior(acc, n, moving_landmarks, spacing):
    """
    The landmark posterior from the accumulators acc (P,11) of n >= 1 samples: a (P,16) fp64 device table per landmark
    (irs_landmark_posterior): [0:3] mean predicted position (moving voxels), [3] TRE of the mean, [4] E[TRE], and for n >= 2
    (NaN for n = 1) [5] std of TRE, [6:12] covariance (xx, xy, xz, yy, yz, zz) in mm^2, [12:15] principal standard deviations
    in mm (descending), [15] squared Mahalanobis distance of the moving landmark from the mean (+inf for a singular covariance).
    """
    lib = _lib.load()
    _lib.require_cuda(acc)
    if acc.dtype != torch.float64 or acc.dim() != 2 or acc.shape[1] != _lib.LANDMARK_ACC:
        raise ValueError(f'acc must be a (P, {_lib.LANDMARK_ACC}) fp64 tensor')
    P = acc.shape[0]
    q = _landmarks_host(moving_landmarks, 'moving_landmarks')
    if q.shape[0] != P or not bool(torch.isfinite(q).all()):
        raise ValueError(f'moving_landmarks must be {P} finite rows')
    sp = landmark_spacing(spacing)
    out = torch.empty(P, _lib.LANDMARK_COLS, device=acc.device, dtype=torch.float64)
    _lib.check(lib.irs_landmark_posterior(_lib.ptr(acc), _lib.ptr(q.to(acc.device)), P, int(n), (ctypes.c_double * 3)(*sp),
                                          _lib.ptr(out), _lib.stream()))
    return out
