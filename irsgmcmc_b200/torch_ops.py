"""
The operators of the SGLD registration step as PyTorch custom ops: ``torch.ops.irsgmcmc.*``.

Each op is a thin ``torch.library`` registration over the C ABI of libirsgmcmc.so (through ``ops.py``): a CUDA kernel
only -- the dispatcher itself refuses CPU tensors ("Could not run 'irsgmcmc::...' with arguments from the 'CPU' backend") --
a fake (meta) implementation for shape propagation under FakeTensorMode / torch.compile tracing, and the autograd formula,
which calls the adjoint op (the closed forms of SURVEY Appendix A, no scatter atomics).

    reference call site                                                   op
    RegistrationModule.forward, float branch (utils/registration.py:29)   irsgmcmc::warp3d, ::warp3d_bwd_grid
    RegistrationModule.forward, seg / mask  (utils/registration.py:20)    irsgmcmc::warp3d_nearest
    SVF_3D.forward + autograd (utils/transformation.py:63-76)             irsgmcmc::svf_exp, ::svf_exp_bwd
    SobolevGrad.apply (utils/functions.py:98-109)                         irsgmcmc::sobolev_smooth (backward = identity)
    GMM.map, one image side (model/loss.py:102-111)                       irsgmcmc::lcc_normalise, ::lcc_normalise_bwd
    RegLoss.forward energy (model/loss.py:152-161)                        irsgmcmc::reg_energy, ::reg_energy_grad
    Cubic_B_spline_FFD_3D.forward (utils/transformation.py:132-152)       irsgmcmc::ffd, ::ffd_adjoint
    SGLD.apply + SobolevGrad.apply (utils/functions.py:76-109)            irsgmcmc::langevin_proposal (Philox or explicit noise)
    GMM.log_pdf + autograd (model/loss.py:87-93)                          irsgmcmc::gmm_log_pdf, ::gmm_log_pdf_param_grads
    rescale_residuals + calc_VD_factor (utils/util.py:330-347,446-485)    irsgmcmc::vd_factor
    calc_posterior_statistics (utils/util.py:114-120)                     irsgmcmc::welford_update (in place), ::welford_std
    (no reference counterpart: convergence check of the chains)           irsgmcmc::split_rhat
    calc_no_non_diffeomorphic_voxels (utils/util.py:209-212)              irsgmcmc::log_det_jacobian
    calc_DSC_GPU (utils/util.py:123-148)                                  irsgmcmc::dice_counts
    calc_metrics, ASD part (utils/util.py:171-176)                        irsgmcmc::average_surface_distance
    (no reference counterpart: Hausdorff distance and HD95, calc_HD_GPU)   irsgmcmc::surface_distances
    (no reference counterpart: posterior of the warped segmentation)      irsgmcmc::label_counts_update (in place), ::label_posterior
    (no reference counterpart: TRE and landmark posterior, calc_TRE_GPU)   irsgmcmc::landmark_map, ::landmark_update (in place),
                                                                          ::landmark_posterior
    Trainer._SGLD_transition (trainer/trainer.py:291-356)                 irsgmcmc::sgld_step (the fused transition, in place)

The drop-in modules (utils/, model/) and the fused sampler use the same launchers; this module adds the dispatcher-visible
surface the north star asks for and nothing else.
"""
from typing import Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib, ops

_NS = 'irsgmcmc'


def _op(name, **kw):
    return torch.library.custom_op(f'{_NS}::{name}', mutates_args=(), device_types='cuda', **kw)


# ---- warps ------------------------------------------------------------------------------------------------------------
@_op('warp3d')
def warp3d(img: Tensor, T: Tensor, jitter_unit: Optional[Tensor], alpha: float) -> Tensor:
    return ops.warp3d(img.contiguous(), T.contiguous(), None if jitter_unit is None else jitter_unit.contiguous(), alpha)


@warp3d.register_fake
def _(img, T, jitter_unit, alpha):
    return T.new_empty(T.shape[0], 1, T.shape[2], T.shape[3], T.shape[4])


@_op('warp3d_bwd_grid')
def warp3d_bwd_grid(img: Tensor, T: Tensor, g_out: Tensor, jitter_unit: Optional[Tensor], alpha: float) -> Tensor:
    return ops.warp3d_bwd_grid(img.contiguous(), T.contiguous(), g_out.contiguous(),
                               None if jitter_unit is None else jitter_unit.contiguous(), alpha)


@warp3d_bwd_grid.register_fake
def _(img, T, g_out, jitter_unit, alpha):
    return torch.empty_like(T)


def _warp3d_setup(ctx, inputs, output):
    img, T, jitter_unit, alpha = inputs
    ctx.has_jitter, ctx.alpha = jitter_unit is not None, alpha
    ctx.save_for_backward(*((img, T, jitter_unit) if ctx.has_jitter else (img, T)))


def _warp3d_backward(ctx, g):
    saved = ctx.saved_tensors
    jitter_unit = saved[2] if ctx.has_jitter else None
    # like the reference, only the grid receives a gradient (the moving image is data: utils/registration.py:29-30)
    return None, torch.ops.irsgmcmc.warp3d_bwd_grid(saved[0], saved[1], g, jitter_unit, ctx.alpha), None, None


warp3d.register_autograd(_warp3d_backward, setup_context=_warp3d_setup)


@_op('warp3d_nearest')
def warp3d_nearest(seg: Tensor, T: Tensor) -> Tensor:
    return ops.warp3d_nearest(seg.contiguous(), T.contiguous())


@warp3d_nearest.register_fake
def _(seg, T):
    return seg.new_empty(T.shape[0], 1, T.shape[2], T.shape[3], T.shape[4])


# ---- stationary velocity field ------------------------------------------------------------------------------------------
@_op('svf_exp')
def svf_exp(v: Tensor, n_steps: int) -> Tuple[Tensor, Tensor, Tensor]:
    """(displacement in voxels, history u_1..u_n, max |u_k| workspace) of scaling and squaring"""
    hist, maxabs = ops.svf_exp_fwd(v.contiguous(), n_steps)
    workspace = maxabs._base if maxabs._base is not None else maxabs   # per-step maxima followed by the per-cell maps
    return hist[-1].clone(), hist, workspace


@svf_exp.register_fake
def _(v, n_steps):
    C, D, H, W = v.shape[0], v.shape[2], v.shape[3], v.shape[4]
    n_max = int(_lib.load().irs_svf_maxabs_floats(int(C), int(D), int(H), int(W), int(n_steps)))
    return torch.empty_like(v), v.new_empty(n_steps, *v.shape), v.new_empty(n_max)


@_op('svf_exp_bwd')
def svf_exp_bwd(v: Tensor, hist: Tensor, maxabs: Tensor, g_u: Tensor, gather_radius_max: int) -> Tensor:
    return ops.svf_exp_bwd(v.contiguous(), hist, maxabs, g_u.contiguous(), gather_radius_max)


@svf_exp_bwd.register_fake
def _(v, hist, maxabs, g_u, gather_radius_max):
    return torch.empty_like(v)


def _svf_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], output[1], output[2])
    ctx.set_materialize_grads(False)


def _svf_backward(ctx, g_disp, g_hist, g_maxabs):
    v, hist, maxabs = ctx.saved_tensors
    if g_disp is None:
        return None, None
    return torch.ops.irsgmcmc.svf_exp_bwd(v, hist, maxabs, g_disp, 3), None


svf_exp.register_autograd(_svf_backward, setup_context=_svf_setup)


# ---- Sobolev smoothing --------------------------------------------------------------------------------------------------
@_op('sobolev_smooth')
def sobolev_smooth(v: Tensor, taps: Sequence[float]) -> Tensor:
    from .utils.functions import langevin_sobolev
    return langevin_sobolev(v.contiguous(), None, 0.0, [float(t) for t in taps])


@sobolev_smooth.register_fake
def _(v, taps):
    return torch.empty_like(v)


# SobolevGrad.backward passes the gradient through unchanged (reference utils/functions.py:107-109; SURVEY Appendix C)
sobolev_smooth.register_autograd(lambda ctx, g: (g, None), setup_context=lambda ctx, inputs, output: None)


# ---- LCC normalisation ----------------------------------------------------------------------------------------------------
@_op('lcc_normalise')
def lcc_normalise(im: Tensor, s: int) -> Tuple[Tensor, Tensor, Tensor]:
    """(zn, a, rs): a = I - Box(I)/k^3, rs = 1/sqrt(Box(a^2)/k^3 + 1e-10), zn = a rs, k = 2 s + 1"""
    return ops.lcc_normalise(im.contiguous(), s)


@lcc_normalise.register_fake
def _(im, s):
    return torch.empty_like(im), torch.empty_like(im), torch.empty_like(im)


@_op('lcc_normalise_bwd')
def lcc_normalise_bwd(g_zn: Tensor, a: Tensor, rs: Tensor, s: int) -> Tensor:
    return ops.lcc_normalise_bwd(g_zn.contiguous(), a, rs, s)


@lcc_normalise_bwd.register_fake
def _(g_zn, a, rs, s):
    return torch.empty_like(a)


def _lcc_setup(ctx, inputs, output):
    ctx.s = inputs[1]
    ctx.save_for_backward(output[1], output[2])
    ctx.set_materialize_grads(False)


def _lcc_backward(ctx, g_zn, g_a, g_rs):
    if g_a is not None or g_rs is not None:
        raise NotImplementedError('irsgmcmc::lcc_normalise: only zn is differentiable')
    if g_zn is None:
        return None, None
    a, rs = ctx.saved_tensors
    return torch.ops.irsgmcmc.lcc_normalise_bwd(g_zn, a, rs, ctx.s), None


lcc_normalise.register_autograd(_lcc_backward, setup_context=_lcc_setup)


# ---- regulariser energy -----------------------------------------------------------------------------------------------------
@_op('reg_energy')
def reg_energy(v: Tensor) -> Tensor:
    """sum of squared forward differences per batch entry, float64 (C,)"""
    return ops.reg_energy(v.contiguous())


@reg_energy.register_fake
def _(v):
    return v.new_empty(v.shape[0], dtype=torch.float64)


@_op('reg_energy_grad')
def reg_energy_grad(v: Tensor, coef: Tensor) -> Tensor:
    """coef[c] * d energy_c / d v"""
    return ops.reg_energy_grad(v.contiguous(), coef.contiguous())


@reg_energy_grad.register_fake
def _(v, coef):
    return torch.empty_like(v)


def _energy_backward(ctx, g_y):
    v, = ctx.saved_tensors
    return torch.ops.irsgmcmc.reg_energy_grad(v, g_y.double())


reg_energy.register_autograd(_energy_backward, setup_context=lambda ctx, inputs, output: ctx.save_for_backward(inputs[0]))


# ---- cubic B-spline FFD -----------------------------------------------------------------------------------------------------
@_op('ffd')
def ffd(cp: Tensor, kernel_d: Sequence[float], kernel_h: Sequence[float], kernel_w: Sequence[float], cps: Sequence[int],
        dims: Sequence[int]) -> Tensor:
    return ops.ffd_fwd(cp.contiguous(), [list(kernel_d), list(kernel_h), list(kernel_w)], list(cps), list(dims))


@ffd.register_fake
def _(cp, kernel_d, kernel_h, kernel_w, cps, dims):
    return cp.new_empty(cp.shape[0], 3, dims[0], dims[1], dims[2])


@_op('ffd_adjoint')
def ffd_adjoint(g_dense: Tensor, kernel_d: Sequence[float], kernel_h: Sequence[float], kernel_w: Sequence[float],
                cps: Sequence[int], grid: Sequence[int]) -> Tensor:
    return ops.ffd_bwd(g_dense.contiguous(), [list(kernel_d), list(kernel_h), list(kernel_w)], list(cps), list(grid))


@ffd_adjoint.register_fake
def _(g_dense, kernel_d, kernel_h, kernel_w, cps, grid):
    return g_dense.new_empty(g_dense.shape[0], 3, grid[0], grid[1], grid[2])


def _ffd_setup(ctx, inputs, output):
    cp, ctx.kd, ctx.kh, ctx.kw, ctx.cps, _ = inputs
    ctx.grid = [int(n) for n in cp.shape[2:]]


def _ffd_backward(ctx, g):
    return torch.ops.irsgmcmc.ffd_adjoint(g, ctx.kd, ctx.kh, ctx.kw, ctx.cps, ctx.grid), None, None, None, None, None


ffd.register_autograd(_ffd_backward, setup_context=_ffd_setup)



# ---- Langevin proposal + Sobolev smoothing ------------------------------------------------------------------------------------
@_op('langevin_proposal')
def langevin_proposal(v: Tensor, sigma: Optional[Tensor], eps: Optional[Tensor], coef: float, taps: Sequence[float], seed: int,
                      iteration: int, chain0: int) -> Tensor:
    """S * (v + coef sigma eps): eps explicit, or Philox4x32-10 N(0,1) keyed (seed, chain0 + chain, iteration, voxel)"""
    from .utils.functions import langevin_sobolev
    return langevin_sobolev(v.contiguous(), None if sigma is None else sigma.contiguous(), coef, [float(t) for t in taps],
                            None if eps is None else eps.contiguous(), seed, iteration, chain0)


@langevin_proposal.register_fake
def _(v, sigma, eps, coef, taps, seed, iteration, chain0):
    return torch.empty_like(v)


def _langevin_setup(ctx, inputs, output):
    ctx.has_sigma = inputs[1] is not None
    if ctx.has_sigma:
        ctx.save_for_backward(inputs[1])


def _langevin_backward(ctx, g):
    # SGLD.backward = sigma^2 * g (utils/functions.py:82-84), SobolevGrad.backward = identity (:107-109)
    g_v = g * ctx.saved_tensors[0] ** 2 if ctx.has_sigma else g
    return g_v, None, None, None, None, None, None, None


langevin_proposal.register_autograd(_langevin_backward, setup_context=_langevin_setup)


# ---- mixture log-density, virtual decimation ------------------------------------------------------------------------------------
@_op('gmm_log_pdf')
def gmm_log_pdf(z: Tensor, log_std: Tensor, logits: Tensor) -> Tuple[Tensor, Tensor]:
    """(log pdf, d log pdf / dz) per element of z; the mixture parameters may live on either device (K scalars)"""
    logp, dz, _ = ops.gmm_log_pdf(z.reshape(-1).contiguous(), log_std, logits, want_dz=True)
    return logp.view(z.shape), dz.view(z.shape)


@gmm_log_pdf.register_fake
def _(z, log_std, logits):
    return torch.empty_like(z), torch.empty_like(z)


@_op('gmm_log_pdf_param_grads')
def gmm_log_pdf_param_grads(z: Tensor, log_std: Tensor, logits: Tensor, weights: Tensor) -> Tensor:
    """float64 (16,): sum_i w_i d log pdf_i / d log_std_k in [0, K), sum_i w_i rho_k(z_i) in [8, 8 + K)"""
    _, _, gp = ops.gmm_log_pdf(z.reshape(-1).contiguous(), log_std, logits, weights=weights.reshape(-1).contiguous(),
                               want_param_grads=True)
    return gp


@gmm_log_pdf_param_grads.register_fake
def _(z, log_std, logits, weights):
    return z.new_empty(2 * _lib.MAX_K, dtype=torch.float64)


def _gmm_setup(ctx, inputs, output):
    z, log_std, logits = inputs
    ctx.save_for_backward(z, output[1], log_std.detach().clone(), logits.detach().clone())
    ctx.set_materialize_grads(False)


def _gmm_backward(ctx, g_logp, g_dz):
    if g_dz is not None:
        raise NotImplementedError('irsgmcmc::gmm_log_pdf: only the log-density is differentiable')
    if g_logp is None:
        return None, None, None
    z, dz, log_std, logits = ctx.saved_tensors
    K = log_std.numel()
    g_z = g_logp * dz if ctx.needs_input_grad[0] else None
    g_ls = g_lg = None
    if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
        gp = torch.ops.irsgmcmc.gmm_log_pdf_param_grads(z, log_std, logits, g_logp.contiguous())
        pi = torch.softmax(logits + 1e-2, dim=0)           # K scalars; d logp / d logits_j = rho_j - pi_j
        g_ls = gp[:K].to(log_std.dtype).to(log_std.device)
        g_lg = (gp[8:8 + K].to(logits.device) - pi.double() * g_logp.double().sum().to(logits.device)).to(logits.dtype)
    return g_z, g_ls, g_lg


gmm_log_pdf.register_autograd(_gmm_backward, setup_context=_gmm_setup)


@_op('vd_factor')
def vd_factor(z: Tensor, mask: Tensor, log_std: Tensor, logits: Tensor) -> Tensor:
    """virtual decimation factor of one chain, float64 scalar tensor"""
    return ops.vd_factor(z.contiguous(), mask.contiguous(), log_std, logits).reshape(())


@vd_factor.register_fake
def _(z, mask, log_std, logits):
    return z.new_empty((), dtype=torch.float64)


# ---- posterior moments ------------------------------------------------------------------------------------------------------------
@torch.library.custom_op(f'{_NS}::welford_update', mutates_args=('mean', 'm2'), device_types='cuda')
def welford_update(sample: Tensor, count_before: int, mean: Tensor, m2: Tensor) -> None:
    """fold sample[0..n) into the running (mean, M2) that already hold count_before samples"""
    ops.welford_update(sample.contiguous(), count_before, mean, m2)


@welford_update.register_fake
def _(sample, count_before, mean, m2):
    return None


@_op('welford_std')
def welford_std(m2: Tensor, count: int) -> Tensor:
    """unbiased standard deviation sqrt(M2 / (count - 1)) like torch.std (utils/util.py:117)"""
    return ops.welford_std(m2.contiguous(), count)


@welford_std.register_fake
def _(m2, count):
    return torch.empty_like(m2)


@_op('split_rhat')
def split_rhat(mean: Tensor, m2: Tensor, n: int, mask: Tensor) -> Tuple[Tensor, Tensor]:
    """split R-hat of the n_seq sequences given (no collectives): per-sequence Welford mean / M2 (n_seq, K, D, H, W) fp32 of n
    draws each, mask (D, H, W) -> (R-hat (K, D, H, W) fp32, summary (K, 3) fp64: max R-hat, voxels > 1.01, voxels > 1.1 over
    the mask)"""
    rhat, summary, _ = ops.split_rhat(mean.contiguous(), m2.contiguous(), n, mask.contiguous(), distributed=False)
    return rhat, summary


@split_rhat.register_fake
def _(mean, m2, n, mask):
    return mean.new_empty(mean.shape[1:]), mean.new_empty(mean.shape[1], 3, dtype=torch.float64)


# ---- per-sample evaluation ----------------------------------------------------------------------------------------------------------
@_op('log_det_jacobian')
def log_det_jacobian(T: Tensor) -> Tuple[Tensor, Tensor]:
    """(number of folded voxels per sample int32 (C,), log det J (C,D,H,W)) of a normalised transformation (C,3,D,H,W)"""
    return ops.log_det_jacobian(T.contiguous())


@log_det_jacobian.register_fake
def _(T):
    return T.new_empty(T.shape[0], dtype=torch.int32), T.new_empty(T.shape[0], T.shape[2], T.shape[3], T.shape[4])


@_op('dice_counts')
def dice_counts(seg_a: Tensor, seg_b: Tensor, labels: Sequence[int]) -> Tensor:
    """int32 (C, n_labels, 3): |A = l|, |B = l|, |A = l and B = l| (seg_a may be one volume shared by all samples)"""
    return ops.dice_counts(seg_a.contiguous(), seg_b.contiguous(), list(labels))


@dice_counts.register_fake
def _(seg_a, seg_b, labels):
    return seg_b.new_empty(seg_b.shape[0], len(labels), 3, dtype=torch.int32)


@_op('average_surface_distance')
def average_surface_distance(seg_a: Tensor, seg_b: Tensor, labels: Sequence[int], spacing: Sequence[float]) -> Tensor:
    """float64 (C, n_labels): average surface distance of seg_a == l and seg_b[c] == l, spacing (x, y, z); inf when either is
    empty (seg_a may be one volume shared by all samples)"""
    return ops.average_surface_distance(seg_a.contiguous(), seg_b.contiguous(), list(labels), list(spacing))


@average_surface_distance.register_fake
def _(seg_a, seg_b, labels, spacing):
    return seg_b.new_empty(seg_b.shape[0], len(labels), dtype=torch.float64)


@_op('surface_distances')
def surface_distances(seg_a: Tensor, seg_b: Tensor, labels: Sequence[int], spacing: Sequence[float],
                      percentile: float = 95.0) -> Tuple[Tensor, Tensor, Tensor]:
    """float64 (asd, hd, hd_q), each (C, n_labels): average surface distance, Hausdorff distance and the larger of the two
    directed percentiles (numpy's method 'linear', 95: HD95) of seg_a == l and seg_b[c] == l from one distance transform"""
    return ops.surface_distances(seg_a.contiguous(), seg_b.contiguous(), list(labels), list(spacing), percentile)


@surface_distances.register_fake
def _(seg_a, seg_b, labels, spacing, percentile=95.0):
    return tuple(seg_b.new_empty(seg_b.shape[0], len(labels), dtype=torch.float64) for _ in range(3))


# ---- posterior of the warped segmentation ---------------------------------------------------------------------------------
@torch.library.custom_op(f'{_NS}::label_counts_update', mutates_args=('counts',), device_types='cuda')
def label_counts_update(seg: Tensor, labels: Sequence[int], counts: Tensor) -> None:
    """counts (L, D, H, W) int32 += per label, the number of the C int16 segmentations seg (C, 1, D, H, W) carrying it"""
    ops.label_counts_update(seg.contiguous(), list(labels), counts)


@label_counts_update.register_fake
def _(seg, labels, counts):
    return None


@_op('label_posterior')
def label_posterior(counts: Tensor, n: int, labels: Sequence[int], seg_fixed: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor,
                                                                                                         Tensor]:
    """(probability (L, D, H, W) fp32, majority label (1, 1, D, H, W) int16, entropy (1, D, H, W) fp32, summary (L, 3) int64)
    from the label counts of n segmentations (ops.label_posterior)"""
    return ops.label_posterior(counts.contiguous(), n, list(labels), None if seg_fixed is None else seg_fixed.contiguous())


@label_posterior.register_fake
def _(counts, n, labels, seg_fixed):
    L, D, H, W = counts.shape
    return (counts.new_empty(L, D, H, W, dtype=torch.float32), counts.new_empty(1, 1, D, H, W, dtype=torch.int16),
            counts.new_empty(1, D, H, W, dtype=torch.float32), counts.new_empty(L, 3, dtype=torch.int64))


# ---- landmark registration error and landmark posterior ---------------------------------------------------------------------------
@_op('landmark_map')
def landmark_map(T: Tensor, fixed_landmarks: Tensor, moving_landmarks: Tensor, spacing: Sequence[float]) -> Tuple[Tensor, Tensor]:
    """(pred (C, P, 3) fp64 moving voxel positions, tre (C, P) fp64 in mm) of the (P, 3) landmark pairs under the C
    transformations T (ops.landmark_map)"""
    return ops.landmark_map(T.contiguous(), fixed_landmarks, moving_landmarks, list(spacing))


@landmark_map.register_fake
def _(T, fixed_landmarks, moving_landmarks, spacing):
    C, P = T.shape[0], fixed_landmarks.shape[0]
    return T.new_empty(C, P, 3, dtype=torch.float64), T.new_empty(C, P, dtype=torch.float64)


@torch.library.custom_op(f'{_NS}::landmark_update', mutates_args=('acc',), device_types='cuda')
def landmark_update(pred: Tensor, tre: Tensor, count_before: int, acc: Tensor) -> Tensor:
    """acc (P, 11) fp64 += the C samples pred / tre in chain order (Welford); returns the (C, 3) per-chain rows sum TRE,
    sum TRE^2, max TRE (ops.landmark_update)"""
    return ops.landmark_update(pred.contiguous(), tre.contiguous(), count_before, acc)


@landmark_update.register_fake
def _(pred, tre, count_before, acc):
    return pred.new_empty(pred.shape[0], 3, dtype=torch.float64)


@_op('landmark_posterior')
def landmark_posterior(acc: Tensor, n: int, moving_landmarks: Tensor, spacing: Sequence[float]) -> Tensor:
    """(P, 16) fp64 per-landmark posterior table from the accumulators of n samples (ops.landmark_posterior)"""
    return ops.landmark_posterior(acc.contiguous(), n, moving_landmarks, list(spacing))


@landmark_posterior.register_fake
def _(acc, n, moving_landmarks, spacing):
    return acc.new_empty(acc.shape[0], _lib.LANDMARK_COLS, dtype=torch.float64)


# ---- the fused transition -------------------------------------------------------------------------------------------------------------
_SAMPLERS = {}


def register_sampler(sampler) -> int:
    """handle of an SGLDSampler for irsgmcmc::sgld_step (the op mutates that sampler's buffers)"""
    handle = id(sampler)
    _SAMPLERS[handle] = sampler
    return handle


@torch.library.custom_op(f'{_NS}::sgld_step', mutates_args=('v', 'hyper', 'stats'), device_types='cuda')
def sgld_step(v: Tensor, hyper: Tensor, stats: Tensor, handle: int, n: int) -> None:
    """n fused SGLD transitions (irs_sgld_step) of the sampler registered under `handle`; v / hyper / stats must be that
    sampler's state tensors (they are what the launch mutates; its other buffers are workspace)"""
    s = _SAMPLERS.get(handle)
    if s is None:
        raise RuntimeError('irsgmcmc::sgld_step: unknown sampler handle (torch_ops.register_sampler)')
    if v.data_ptr() != s.v.data_ptr() or hyper.data_ptr() != s.hyper.data_ptr() or stats.data_ptr() != s.stats.data_ptr():
        raise RuntimeError('irsgmcmc::sgld_step: v / hyper / stats are not the state tensors of that sampler')
    s.step(n, use_graph=False)


@sgld_step.register_fake
def _(v, hyper, stats, handle, n):
    return None


OPS = ('warp3d', 'warp3d_bwd_grid', 'warp3d_nearest', 'svf_exp', 'svf_exp_bwd', 'sobolev_smooth', 'lcc_normalise',
       'lcc_normalise_bwd', 'reg_energy', 'reg_energy_grad', 'ffd', 'ffd_adjoint', 'langevin_proposal', 'gmm_log_pdf',
       'gmm_log_pdf_param_grads', 'vd_factor', 'welford_update', 'welford_std', 'split_rhat', 'log_det_jacobian', 'dice_counts', 'average_surface_distance',
       'label_counts_update', 'label_posterior', 'sgld_step')
