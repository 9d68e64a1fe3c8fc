"""
fp64 references of the warp, the warp adjoint epilogue, dL/dz, the regulariser energy and scalars and the regulariser
gradient + SGD update of the SGLD transition, with per-voxel rounding bounds.

Like tests/helpers/transition_ref.py, each function takes the fp32 inputs the kernel itself read for that stage and
returns (ref, bound) in fp64, so stages are checked one at a time and errors never compound.  Given fp64 inputs the
functions compute the exact operations (test_step_stage_ref.py checks them against the oracle).

Decisions.  The warp takes decisions on rounded values (floor, the border clamp, the inside test).  As in svf_step_ref,
they are taken here in the input's precision, exactly as csrc/irs_warp.cu position_from_u and csrc/irs_common.cuh take
them: p = fl(fl(x + u) + t), t = alpha - 2 alpha r, then inside = 0 < p < n - 1 on the unclamped p, clamp to [0, n - 1],
floor.  t is exact when alpha is a power of two (2 alpha r has the 24 bits of r), so a contraction of the jitter into
an FMA cannot change p; positions() asserts it.  Everything after the decisions is evaluated in fp64.  The mixture's
choice of the maximum m is also a decision, but one that does not change the mathematical result.

The library is compiled without --use_fast_math: 1.0f / x and sqrtf are correctly rounded, expf has at most 2 ulp and
logf at most 1 ulp of error (CUDA C Programming Guide, mathematical functions; host libm is within the same bounds).  A
product followed by a sum may be contracted into an FMA; the bounds hold either way (an FMA only removes a rounding).

Rounding bounds (u = 2^-24, first order; SO = 1 + 2^-10 covers the second-order terms)
--------------------------------------------------------------------------------------------------------------------
Warp value and gradient (irs_interp_grad), M = max |corner| of the cell.  A lerp a + f (b - a) of values bounded by M
rounds by 5uM (difference 2uM, product 2uM, sum uM) and passes on its inputs' errors as a convex combination:
  * value: three lerp levels, 15uM;
  * the differences d00..d11 (|d| <= 2M) round by 2uM; a00..a11 are one lerp level (5uM); e = a01 - a00 carries
    10uM + 2uM; the second level b0, b1 carries 10uM; gz = b1 - b0 carries 20uM + 2uM; gy = e0 + fz (e1 - e0) and
    gx = dx0 + fz (dx1 - dx0) are lerps on values <= 2M (10uM each level) of inputs with 12uM:   22uM for each component.
    The gradient is multiplied by inside (0 or 1, exact), so it is exactly 0 on and outside the border.
Adjoint epilogue field_a = g_I grad:  |g_I| b_grad + b_g |grad| + u |g_I grad|  (one rounding for the product).
dL/dz = alpha z sum_k rho_k prec_k (irs_gmm_eval_t), e_k = lw_k - z^2 prec_k / 2:
  * e_k is off by de_k = u (2 |z^2 prec_k / 2| + |e_k|) ABSOLUTELY (the terms cancel, so no relative bound exists);
    e_k - m adds the error of m (<= max_j de_j) and one rounding; expf adds 2 ulp <= 4u relative:
        eps_k = de_k + max_j de_j + u |e_k - m| + 4u            (relative error of exp(e_k - m))
  * S = sum_k exp(..) (positive terms): eps_S = sum_k rho_k eps_k + (K - 1) u; 1 / S and rho_k = e_k / S add 2u;
    wprec = sum rho_k prec_k (positive): eps_w = sum_k rho_k prec_k (eps_k + eps_S + 3u) / wprec + (K - 1) u;
    the two products alpha z wprec add 2u.  An exp that underflows (e_k - m < -87) has an absolute error below 2^-126
    (S >= 1), covered by an absolute K max(prec) 2^-120 on wprec.
  * the logged data term alpha sum(-log p): log p = m + logf(S) - log sqrt(2 pi) is off by
        b_lp = max_j de_j + eps_S + 3u |log S| + u |m + log S| + u |log p| + u 0.92   (logf 1 ulp; the fp32 constant)
    and gmm_grad_kernel sums -log p in one fp32 register per thread (at most L = 4 ceil(V / (4 G 256)) updates with G
    blocks, the vector sweep's worst case) and then over the warp in fp32 (5 levels), above in fp64:
        |DATA - ref| <= alpha ( sum b_lp + (L + 5) u sum |log p| ) + 1e-13 |ref|
Energy sum |D css|^2 with the doubled last difference (irs_diff_energy): a term (w d) d is off by 3u relative; every
term is positive, so a sum whose longest fp32 addition chain is L is off by (L + 3) u relative, plus the fp64 levels
(1e-13 relative).  L is taken from the code that runs (energy_chain()).
Regulariser gradient irs_diff_energy_grad along one axis, 2 (w1 (vj - vm) - w2 (vp - vj)): the two differences and the
subtraction round, 4u A with A = w1 |d1| + w2 |d2| (|axis gradient| <= 2A); adding the three axes rounds twice,
4u sum A.  With Ge = 2 sum_axes A the energy gradient is off by 4u Ge.  The interior fast path (energy_grad4's g1) is
the same expression with weights one.  grad_v = sigma^2 (g_css + k ge), k = (float) REG_COEF:
        sigma^2 ( |k| 4u Ge + u |k ge| + u |g_css + k ge| + b_gcss ) + 2u |grad_v|
SGD update v - tau grad_v from the kernel's own grad_v: u (|tau grad_v| + |v_new|), the two roundings themselves, so
margins close to 1 are expected there.
"""
import math

import numpy as np
import torch

from tests.helpers.transition_ref import worst  # noqa: F401  (re-exported for the tests)

U24 = 2.0 ** -24
SO = 1.0 + 2.0 ** -10
LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
MAX_K = 8


# ---- warp ------------------------------------------------------------------------------------------------------------
def positions(u, r=None, alpha=0.0):
    """the kernel's sampling positions [px, py, pz] (each (C, D, H, W), u's precision) for displacement u (C, 3, D, H, W)
    and jitter r (C, 3, D, H, W) in [0, 1) or None"""
    C, _, D, H, W = u.shape
    z, y, x = torch.meshgrid(torch.arange(D), torch.arange(H), torch.arange(W), indexing='ij')
    p = [xyz.to(u.dtype) + u[:, a] for a, xyz in enumerate((x, y, z))]
    if r is not None:
        alpha = float(np.float32(alpha)) if u.dtype == torch.float32 else float(alpha)
        for a in range(3):
            t = alpha - (2.0 * alpha) * r[:, a].to(u.dtype)
            if u.dtype == torch.float32:
                assert torch.equal(t.double(), alpha - 2.0 * alpha * r[:, a].double()), 'jitter not exact: alpha not dyadic'
            p[a] = p[a] + t
    return p


def warp(img, p):
    """((value, bound), (grad (C, 3, D, H, W), bound), inside (C, 3, D, H, W)) of the trilinear sample of img (D, H, W) at
    the unclamped positions p, with the kernel's decisions taken in p's precision"""
    D, H, W = img.shape
    dims, strides = (W, H, D), (1, W, W * H)
    flat = img.double().reshape(-1)
    inside, i0, i1, f = [], [], [], []
    for a in range(3):
        n = dims[a]
        inside.append(((p[a] > 0) & (p[a] < n - 1)).double())
        pc = p[a].clamp(0, n - 1)
        fl = torch.floor(pc)
        f.append((pc - fl).double())                 # exact
        i0.append(fl.long())
        i1.append((fl.long() + 1).clamp(max=n - 1))  # far border: stride 0
    v = {}
    for b in range(8):
        bx, by, bz = b & 1, (b >> 1) & 1, b >> 2
        idx = (i1[0] if bx else i0[0]) + (i1[1] if by else i0[1]) * strides[1] + (i1[2] if bz else i0[2]) * strides[2]
        v[bz, by, bx] = flat[idx]
    M = torch.stack(list(v.values())).abs().amax(0)
    fx, fy, fz = f
    a = {(bz, by): v[bz, by, 0] + fx * (v[bz, by, 1] - v[bz, by, 0]) for bz in (0, 1) for by in (0, 1)}
    b0, b1 = a[0, 0] + fy * (a[0, 1] - a[0, 0]), a[1, 0] + fy * (a[1, 1] - a[1, 0])
    value = b0 + fz * (b1 - b0)
    d = {(bz, by): v[bz, by, 1] - v[bz, by, 0] for bz in (0, 1) for by in (0, 1)}
    dx0, dx1 = d[0, 0] + fy * (d[0, 1] - d[0, 0]), d[1, 0] + fy * (d[1, 1] - d[1, 0])
    e0, e1 = a[0, 1] - a[0, 0], a[1, 1] - a[1, 0]
    grad = torch.stack([dx0 + fz * (dx1 - dx0), e0 + fz * (e1 - e0), b1 - b0], 1)
    ins = torch.stack(inside, 1)
    grad = grad * ins
    b_val = U24 * SO * 15.0 * M
    b_grad = U24 * SO * 22.0 * M.unsqueeze(1) * ins
    return (value.unsqueeze(1), b_val.unsqueeze(1)), (grad, b_grad), ins


def warp_adjoint(g_img, b_gimg, grad, b_grad):
    """(field_a, bound): g_I (C, 1, ...) times the warp gradient (C, 3, ...), each with its bound"""
    g = g_img.double()
    ref = g * grad
    bound = g.abs() * b_grad + b_gimg * grad.abs() + U24 * SO * ref.abs()
    return ref, bound


# ---- dL/dz and the logged data term ----------------------------------------------------------------------------------
def gmm_grad(z, mask, table, K, alpha):
    """((dL/dz, bound), (data term, bound)) for one chain: z (V,), mask (V,) bool, table (16,) = lw[8], prec[8] as the
    kernel reads it, alpha the fp32 VD factor"""
    z = z.double().reshape(-1)
    m_on = mask.reshape(-1).bool()
    lw, prec = table[:K].double(), table[MAX_K:MAX_K + K].double()
    hz2p = 0.5 * (z * z).unsqueeze(1) * prec           # (V, K)
    e = lw - hz2p
    m = e.amax(1, keepdim=True)
    ex = torch.exp(e - m)
    S = ex.sum(1, keepdim=True)
    rho = ex / S
    wprec = (rho * prec).sum(1)
    g = alpha * z * wprec
    de = U24 * (2.0 * hz2p.abs() + e.abs())
    de_max = de.amax(1, keepdim=True)
    eps_k = de + de_max + U24 * (e - m).abs() + 4.0 * U24
    eps_S = (rho * eps_k).sum(1, keepdim=True) + (K - 1) * U24
    eps_w = (rho * prec * (eps_k + eps_S + 3.0 * U24)).sum(1) / wprec + (K - 1) * U24
    tiny = K * float(prec.max()) * 2.0 ** -120
    b_g = SO * ((g.abs() * (eps_w + 2.0 * U24)) + abs(alpha) * z.abs() * tiny)
    g, b_g = torch.where(m_on, g, 0.0), torch.where(m_on, b_g, 0.0)

    logS = torch.log(S.squeeze(1))
    lp = m.squeeze(1) + logS - LOG_SQRT_2PI
    b_lp = (de_max + eps_S).squeeze(1) + U24 * (3.0 * logS.abs() + (m.squeeze(1) + logS).abs() + lp.abs() + 0.92)
    return (g, b_g), (lp, b_lp)


def data_blocks(V):
    """irs_data_blocks: the grid of gmm_grad_kernel"""
    limit = 296 if V <= 128 ** 3 else 592
    return min((V + 255) // 256, limit)


def data_term(lp, b_lp, mask, alpha):
    """(alpha sum_mask -log p, bound) with the accumulation of gmm_grad_kernel"""
    on = mask.reshape(-1).bool()
    V = on.numel()
    L = 4 * -(-V // (4 * data_blocks(V) * 256))
    ref = alpha * float((-lp[on]).sum())
    bound = abs(alpha) * SO * (float(b_lp[on].sum()) + (L + 5) * U24 * float(lp[on].abs().sum())) + 1e-13 * abs(ref)
    return ref, bound


# ---- regulariser energy, scalars, gradient and the SGD update --------------------------------------------------------
def _axis_diffs(x, axis):
    """forward differences d_j (j = 0 .. n-2) and their weights w_j (2 for the doubled last one) along `axis`"""
    n = x.shape[axis]
    d = x.narrow(axis, 1, n - 1) - x.narrow(axis, 0, n - 1)
    w = torch.ones(n - 1, dtype=x.dtype)
    w[-1] = 2.0
    shape = [1] * x.dim()
    shape[axis] = n - 1
    return d, w.view(shape)


def energy(css):
    """(C,) fp64: sum over components and axes of w d^2"""
    x = css.double()
    out = torch.zeros(x.shape[0], dtype=torch.float64)
    for axis in (2, 3, 4):
        d, w = _axis_diffs(x, axis)
        out += (w * d * d).sum(dim=(1, 2, 3, 4))
    return out


def energy_chain(dims, ffd):
    """the longest fp32 addition chain of the energy reduction over the paths that can run for a state grid `dims`
    (D, H, W): the first squaring step's epilogue (W % 4 == 0, no FFD: a thread adds (x + y) + z per plane and channel
    over at most D planes), the stand-alone vector kernel (W % 4 == 0: ((t + t) + t) + t, nine per iteration) or the
    scalar one ((x + y) + z, three per iteration); 592-block grid-stride loops; then 5 fp32 warp-shuffle levels"""
    D, H, W = dims
    V = D * H * W
    G = min((V + 255) // 256, 592)
    L = 2 + 3 * -(-V // (G * 256))
    if W % 4 == 0:
        L = max(L, 3 + 9 * -(-V // (4 * G * 256)))
        if not ffd:
            L = max(L, 2 + 3 * D)
    return L + 5


def energy_bound(E, chain):
    return (chain + 3) * U24 * SO * E.abs() + 1e-13 * E.abs()


def energy_grad(css):
    """(dE/dcss, Ge) fp64, Ge = the sum over axes of 2 (w_{j-1} |d_{j-1}| + w_j |d_j|), the magnitude the bound uses"""
    x = css.double()
    g, Ge = torch.zeros_like(x), torch.zeros_like(x)
    for axis in (2, 3, 4):
        n = x.shape[axis]
        d, w = _axis_diffs(x, axis)
        wd = w * d
        # voxel j gets + 2 w_{j-1} d_{j-1} (j >= 1) and - 2 w_j d_j (j <= n - 2)
        g.narrow(axis, 1, n - 1).add_(2.0 * wd)
        g.narrow(axis, 0, n - 1).sub_(2.0 * wd)
        Ge.narrow(axis, 1, n - 1).add_(2.0 * wd.abs())
        Ge.narrow(axis, 0, n - 1).add_(2.0 * wd.abs())
    return g, Ge


def sgd_grad(css, sigma, g_css, k, b_gcss=None):
    """(grad_v, bound): sigma^2 (g_css + k dE/dcss); sigma None = 1 or broadcast over chains; k the fp32 coefficient
    per chain (C,) as the kernel holds it; b_gcss a bound on g_css's own error"""
    ge, Ge = energy_grad(css)
    kk = torch.as_tensor(k, dtype=torch.float64).view(-1, 1, 1, 1, 1)
    sg2 = torch.ones(1, dtype=torch.float64) if sigma is None else sigma.double() ** 2
    gc = g_css.double()
    inner = gc + kk * ge
    ref = sg2 * inner
    b = 0.0 if b_gcss is None else b_gcss
    bound = SO * (sg2 * (kk.abs() * 4.0 * U24 * Ge + U24 * (kk * ge).abs() + U24 * inner.abs() + b) + 2.0 * U24 * ref.abs())
    return ref, bound


def sgd_step(v, grad_v, tau):
    """(v_new, bound) from the kernel's own grad_v; tau as the kernel holds it (fp32)"""
    tau = float(np.float32(tau))
    step = tau * grad_v.double()
    ref = v.double() - step
    return ref, U24 * SO * (step.abs() + ref.abs())


def reg_lognormal(y, loc, log_scale, dof, w_reg, learnable):
    """(REG, REG_COEF, g0, g1) of one chain, fp64 throughout (irs_reg_chain_terms, LogNormal)"""
    s2 = math.exp(log_scale) ** 2
    ly = math.log(y)
    r = ly - loc
    reg = ly + log_scale + 0.5 * r * r / s2 + (0.5 * dof - 1.0) * ly
    coef = 0.5 * w_reg + r / (s2 * y) if learnable else (r / s2 + 0.5 * dof) / y
    return reg, coef, -r / s2, 1.0 - r * r / s2


def reg_l2(y, log_w, dof):
    w = math.exp(log_w)
    return 0.5 * w * y - 0.5 * dof * log_w, 0.5 * w, 0.5 * w * y - 0.5 * dof, 0.0


def adam_bias(step, beta_pow, b1, b2):
    """the running powers of beta after this step and the bias corrections"""
    p1, p2 = (1.0, 1.0) if step == 0 else beta_pow
    p1, p2 = p1 * b1, p2 * b2
    return (p1, p2), 1.0 - p1, 1.0 - p2


def adam64(p, m, v, g, lr, decay, bc1, bc2, b1, b2, eps):
    m = b1 * m + (1.0 - b1) * g
    v = b2 * v + (1.0 - b2) * g * g
    return p - (lr / decay) / bc1 * (m / (math.sqrt(v) / math.sqrt(bc2) + eps)), m, v


def reg_config(cc):
    """the fields of a C-ABI sampler config (irsgmcmc_b200._lib.SgldConfig) that the regulariser step reads"""
    from irsgmcmc_b200 import _lib
    return dict(lognormal=cc.reg_type == _lib.REG_LOGNORMAL, learnable=bool(cc.reg_learnable), w_reg=cc.w_reg,
                dof=cc.dof, lr0=cc.lr_reg0, lr1=cc.lr_reg1, lr_decay=cc.lr_decay, beta1=cc.beta1, beta2=cc.beta2,
                eps=cc.adam_eps, prior_loc=cc.reg_scale_prior_loc, prior_scale=cc.reg_scale_prior_scale,
                shape=cc.w_reg_prior_shape, rate=cc.w_reg_prior_rate)


def reg_hyper(energy, hyper, c):
    """reference of the regulariser step of reg_hyper_kernel with one shared parameter block (hyper mode 'reference'):
    the chains' energies y_c (the kernel's own), the parameter block before the step and reg_config(...) ->
    ([(REG_c, REG_COEF_c)], {hyper slot: (value after the step, bound)}).  The LogNormal path is fp64 throughout, held
    to 1e-12 relative; the L2 path's parameter goes through adam32."""
    from irsgmcmc_b200 import _lib
    h = [float(x) for x in hyper]
    P, M, V = _lib.HYPER_REG_P, _lib.HYPER_REG_M, _lib.HYPER_REG_V
    S, BP = _lib.HYPER_REG_STEP, _lib.HYPER_REG_BETA_POW
    rel = lambda x: 1e-12 * abs(x)
    scalars, g0, g1 = [], 0.0, 0.0
    for y in energy:
        if c['lognormal']:
            reg, coef, a, b = reg_lognormal(float(y), h[P], h[P + 1], c['dof'], c['w_reg'], c['learnable'])
        else:
            reg, coef, a, b = reg_l2(float(y), h[P], c['dof'])
        scalars.append((reg, coef))
        g0, g1 = g0 + a, g1 + b
    out = {k: (h[k], 0.0) for k in (P, P + 1, M, M + 1, V, V + 1, S)}
    if not c['learnable']:
        return scalars, out
    step0 = h[S]
    (p1, p2), bc1, bc2 = adam_bias(step0, (h[BP], h[BP + 1]), c['beta1'], c['beta2'])
    decay = 1.0 + step0 * c['lr_decay']
    args = (decay, bc1, bc2, c['beta1'], c['beta2'], c['eps'])
    if c['lognormal']:
        g1 += (h[P + 1] - c['prior_loc']) / (c['prior_scale'] * c['prior_scale'])
        for j, g, lr in ((0, g0, c['lr0']), (1, g1, c['lr1'])):
            p, m, v = adam64(h[P + j], h[M + j], h[V + j], g, lr, *args)
            out.update({P + j: (p, rel(p)), M + j: (m, rel(m)), V + j: (v, rel(v))})
    else:
        g0 += -(c['shape'] - c['rate'] * math.exp(h[P]))
        p, m, v, b = adam32(h[P], h[M], h[V], g0, c['lr0'], *args)
        out.update({P: (p, b), M: (m, 8.0 * U24 * abs(m)), V: (v, 8.0 * U24 * abs(v))})
    out.update({S: (step0 + 1.0, 0.0), BP: (p1, rel(p1)), BP + 1: (p2, rel(p2))})
    return scalars, out


def adam32(p, m, v, g, lr, decay, bc1, bc2, b1, b2, eps):
    """(p, m, v, bound on p): the fp32 Adam of irs_adam_update, each operation rounded to fp32 and not contracted.  A
    contraction removes roundings; the bound covers any choice: m and v are off by a few u relative, the step
    lr / decay / bc1 * m / denom by at most 12u of itself, and p rounds once more"""
    f = np.float32
    gf = f(g)
    mf = f(f(b1) * f(m)) + f(f(1.0 - b1) * gf)
    vf = f(f(b2) * f(v)) + f(f(f(1.0 - b2) * gf) * gf)
    denom = f(f(np.sqrt(vf)) / f(math.sqrt(bc2))) + f(eps)
    step = f((lr / decay) / bc1)
    q = f(step * f(mf / denom))
    pn = f(f(p) - q)
    return float(pn), float(mf), float(vf), 12.0 * U24 * abs(float(q)) + 2.0 * U24 * abs(float(pn))
