"""
CPU checks of tests/helpers/step_stage_ref.py, the per-voxel references of the warp, dL/dz, the regulariser energy and
the regulariser gradient + SGD update: with fp64 inputs they equal the oracle (oracle/sgld_oracle.py) and autograd;
with fp32 inputs the kernels' own __host__ __device__ bodies, run through the host emulation (tests/host_emul), lie
inside the bounds on every voxel, faces, edges and corners included; and the comparison rejects the errors these
stages could plausibly make (a 4-component sweep for a 5-component mixture, a single weight on a doubled last difference,
a gradient let through on the border).
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sgld_oracle as O
from tests.helpers import step_stage_ref as R
from tests.util import smooth_field


@pytest.fixture(scope='module')
def emul(built):
    return ctypes.CDLL(built['emul'])


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def np32(t):
    return np.ascontiguousarray(t.float().numpy())


def expect_within(out, ref, bound, what):
    nbad, at, r, med = R.worst(out, ref, bound)
    print(f'{what}: max |err| / bound = {r:.3g}, median {med:.3g}')
    assert nbad == 0, f'{what}: {nbad} voxels outside the bound; worst {at} at {r:.3g} x bound'
    return r


def border_displacements(n, C, seed):
    """smooth |u| < 2.5 plus integer and half-integer displacements that put samples exactly on nodes, on the border
    p = 0 / p = n - 1, and outside the volume, along every axis"""
    u = smooth_field((C, 3, n, n, n), 2.5, seed)
    for c in range(C):
        for a in range(3):
            u[c, a, :, 1] = -1.0 - c                          # whole planes shifted by integers: nodes, p = 0, outside
            u[c, a, :, :, 2] = 0.5                            # half a voxel: mid-cell, the far face p = n - 1/2
            u[c, a, 3] = float(n - 1) - torch.arange(n).float().view(1, n) if a == 0 else u[c, a, 3]
        x = torch.arange(n).float()
        u[c, 0, 4, 4] = -x                                     # p_x = 0 exactly
        u[c, 1, 5, :, 3] = float(n - 1) - x                    # p_y = n - 1 exactly
        u[c, 2, :, 6, 7] = float(n + 2) - x                    # p_z beyond n - 1: clamped
    return u.contiguous()


# ---- fp64: the references are the exact operations ------------------------------------------------------------------
def test_warp_reference_matches_oracle_fp64():
    n, C = 9, 2
    img = smooth_field((1, 1, n, n, n), 1.0, 1).double()[0, 0]
    u = smooth_field((C, 3, n, n, n), 3.0, 2).double()
    r = torch.rand(C, 3, n, n, n, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    p = R.positions(u, r, 0.1)
    (val, _), (grad, _), ins = R.warp(img, p)
    pc = [p[a].clamp(0, n - 1).requires_grad_(True) for a in range(3)]
    out = O.trilinear_sample_voxel(img.view(1, 1, n, n, n).expand(C, 1, n, n, n), *pc)
    assert float((out.detach() - val).abs().max()) <= 1e-13
    g = torch.autograd.grad(out.sum(), pc)
    g = torch.stack(g, 1) * ins
    assert float((g - grad).abs().max()) <= 1e-12
    assert 0 < float(ins.mean()) < 1


def test_gmm_reference_matches_oracle_fp64():
    gen = torch.Generator().manual_seed(5)
    for K in (1, 3, 8):
        log_std = torch.linspace(-3.0, 1.0, K, dtype=torch.float64)
        logits = torch.randn(K, generator=gen, dtype=torch.float64)
        table = torch.zeros(16, dtype=torch.float64)
        table[:K] = O.gmm_log_proportions(logits) - log_std
        table[8:8 + K] = torch.exp(-2.0 * log_std)
        z = 3.0 * torch.randn(500, generator=gen, dtype=torch.float64)
        mask = torch.rand(500, generator=gen) > 0.3
        alpha = 0.37
        (g, _), (lp, _) = R.gmm_grad(z, mask, table, K, alpha)
        rho = O.gmm_responsibilities(z, log_std, logits)
        g_or = alpha * z * (rho * torch.exp(-2.0 * log_std)).sum(-1) * mask
        assert float((g - g_or).abs().max()) <= 1e-12 * float(g_or.abs().max())
        lp_or = O.gmm_log_pdf(z, log_std, logits).reshape(-1)
        assert float(((lp - lp_or).abs() / lp_or.abs().clamp_min(1.0)).max()) <= 1e-13
        d, _ = R.data_term(lp, torch.zeros_like(lp), mask, alpha)
        assert abs(d - alpha * float(O.gmm_nll(z[mask], log_std, logits))) <= 1e-10 * abs(d)


def test_energy_and_gradient_match_oracle_fp64():
    for shape in ((2, 3, 6, 7, 5), (1, 3, 2, 3, 4)):
        v = torch.randn(*shape, generator=torch.Generator().manual_seed(6), dtype=torch.float64).requires_grad_(True)
        E_or = O.reg_energy(v)
        assert torch.allclose(R.energy(v.detach()), E_or.detach(), rtol=1e-13, atol=0)
        g_or, = torch.autograd.grad(E_or.sum(), v)
        g, _ = R.energy_grad(v.detach())
        assert float((g - g_or).abs().max()) <= 1e-12


# ---- fp32: the kernels' per-voxel bodies lie inside the bounds ----------------------------------------------------------
@pytest.mark.parametrize('n,jitter', [(8, None), (9, 'dyadic'), (13, 'dyadic')])
def test_warp_bodies_within_bounds(emul, n, jitter):
    C = 2
    img = (0.5 + smooth_field((1, 1, n, n, n), 1.0, n)).float()[0, 0].contiguous()
    u = border_displacements(n, C, n + 1)
    r = None if jitter is None else torch.rand(C, 3, n, n, n, generator=torch.Generator().manual_seed(n))
    alpha = 0.125
    out, grad = np.zeros((C, 1, n, n, n), np.float32), np.zeros((C, 3, n, n, n), np.float32)
    rn = None if r is None else np32(r)
    emul.emul_warp_vox(P(np32(img)), P(np32(u)), None if rn is None else P(rn), ctypes.c_float(alpha), P(out), P(grad),
                       C, n, n, n)
    (val, b_val), (g, b_g), ins = R.warp(img, R.positions(u, r, alpha))
    expect_within(torch.from_numpy(out), val, b_val, f'warp value n={n} jitter={jitter}')
    expect_within(torch.from_numpy(grad), g, b_g, f'warp gradient n={n} jitter={jitter}')
    assert float(ins.min()) == 0.0 and bool((torch.from_numpy(grad)[ins == 0] == 0).all())


def gmm_case(K, seed):
    gen = torch.Generator().manual_seed(seed)
    log_std = torch.linspace(-4.0, 0.5, K)
    logits = 0.5 * torch.randn(K, generator=gen)
    table = torch.zeros(16)
    table[:K] = (O.gmm_log_proportions(logits.double()) - log_std.double()).float()
    table[8:8 + K] = torch.exp(-2.0 * log_std.double()).float()
    z = torch.cat([0.02 * torch.randn(2000, generator=gen), torch.randn(2000, generator=gen),
                   40.0 * torch.randn(2000, generator=gen), torch.tensor([0.0, -0.0, 1e-20, 200.0])])
    mask = (torch.rand(z.numel(), generator=gen) > 0.2).to(torch.uint8)
    return z, mask, table


def _emul_gmm(emul, z, mask, table, K, kk, alpha):
    g, lp = np.zeros(z.numel(), np.float32), np.zeros(z.numel(), np.float32)
    emul.emul_gmm_grad(P(np32(z)), P(np.ascontiguousarray(mask.numpy())), P(np32(table)), K, kk, ctypes.c_float(alpha),
                       P(g), P(lp), ctypes.c_longlong(z.numel()))
    return torch.from_numpy(g), torch.from_numpy(lp)


@pytest.mark.parametrize('K', [1, 2, 4, 5, 8])
def test_gmm_bodies_within_bounds(emul, K):
    z, mask, table = gmm_case(K, K)
    alpha = float(np.float32(0.8125))
    (g_ref, b_g), (lp_ref, b_lp) = R.gmm_grad(z, mask, table, K, alpha)
    for kk in ((4, 8) if K <= 4 else (8,)):
        g, lp = _emul_gmm(emul, z, mask, table, K, kk, alpha)
        expect_within(g, g_ref, b_g, f'dL/dz K={K} KK={kk}')
        on = mask.bool()
        expect_within(lp[on], lp_ref[on], b_lp[on], f'log p K={K} KK={kk}')


def test_gmm_four_component_sweep_fails_for_five(emul):
    """the mutant that picks the KK = 4 sweep for K = 5 drops a component: far outside the bound"""
    K = 5
    z, mask, table = gmm_case(K, 11)
    (g_ref, b_g), _ = R.gmm_grad(z, mask, table, K, 1.0)
    g, _ = _emul_gmm(emul, z, mask, table, K, 4, 1.0)
    assert R.worst(g, g_ref, b_g)[0] > 100


def _emul_sgd(emul, v, sigma, css, gc, k, tau):
    D, H, W = v.shape[-3:]
    vn, gv = np32(v[0]).copy(), np.zeros((3, D, H, W), np.float32)   # updated in place
    emul.emul_sgd_update(P(vn), None if sigma is None else P(np32(sigma[0])), P(np32(css[0])), P(np32(gc[0])),
                         ctypes.c_float(k), ctypes.c_float(tau), P(gv), D, H, W)
    return torch.from_numpy(vn)[None], torch.from_numpy(gv)[None]


@pytest.mark.parametrize('shape', [(2, 2, 2), (5, 3, 8), (9, 12, 7)])
def test_sgd_update_body_within_bounds(emul, shape):
    gen = torch.Generator().manual_seed(sum(shape))
    css = 3.0 * torch.randn(1, 3, *shape, generator=gen)
    v = torch.randn(1, 3, *shape, generator=gen)
    sigma = torch.rand(1, 3, *shape, generator=gen) + 0.5
    gc = torch.randn(1, 3, *shape, generator=gen)
    k, tau = float(np.float32(0.73)), float(np.float32(0.4))
    for sg, g_css in ((None, torch.zeros_like(gc)), (sigma, gc)):
        v_new, gv = _emul_sgd(emul, v, sg, css, g_css, k, tau)
        ref, bound = R.sgd_grad(css, sg, g_css, [k])
        expect_within(gv, ref, bound, f'grad_v {shape} sigma={sg is not None}')
        expect_within(v_new, *R.sgd_step(v, gv, tau), f'v {shape} sigma={sg is not None}')


def test_comparator_rejects_single_weight_on_last_difference(emul):
    """a field that differs only in the last x difference: dropping the factor 2 there moves grad_v at x = W - 2, W - 1
    far outside the bound"""
    D, H, W = 6, 5, 12
    css = torch.zeros(1, 3, D, H, W)
    css[..., -1] = 1.0
    v, gc = torch.zeros_like(css), torch.zeros_like(css)
    _, gv = _emul_sgd(emul, v, None, css, gc, 1.0, 0.4)
    ref, bound = R.sgd_grad(css, None, gc, [1.0])
    assert R.worst(gv, ref, bound)[0] == 0
    bad = gv.clone()
    bad[..., -2:] /= 2.0     # what irs_diff_energy_grad gives with weight 1 on d_{n-2}
    assert R.worst(bad, ref, bound)[0] == 2 * 3 * D * H


def test_energy_chain_lengths():
    """the addition chain follows the path: epilogue (D planes), vector and scalar stand-alone kernels"""
    assert R.energy_chain((64, 64, 64), False) == 2 + 3 * 64 + 5
    assert R.energy_chain((7, 8, 11), True) == 2 + 3 + 5
    assert R.energy_chain((11, 7, 8), True) == 3 + 9 + 5
    E = torch.tensor([2.0])
    assert float(R.energy_bound(E, 10)[0]) == pytest.approx(2.0 * 13 * R.U24 * R.SO + 2e-13)


@pytest.mark.parametrize('lognormal,learnable', [(True, True), (True, False), (False, True), (False, False)])
def test_reg_hyper_reference_matches_host_body(emul, lognormal, learnable):
    """reg_hyper() against irs_reg_hyper_step (the kernel's own body, serial over the chains) for three chains and two
    consecutive steps (the second with non-zero Adam moments and running powers of beta), on the LogNormal and L2
    paths: REG and REG_COEF of every chain and every slot of the parameter block the step writes"""
    from irsgmcmc_b200 import _lib
    from irsgmcmc_b200.sampler import lognormal_init
    C, V = 3, 20 ** 3
    dof = 3.0 * V
    c = dict(lognormal=lognormal, learnable=learnable, w_reg=1.6 if lognormal else 1.4, dof=dof, lr0=0.01, lr1=0.02,
             lr_decay=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, prior_loc=2.8, prior_scale=5.0, shape=0.5 * dof,
             rate=1.0 / (0.5 * dof))
    cfg_d = np.array([_lib.REG_LOGNORMAL if lognormal else _lib.REG_L2, learnable, c['lr0'], c['lr1'], c['lr_decay'],
                      c['beta1'], c['beta2'], c['eps'], c['prior_loc'], c['prior_scale'], c['w_reg'], dof, c['shape'],
                      c['rate']], np.float64)
    hyper = np.zeros(_lib.HYPER_SIZE, np.float64)
    if lognormal:
        hyper[_lib.HYPER_REG_P:_lib.HYPER_REG_P + 2] = lognormal_init(c['w_reg'], dof)
    else:
        hyper[_lib.HYPER_REG_P] = float(np.float32(np.log(c['w_reg'])))
    for step, energy in enumerate(([5.1e3, 7.3e3, 6.2e3], [4.4e3, 9.0e3, 1.2e3])):
        before = hyper.copy()
        stats = np.zeros((C, _lib.STAT_SIZE), np.float64)
        stats[:, _lib.STAT_ENERGY] = energy
        emul.emul_reg_hyper_step(P(hyper), P(cfg_d), C, P(stats))
        scalars, slots = R.reg_hyper(energy, before, c)
        for ch, (reg, coef) in enumerate(scalars):
            assert abs(stats[ch, _lib.STAT_REG] - reg) <= 1e-12 * abs(reg), (step, ch)
            assert abs(stats[ch, _lib.STAT_REG_COEF] - coef) <= 1e-12 * abs(coef), (step, ch)
        for k, (ref, bound) in slots.items():
            assert abs(hyper[k] - ref) <= bound, (step, k, hyper[k], ref, bound)
        if learnable:
            assert hyper[_lib.HYPER_REG_STEP] == step + 1 and hyper[_lib.HYPER_REG_P] != before[_lib.HYPER_REG_P]
