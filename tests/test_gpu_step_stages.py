"""
The warp, the warp adjoint epilogue, dL/dz, the regulariser energy and scalars and the regulariser gradient + SGD update
of one eager SGLD transition (SGLDSampler.step(1, use_graph=False)), voxel by voxel against the fp64 references of
tests/helpers/step_stage_ref.py.  No voxel is exempt.  Every stage is fed the inputs the kernel itself read, taken from
the buffers that still hold them after the step, so errors never compound:

  stage                                   kernel input                         kernel output
  (4) warp + spatial gradient             hist[-1], jitter r                   im_warped (the gradient via field_a)
  (7) dL/dz, logged data term             z, mask, _gmm_table, stats[ALPHA]    _scratch1, stats[DATA]
  (8) residual adjoint x warp gradient    LCC: _scratch2 (ga); SSD: _scratch1  _field_a (survives with svf_steps <= 2)
  (2) energy                              css                                  stats[ENERGY]
  (9) regulariser scalars + Adam          stats[ENERGY], hyper before          stats[REG], stats[REG_COEF], hyper
  (11) energy gradient + SGD update       css, sigma, stats[REG_COEF], v       grad_v, v

Inputs make every fp32 decision exact and reach the edges:
  * Sobolev smoothing off and eps = 0 injected: css == v bit for bit (asserted).
  * Constant integer / half-integer velocities with svf_steps = 1 give exact displacements: samples on nodes, on the
    border p = 0 / p = n - 1 (gradient 0) and outside the volume (clamped).  Their energy is 0, so they run with the L2
    regulariser (the LogNormal one takes log y).  Smooth random velocities give the generic case.
  * Jitter with alpha = 0.125 (2 alpha r exact): injected U[0,1) numbers, or Philox numbers regenerated on the CPU
    (emul_uniform3) at the pre-step iteration counter and the global chain ids.
  * A constant moving image makes the warp gradient, field_a and the data gradient g_css exactly 0 (asserted where
    field_a survives), which holds the regulariser stencil alone: energy_grad4's interior and face paths (W % 4 == 0),
    the scalar kernel (odd W).  W = 8 has no 4-voxel group with x >= 4 && x + 8 <= W, W = 12 only the middle one.
  * One case per data term with a non-zero data gradient (svf_steps = 1, no FFD) takes g_css from svf_step_ref on the
    kernel's field_a with its composed bound.
  * SVFFD_3D with unequal control point spacings: a non-cubic state grid, with W % 4 == 0 and != 0.
"""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import step_stage_ref as R
from tests.helpers import svf_step_ref as SVF
from tests.helpers import transition_ref as TR
from tests.util import smooth_field

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ALPHA = 0.125


@pytest.fixture(scope='module')
def emul(built):
    return ctypes.CDLL(built['emul'])


def expect_within(out, ref, bound, what):
    nbad, at, r, med = R.worst(out.cpu(), ref.cpu(), bound.cpu())
    print(f'{what}: max |err| / bound = {r:.3g}, median {med:.3g}')
    assert nbad == 0, f'{what}: {nbad} voxels outside the bound; worst {at} at {r:.3g} x bound'


def expect_close(out, ref, bound, what):
    r = abs(out - ref) / bound if bound > 0 else (0.0 if out == ref else float('inf'))   # energy 0: exact
    print(f'{what}: |err| / bound = {r:.3g}')
    assert r <= 1.0, f'{what}: {out!r} vs {ref!r}, {r:.3g} x bound'


def mask_with_holes(n, seed):
    """random holes, half of the z = 0 and x = n - 1 faces, one whole aligned 4-voxel group and mixed groups"""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(n, n, n, generator=g) > 0.25
    m[0, :, : n // 2] = False
    m[:, : n // 2, n - 1] = False
    m[n // 2, 1, 4:8] = False
    m[n // 2, 2, 0:4] = torch.tensor([True, False, True, False])
    return m


def constant_velocity(C, dims):
    """integer and half-integer displacements per chain and component (exact with svf_steps = 1)"""
    vals = [[1.0, -2.0, 0.5], [-0.5, 3.0, -1.0], [2.5, 0.0, -3.5]]
    v = torch.zeros(C, 3, *dims)
    for c in range(C):
        for a in range(3):
            v[c, a] = vals[c % 3][a]
    return v


def run_step(emul, n, C, data='lcc', s=2, K=4, reg='lognormal', learnable=True, svf_steps=1, sigma='none',
             jitter='inject', velocity='smooth', const_moving=False, cps=None, chain_offset=0, seed=0):
    from irsgmcmc_b200 import _lib
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    assert velocity != 'constant' or reg == 'l2', 'a constant velocity has energy 0: log y is -inf'
    fixed_im = 0.5 + 0.3 * smooth_field((1, 1, n, n, n), 1.0, seed + 1)
    moving_im = torch.full_like(fixed_im, 0.7) if const_moving else 0.5 + 0.3 * smooth_field((1, 1, n, n, n), 1.0, seed + 2)
    mask = mask_with_holes(n, seed + 3)
    cfg = SGLDConfig(data_loss=data, no_components=K, s=s, reg_loss='RegLoss_LogNormal' if reg == 'lognormal' else 'RegLoss_L2',
                     w_reg=1.6 if reg == 'lognormal' else 1.4, reg_learnable=learnable, sobolev_enabled=False,
                     svf_steps=svf_steps, uniform_noise=jitter != 'none', uniform_noise_magnitude=ALPHA,
                     transformation='SVFFD_3D' if cps else 'SVF_3D', cps=cps, seed=77 + seed)
    smp = SGLDSampler({'im': fixed_im, 'mask': mask.view(1, 1, n, n, n)}, {'im': moving_im}, C, cfg, device=DEV,
                      chain_offset=chain_offset)
    smp.init_gmm(sigma_hat=0.3)
    dims = smp.state_dims
    g = torch.Generator().manual_seed(seed + 4)
    v = constant_velocity(C, dims) if velocity == 'constant' else smooth_field((C, 3, *dims), 2.0, seed + 5)
    sg = {'none': None, 'shared': torch.rand(1, 3, *dims, generator=g) + 0.5,
          'per_chain': torch.rand(C, 3, *dims, generator=g) + 0.5}[sigma]
    smp.set_state(v, sg)
    ju = torch.rand(C, 3, n, n, n, generator=g) if jitter == 'inject' else None
    smp.set_noise(torch.zeros(C, 3, *dims), ju)
    hyper0 = smp.hyper.cpu().clone()
    iter0 = int(hyper0[..., _lib.HYPER_ITER].reshape(-1)[0])
    smp.step(1, use_graph=False)
    torch.cuda.synchronize()
    if jitter == 'philox':
        V = n ** 3
        ju = torch.zeros(C, 3, V)
        for c in range(C):
            r = np.zeros((V, 3), np.float32)
            emul.emul_uniform3(ctypes.c_ulonglong(cfg.seed), V, chain_offset + c, ctypes.c_ulonglong(iter0), r.ctypes.data_as(ctypes.c_void_p))
            ju[c] = torch.from_numpy(r).t()
        ju = ju.view(C, 3, n, n, n)
    out = {k: getattr(smp, k).cpu() for k in ('css', 'im_warped', 'z', 'stats', 'hyper', 'grad_v', 'v')}
    out.update(hist=smp.hist[-1].cpu(), s1=smp._scratch1.cpu(), s2=smp._scratch2.cpu(), field_a=smp._field_a.cpu(),
               table=smp._gmm_table.cpu(), v0=v, sigma=sg, r=ju, hyper0=hyper0, moving=moving_im[0, 0], mask=mask,
               cfg=cfg, smp=smp)
    return out


def check_stages(o, label, s=2):
    from irsgmcmc_b200 import _lib
    cfg, smp = o['cfg'], o['smp']
    C = smp.C
    ffd = smp.ffd
    assert torch.equal(o['css'], o['v0']), 'Sobolev off and eps = 0: css must equal v'

    # (4) warp value
    p = R.positions(o['hist'], o['r'] if cfg.uniform_noise else None, ALPHA)
    (val, b_val), (grad, b_grad), ins = R.warp(o['moving'], p)
    expect_within(o['im_warped'], val, b_val, f'{label} warp value')

    # (7) dL/dz and the data term, with each chain's table and fp32 VD factor
    for c in range(C):
        alpha = float(np.float32(o['stats'][c, _lib.STAT_ALPHA]))
        (g, b_g), (lp, b_lp) = R.gmm_grad(o['z'][c], o['mask'], o['table'][c], cfg.no_components, alpha)
        expect_within(o['s1'][c].reshape(-1), g, b_g, f'{label} dL/dz chain {c}')
        ref, bound = R.data_term(lp, b_lp, o['mask'], alpha)
        expect_close(float(o['stats'][c, _lib.STAT_DATA]), ref, bound, f'{label} data term chain {c}')

    # (8) adjoint epilogue: g_I times the warp gradient
    if cfg.svf_steps <= 2:
        if cfg.data_loss == 'lcc':
            g_img, b_img = TR.lcc_bwd_mean(o['s2'], s)
        else:
            g_img, b_img = -o['s1'].double(), torch.zeros(1, dtype=torch.float64)
        fa, b_fa = R.warp_adjoint(g_img, b_img, grad, b_grad)
        expect_within(o['field_a'], fa, b_fa, f'{label} field_a = g_I grad')

    # (2) energy of css
    E = R.energy(o['css'])
    chain = R.energy_chain(tuple(smp.state_dims), ffd)
    for c in range(C):
        expect_close(float(o['stats'][c, _lib.STAT_ENERGY]), float(E[c]), float(R.energy_bound(E[c:c + 1], chain)[0]),
                     f'{label} energy chain {c}')

    # (9) regulariser scalars and Adam step, from the kernel's own energy, the hyper-parameters before the step and the
    # sampler's C-ABI config (what reg_hyper_kernel reads)
    scalars, slots = R.reg_hyper(o['stats'][:, _lib.STAT_ENERGY].tolist(), o['hyper0'].double(), R.reg_config(smp._cconf))
    for c, (reg, coef) in enumerate(scalars):
        expect_close(float(o['stats'][c, _lib.STAT_REG]), reg, 1e-12 * abs(reg) + 1e-300, f'{label} REG chain {c}')
        expect_close(float(o['stats'][c, _lib.STAT_REG_COEF]), coef, 1e-12 * abs(coef), f'{label} REG_COEF chain {c}')
    for k, (ref, bound) in slots.items():
        expect_close(float(o['hyper'][k]), ref, bound, f'{label} regulariser hyper[{k}]')

    # (11) regulariser gradient + SGD update
    k = [float(np.float32(o['stats'][c, _lib.STAT_REG_COEF])) for c in range(C)]
    if torch.count_nonzero(o['moving'] - o['moving'].reshape(-1)[0]) == 0:
        if cfg.svf_steps <= 2:
            assert torch.count_nonzero(o['field_a']) == 0, 'constant image: the data gradient must vanish'
        g_css, b_css = torch.zeros_like(o['css']), None
    else:
        assert cfg.svf_steps == 1 and not ffd, 'a data gradient is composed through one squaring step only'
        g_css, b_css = SVF.bwd_step(o['css'], 0.5, o['field_a'], 0.5)
    ref, bound = R.sgd_grad(o['css'], o['sigma'], g_css, k, b_css)
    expect_within(o['grad_v'], ref, bound, f'{label} grad_v')
    expect_within(o['v'], *R.sgd_step(o['v0'], o['grad_v'], cfg.tau), f'{label} SGD update v')


# (n, C, data, s, K, reg, learnable, svf_steps, sigma, jitter, velocity, const_moving, cps, chain_offset)
CASES = {
    # warp and data term: smooth velocities, the two KK sweeps, every LCC radius, SSD, injected and Philox jitter
    'lcc-s1-K4-16': (16, 2, 'lcc', 1, 4, 'lognormal', True, 1, 'shared', 'inject', 'smooth', False, None, 0),
    'lcc-s2-K5-13': (13, 3, 'lcc', 2, 5, 'lognormal', True, 1, 'per_chain', 'philox', 'smooth', False, None, 5),
    'lcc-s3-K8-24': (24, 1, 'lcc', 3, 8, 'lognormal', False, 1, 'none', 'inject', 'smooth', False, None, 0),
    'ssd-K1-17': (17, 2, 'ssd', 2, 1, 'l2', True, 1, 'per_chain', 'philox', 'smooth', False, None, 1),
    'ssd-K1-12-steps4': (12, 2, 'ssd', 2, 1, 'lognormal', True, 4, 'none', 'inject', 'smooth', True, None, 0),
    # border positions: constant integer / half-integer displacements (L2 regulariser: their energy is 0)
    'border-lcc-K4-12': (12, 3, 'lcc', 2, 4, 'l2', True, 1, 'none', 'none', 'constant', False, None, 0),
    'border-ssd-9': (9, 3, 'ssd', 2, 1, 'l2', False, 1, 'shared', 'inject', 'constant', False, None, 0),
    # regulariser stencil alone (constant moving image): interior / face paths, vec / scalar sweeps, 64^3 epilogue
    'stencil-W8': (8, 2, 'lcc', 1, 4, 'lognormal', True, 1, 'per_chain', 'inject', 'smooth', True, None, 0),
    'stencil-W12': (12, 1, 'lcc', 2, 8, 'lognormal', False, 2, 'shared', 'philox', 'smooth', True, None, 0),
    'stencil-W64': (64, 2, 'lcc', 2, 4, 'lognormal', True, 2, 'shared', 'inject', 'smooth', True, None, 0),
    'stencil-W9': (9, 3, 'ssd', 2, 1, 'lognormal', True, 1, 'per_chain', 'none', 'smooth', True, None, 0),
    'stencil-W33': (33, 1, 'lcc', 1, 5, 'l2', True, 2, 'none', 'inject', 'smooth', True, None, 0),
    # SVFFD_3D: non-cubic state grids (11, 7, 8) with W % 4 == 0 and (11, 8, 7) with W % 4 != 0
    'ffd-2-4-3': (16, 2, 'lcc', 2, 4, 'lognormal', True, 2, 'per_chain', 'inject', 'smooth', True, (2, 4, 3), 0),
    'ffd-2-3-4': (16, 3, 'ssd', 2, 1, 'l2', True, 1, 'shared', 'philox', 'smooth', True, (2, 3, 4), 0),
}


@pytest.mark.parametrize('name', list(CASES))
def test_step_stages(emul, name):
    n, C, data, s, K, reg, learnable, steps, sigma, jitter, velocity, const, cps, off = CASES[name]
    o = run_step(emul, n, C, data, s, K, reg, learnable, steps, sigma, jitter, velocity, const, cps, off,
                 seed=sum(map(ord, name)))
    check_stages(o, name, s)
