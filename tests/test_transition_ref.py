"""
The per-voxel references of the Langevin + Sobolev proposal and of the LCC box passes (tests/helpers/transition_ref.py),
on the CPU:
  * with fp64 inputs every reference is the exact operation: it equals the oracle (oracle/sgld_oracle.py) to ~1e-12,
    the adjoint passes equal autograd through oracle.lcc_normalise;
  * fp32 evaluations of the same operations in other orders (what a kernel may do) lie within the bounds;
  * the comparator fails a single-voxel and a single-row error that the norm-based checks accept, and a face fold
    weight one short.
"""
import math

import numpy as np
import pytest
import torch

from oracle import sgld_oracle as O
from irsgmcmc_b200.utils.functions import Sobolev_kernel_1D
from tests.helpers import transition_ref as R
from tests.util import grad_ok, rel, smooth_field


def taps_for(s):
    return R.fp32_taps(Sobolev_kernel_1D(s, 0.5)[0])


def close64(a, b, tol=1e-12):
    a, b = a.double(), b.double()
    return float((a - b).abs().max()) <= tol * max(1.0, float(b.abs().max()))


# ---- fp64: the references are the exact operations ----------------------------------------------------------------------
@pytest.mark.parametrize('s,shape', [(1, (5, 6, 8)), (2, (4, 9, 7)), (3, (3, 2, 11)), (3, (7, 7, 7))])
def test_langevin_smooth_equals_oracle(s, shape):
    C = 2
    g = torch.Generator().manual_seed(s)
    v, eps = torch.randn(C, 3, *shape, generator=g).double(), torch.randn(C, 3, *shape, generator=g).double()
    sigma = (torch.rand(1, 3, *shape, generator=g) + 0.5).double()
    taps = taps_for(s)
    out, bound = R.langevin_smooth(v, sigma, 0.5, eps, taps)   # coef 0.5 = sqrt(2 tau) at tau = 1/8, exact in fp32
    ref = O.sobolev_smooth(O.langevin_proposal(v, sigma, 0.125, eps), taps)
    assert close64(out, ref)
    assert bool((bound > 0).all())
    out0, _ = R.langevin_smooth(v, None, 0.0, None, taps)
    assert close64(out0, O.sobolev_smooth(v, taps))
    p, _ = R.langevin_smooth(v, None, 0.5, eps, [])
    assert close64(p, v + 0.5 * eps)


@pytest.mark.parametrize('S,shape', [(1, (2, 2, 2)), (1, (9, 10, 33)), (2, (3, 4, 5)), (2, (6, 17, 9)), (3, (2, 5, 7)),
                                     (3, (8, 8, 8)), (3, (13, 4, 3))])
def test_lcc_passes_equal_oracle(S, shape):
    C = 2
    g = torch.Generator().manual_seed(10 * S + shape[0])
    im = (smooth_field((C, 1, *shape), 1.0, S, passes=1) + 0.1 * torch.randn(C, 1, *shape, generator=g)).double()
    a, _ = R.lcc_fwd_mean(im, S)
    (rs, _), (zn, _) = R.lcc_fwd_var(a, None, S)
    im_ad = im.clone().requires_grad_(True)
    zn_ad = O.lcc_normalise(im_ad, S)
    assert close64(zn, zn_ad.detach())
    zF = torch.randn(C, 1, *shape, generator=g).double()
    _, (z, _) = R.lcc_fwd_var(a, zF, S)
    assert close64(z, zF - zn_ad.detach())
    G = torch.randn(C, 1, *shape, generator=g).double()
    (zn_ad * G).sum().backward()
    for sign in (1.0, -1.0):
        ga, _ = R.lcc_bwd_var(G, sign, a, rs, S)
        gi, _ = R.lcc_bwd_mean(ga, S)
        assert close64(gi, sign * im_ad.grad)


def test_box_adjoint_is_the_transpose():
    """<B x, y> = <x, B^T y> for every n from 1 to 2S + 2 along every axis (the fold at both faces)"""
    g = torch.Generator().manual_seed(3)
    for S in (1, 2, 3):
        for n in range(1, 2 * S + 3):
            x = torch.randn(1, 1, n, n + 1, 2, generator=g).double()
            y = torch.randn(1, 1, n, n + 1, 2, generator=g).double()
            lhs = (R._box(x, S) * y).sum()
            rhs = (x * R._box(y, S, adjoint=True)).sum()
            assert abs(float(lhs - rhs)) <= 1e-12 * float(R._box(x.abs(), S).sum() * y.abs().max())


# ---- fp32 evaluations in the kernels' orders lie within the bounds --------------------------------------------------------
def within(out, ref, bound, what):
    nbad, at, r, med = R.worst(out, ref, bound)
    print(f'{what}: max |err| / bound = {r:.3g}, median {med:.3g}')
    assert nbad == 0, f'{what}: {nbad} voxels outside the bound, worst at {at} ({r:.3g} x bound)'


def smooth32(x, w, order):
    for axis in order:
        x = R.filter_axis(x, axis, w)   # fp32 in, fp32 out: every product and sum rounds in fp32
    return x


@pytest.mark.parametrize('s', [1, 2, 3, 5])
def test_langevin_fp32_within_bound(s):
    C, shape = 2, (9, 12, 16)
    g = torch.Generator().manual_seed(20 + s)
    v = 3.0 * torch.randn(C, 3, *shape, generator=g)
    eps, sigma = torch.randn(C, 3, *shape, generator=g), torch.rand(C, 3, *shape, generator=g) + 0.5
    coef, taps = math.sqrt(0.8), taps_for(s)
    w32 = [np.float32(t) for t in taps]
    p32 = v + (np.float32(coef) * sigma) * eps
    ref, bound = R.langevin_smooth(v, sigma, coef, eps, taps)
    for order in ((2, 3, 4), (4, 3, 2)):
        within(smooth32(p32, w32, order), ref, bound, f'langevin s={s} order={order}')


@pytest.mark.parametrize('S,shape', [(1, (6, 9, 33)), (2, (4, 5, 3)), (3, (10, 9, 8))])
def test_lcc_fp32_within_bound(S, shape):
    C = 2
    g = torch.Generator().manual_seed(30 + S)
    im = 100.0 + 5.0 * smooth_field((C, 1, *shape), 1.0, S, passes=1) + torch.randn(C, 1, *shape, generator=g)
    inv_k3 = np.float32(1.0 / (2 * S + 1) ** 3)
    box32 = lambda x, adj=False: R.smooth3(x, [1.0] * (2 * S + 1), adj)
    a32 = im - box32(im) * inv_k3
    within(a32, *R.lcc_fwd_mean(im, S), f'FWD_MEAN S={S}')
    rs32 = 1.0 / torch.sqrt(box32(a32 * a32) * inv_k3 + np.float32(1e-10))
    zF = torch.randn(C, 1, *shape, generator=g)
    (rs, b_rs), (z, b_z) = R.lcc_fwd_var(a32, zF, S)
    within(rs32, rs, b_rs, f'FWD_VAR rs S={S}')
    within(zF - a32 * rs32, z, b_z, f'FWD_VAR z S={S}')
    G = torch.randn(C, 1, *shape, generator=g)
    ga32 = -G * rs32 + 2.0 * a32 * (box32(-0.5 * -G * a32 * rs32 * rs32 * rs32, True) * inv_k3)
    within(ga32, *R.lcc_bwd_var(G, -1.0, a32, rs32, S), f'BWD_VAR S={S}')
    within(ga32 - box32(ga32, True) * inv_k3, *R.lcc_bwd_mean(ga32, S), f'BWD_MEAN S={S}')


# ---- the comparator sees what the norm checks miss ------------------------------------------------------------------------
def _face_tap(x, S):
    """one extra fold copy of every far-x-face voxel in B^T(x) at that face: its own tap, boxed over y and z"""
    face = torch.zeros_like(x)
    face[..., -1] = x[..., -1]
    return R.filter_axis_adjoint(R.filter_axis_adjoint(face, 2, [1.0] * (2 * S + 1)), 3, [1.0] * (2 * S + 1))[..., -1]


def test_comparator_catches_local_errors():
    """one voxel off by 1e-4 of its magnitude and one row scaled by 1 + 2e-5 pass rel < 1e-5 and grad_ok, but not the
    bound; neither does a far-face fold weight one short"""
    S, C, shape = 2, 2, (12, 16, 20)
    k3 = float((2 * S + 1) ** 3)
    g = torch.Generator().manual_seed(40)
    im = 10.0 + smooth_field((C, 1, *shape), 1.0, 4, passes=1) + 0.2 * torch.randn(C, 1, *shape, generator=g)
    a32 = R.lcc_fwd_mean(im, S)[0].float()
    rs32 = R.lcc_fwd_var(a32, None, S)[0][0].float()
    G = torch.randn(C, 1, *shape, generator=g)
    ga32 = R.lcc_bwd_var(G, 1.0, a32, rs32, S)[0].float()
    ref, bound = R.lcc_bwd_mean(ga32, S)
    good = ref.float()
    assert R.worst(good, ref, bound)[0] == 0

    one = good.clone()
    one[1, 0, 5, 7, 9] *= 1.0 + 1e-4
    row = good.clone()
    row[0, 0, 3, 15, :] *= 1.0 + 2e-5                                 # the last row of a 32 x 8 tile
    for what, bad in (('one voxel', one), ('one row', row)):
        assert R.worst(bad, ref, bound)[0] > 0, what
        assert rel(bad, ref) < 1e-5, what
        assert grad_ok(bad, good, ref, what)
    adj = R._box(ga32.double(), S, adjoint=True)
    adj[..., -1] -= _face_tap(ga32.double(), S)
    fold = (ga32.double() - adj / k3).float()
    assert R.worst(fold, ref, bound)[0] > 0
