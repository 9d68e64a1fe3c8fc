"""
CPU checks of tests/helpers/svf_step_ref.py, the per-voxel oracle of the scaling-and-squaring steps: the reference against
the oracle's ATen pipeline in fp64, against the host emulation of the kernels' per-voxel bodies within its rounding
bound, and the comparator's power: it rejects corruptions that the global acceptance rule `grad_ok` lets through.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sgld_oracle as O
from tests.helpers import svf_step_ref as R
from tests.helpers.svf_step_ref import threshold_field
from tests.util import grad_ok, smooth_field


@pytest.fixture(scope='module')
def emul(built):
    return ctypes.CDLL(built['emul'])


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def no_face_field(n, C, seed):
    """a field whose sampling positions keep >= 1e-6 from every cell face over all 12 steps: every component keeps
    one sign and 0.3 <= |v| <= 0.7, so |u_k| lies in (7e-5, 1) and never crosses an integer"""
    g = torch.Generator().manual_seed(seed)
    sign = torch.where(torch.rand(C, 3, 1, 1, 1, generator=g) < 0.5, -1.0, 1.0)
    m = smooth_field((C, 3, n, n, n), 1.0, seed)
    return (sign * (0.5 + 0.2 * m)).double()


def test_composed_reference_matches_aten_fp64():
    n, C, steps = 10, 2, 12
    v = no_face_field(n, C, 3)
    hist = []
    u, s = v, 2.0 ** -steps
    for k in range(steps):
        st = R.Step(u, s)
        for a in range(3):   # the precondition: no unclamped position within 1e-6 of a cell face
            xyz = R._coords(u.shape, u.device, u.dtype)[a]
            q = xyz + st.us64[:, a]
            assert float((q - q.round()).abs().min()) > 1e-6
        out, _ = st.fwd()
        hist.append(out)
        u, s = out, 1.0
    v64 = v.clone().requires_grad_(True)
    _, d64 = O.svf_exp_aten(v64, steps, exact_grid=True)
    d = (hist[-1] - d64.detach()).abs().max()
    assert float(d) <= 1e-12 * float(d64.abs().max()), float(d)

    G = torch.randn(C, 3, n, n, n, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    g_aten, = torch.autograd.grad((d64 * G).sum(), v64)
    g_ref, _ = R.compose(v, hist, G, steps)
    d = (g_ref - g_aten).abs().max()
    assert float(d) <= 1e-12 * float(g_aten.abs().max()), float(d)


def _emul_step(emul, v, g):
    """the host emulation of one step (n_steps = 1, in_scale = out_scale = 1/2): hist, maxabs and both adjoint modes"""
    C, _, n = v.shape[:3]
    vn = np.ascontiguousarray(v.numpy())
    hist, maxabs = np.zeros((1,) + vn.shape, np.float32), np.zeros(1, np.float32)
    emul.emul_svf_fwd(P(vn), P(hist), P(maxabs), 1, C, n, n, n)
    gn = np.ascontiguousarray(g.numpy())
    outs = []
    for mode in (0, 1):   # gather with radius floor(maxabs) + 1 / scatter
        gv = np.zeros_like(vn)
        emul.emul_svf_bwd(P(vn), P(hist), P(maxabs), P(gn), P(gv), 1, mode, C, n, n, n)
        outs.append(torch.from_numpy(gv))
    return torch.from_numpy(hist[0]), float(maxabs[0]), outs


@pytest.mark.parametrize('n,C,field', [(12, 2, 'smooth0.8'), (17, 1, 'smooth4'), (12, 3, 'smooth10'), (20, 2, 'threshold'),
                                       (33, 1, 'threshold')])
def test_reference_vs_host_emulation_one_step(emul, n, C, field):
    if field == 'threshold':
        U = threshold_field(n, C, 5)
    else:
        U = smooth_field((C, 3, n, n, n), float(field[6:]), 7)
    v = (2.0 * U).contiguous()   # n_steps = 1: u_0 = v / 2 = U exactly
    g = torch.randn(C, 3, n, n, n, generator=torch.Generator().manual_seed(8))
    hist, m, gvs = _emul_step(emul, v, g)
    ref, bound = R.fwd_step(v, 0.5)
    nbad, at, r = R.worst(hist, ref, bound)
    assert nbad == 0, f'forward: {nbad} voxels outside the bound, worst {at} at {r:.2f} x bound'
    assert np.float32(m) == R.max_abs(v, 0.5).item()
    ref, bound = R.bwd_step(v, 0.5, g, 0.5)
    for mode, gv in enumerate(gvs):
        nbad, at, r = R.worst(gv, ref, bound)
        assert nbad == 0, f'adjoint mode {mode}: {nbad} voxels outside the bound, worst {at} at {r:.2f} x bound'


def test_reference_vs_host_emulation_twelve_steps(emul):
    """every forward step against its own input, and the whole adjoint against compose() within the propagated bound"""
    n, C, steps = 12, 2, 12
    v = smooth_field((C, 3, n, n, n), 6.0, 9)
    vn = np.ascontiguousarray(v.numpy())
    hist, maxabs = np.zeros((steps,) + vn.shape, np.float32), np.zeros(steps, np.float32)
    emul.emul_svf_fwd(P(vn), P(hist), P(maxabs), steps, C, n, n, n)
    hist = torch.from_numpy(hist)
    assert float(maxabs[-1]) > 2.0
    for k in range(steps):
        u, s = (v, 2.0 ** -steps) if k == 0 else (hist[k - 1], 1.0)
        ref, bound = R.fwd_step(u, s)
        assert R.worst(hist[k], ref, bound)[0] == 0, k
        assert np.float32(maxabs[k]) == R.max_abs(u, s).item(), k
    g = torch.randn(C, 3, n, n, n, generator=torch.Generator().manual_seed(10))
    ref, bound = R.compose(v, hist, g, steps)
    for mode in (0, 1):
        gv = np.zeros_like(vn)
        emul.emul_svf_bwd(P(vn), P(hist.numpy()), P(maxabs), P(np.ascontiguousarray(g.numpy())), P(gv), steps, mode, C, n, n, n)
        nbad, at, r = R.worst(torch.from_numpy(gv), ref, bound)
        assert nbad == 0, f'mode {mode}: {nbad} voxels outside the bound, worst {at} at {r:.2f} x bound'


def test_comparator_rejects_what_grad_ok_accepts(emul):
    """one adjoint step at 40^3 (|u| <= 0.75): a correct fp32 result (the host emulation) passes the per-voxel comparison;
    one voxel off by 1e-4 S(t), or one 32-voxel row scaled by 0.99, fails it -- while grad_ok, the global rule the
    older SVF tests use, accepts both corruptions"""
    n, C = 40, 1
    v = smooth_field((C, 3, n, n, n), 1.5, 11)
    g = torch.randn(C, 3, n, n, n, generator=torch.Generator().manual_seed(5))
    _, _, (gv, _) = _emul_step(emul, v, g)
    ref, bound = R.bwd_step(v, 0.5, g, 0.5)
    S = R.abs_sum(v, 0.5, g, 0.5)
    assert R.worst(gv, ref, bound)[0] == 0

    v64 = v.double().requires_grad_(True)
    g64, = torch.autograd.grad((O.svf_exp_aten(v64, 1, exact_grid=True)[1] * g.double()).sum(), v64)
    v32 = v.clone().requires_grad_(True)
    g32, = torch.autograd.grad((O.svf_exp_aten(v32, 1)[1] * g).sum(), v32)
    assert grad_ok(gv, g32, g64, 'host emulation, one step')

    for at in [(0, 0, 20, 17, 13), (0, 1, 0, 0, 0), (0, 2, 39, 15, 31), (0, 1, 8, 16, 32)]:
        bad = gv.clone()
        bad[at] += float(1e-4 * S[at])
        assert grad_ok(bad, g32, g64, f'one voxel {at} off by 1e-4 S(t)')
        nbad, worst_at, _ = R.worst(bad, ref, bound)
        assert nbad == 1 and worst_at == at

    bad = gv.clone()
    bad[0, 0, 20, 9, 4:36] *= 0.99
    assert grad_ok(bad, g32, g64, 'one 32-voxel row scaled by 0.99')
    nbad, worst_at, _ = R.worst(bad, ref, bound)
    assert nbad >= 30 and worst_at[:4] == (0, 0, 20, 9)


def test_maxabs_layout():
    """cell_map / split_maxabs agree with the layout of irs_svf_maxabs_floats on a partial-cell volume"""
    C, D, H, W, n_steps = 2, 20, 12, 40, 3
    u = torch.zeros(C, 3, D, H, W)
    u[1, 2, 17, 9, 33] = -5.0
    u[0, 0, 3, 2, 1] = 2.0
    m = R.cell_map(u, 0.25)
    assert m.shape == (C, 3, 2, 2)
    assert m[1, 2, 1, 1] == 1.25 and m[0, 0, 0, 0] == 0.5 and float(m.sum()) == 1.75
    block = torch.zeros(R.maxabs_floats(C, D, H, W, n_steps))
    glob, maps = R.split_maxabs(block, n_steps, C, D, H, W)
    maps[2] = m
    assert block[n_steps + 2 * C * 12 + 12 + 2 * 4 + 1 * 2 + 1] == 1.25   # step 2, chain 1, cell (z 2, y 1, x 1)
    assert R.gather_radius(0.999) == 2 and R.gather_radius(0.9989) == 1 and R.gather_radius(1.999) == 3
