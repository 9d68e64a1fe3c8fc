"""
Every scaling-and-squaring step and every adjoint step of csrc/irs_svf.cu, voxel by voxel, against the fp64 reference that
takes the kernels' own fp32 decisions (tests/helpers/svf_step_ref.py).  No voxel is exempt: each result must lie within
the reference's rounding bound, and the max |u_k| and the cell maps the forward pass leaves must be bit-equal.

Forward: the input of step k is the kernel's own hist[k - 1], so each step is checked in isolation.
Adjoint: ops.svf_exp_bwd reads only v, hist[0 .. n-2] and the maxabs block, so a test builds them itself with one
non-zero step input U at step k.  A step whose input is zero maps g to exactly 2 g, hence g_v = 2^(n-1) 2^-n A_U^T g.
"""
import pytest
import torch

from tests.helpers import svf_step_ref as R
from tests.util import smooth_field

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def ops(built):
    from irsgmcmc_b200 import ops
    return ops


def chains(n, C, amp, seed):
    """C chains with different content, so that the TMA dimension 3 C is really indexed"""
    return torch.cat([smooth_field((1, 3, n, n, n), amp * (1.0 - 0.1 * c), seed + 17 * c) for c in range(C)]).contiguous()


def misaligned(t):
    """a copy of t that starts 4 bytes past a 16-byte boundary (the TMA unit cannot address it)"""
    buf = torch.zeros(t.numel() + 8, device=DEV)
    out = buf[1:1 + t.numel()].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 == 4
    return out


def expect_within(out, ref, bound, what):
    nbad, at, r = R.worst(out, ref, bound)
    assert nbad == 0, f'{what}: {nbad} voxels outside the bound; worst (chain, component, z, y, x) = {at} at {r:.3g} x bound'


# ---- forward ------------------------------------------------------------------------------------------------------------
def run_forward(v, n_steps):
    """the C ABI with hist pre-filled with NaN (a voxel the pass does not write fails) and a maxabs block pre-filled with
    -1 (maps the pass does not write must keep it)"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    C, _, D, H, W = v.shape
    assert lib.irs_svf_maxabs_floats(C, D, H, W, n_steps) == R.maxabs_floats(C, D, H, W, n_steps)
    hist = torch.full((n_steps, C, 3, D, H, W), float('nan'), device=DEV)
    block = torch.full((R.maxabs_floats(C, D, H, W, n_steps),), -1.0, device=DEV)
    _lib.check(lib.irs_svf_exp_fwd(_lib.ptr(v), _lib.ptr(hist), _lib.ptr(block), n_steps, C, D, H, W, _lib.stream()))
    torch.cuda.synchronize()
    return hist, block


def check_forward(v, n_steps, label):
    C, _, D, H, W = v.shape
    hist, block = run_forward(v, n_steps)
    glob, maps = R.split_maxabs(block, n_steps, C, D, H, W)
    k_first = n_steps - 4 if n_steps > 4 else 1   # svf_cells_kernel covers the last four steps
    for k in range(n_steps):
        u, s = (v, 2.0 ** -n_steps) if k == 0 else (hist[k - 1], 1.0)
        ref, bound = R.fwd_step(u, s)
        expect_within(hist[k], ref, bound, f'{label} step {k}')
        m = R.max_abs(u, s)
        assert torch.equal(glob[k], m), f'{label} step {k}: maxabs {glob[k].item()!r} != {m.item()!r}'
        if k >= k_first and R.gather_radius(glob[k].item()) >= 2:
            assert torch.equal(maps[k], R.cell_map(u, s)), f'{label} step {k}: cell map'
        else:
            assert bool((maps[k] == -1.0).all()), f'{label} step {k}: a cell map nobody reads was written'
    return glob


FWD_CASES = [  # n, C, amp; TMA for n % 4 == 0 (exact and partial 32 x 8 tiles), rings for 17 / 33
    (16, 3, 0.8), (16, 1, 10.0), (20, 2, 4.0), (20, 3, 0.8), (36, 1, 10.0), (36, 2, 4.0), (40, 3, 10.0), (40, 1, 4.0),
    (64, 2, 10.0), (64, 1, 0.8), (17, 2, 10.0), (17, 3, 0.8), (33, 1, 4.0), (33, 2, 10.0)]


@pytest.mark.parametrize('n,C,amp', FWD_CASES, ids=[f'n{n}-C{C}-amp{a:g}' for n, C, a in FWD_CASES])
def test_forward_steps(n, C, amp):
    v = chains(n, C, amp, 31).to(DEV)
    glob = check_forward(v, 12, f'n={n} C={C} amp={amp}')
    if amp == 10.0:   # the late steps reach the per-voxel fallback (>= 0.999) and the wide ring (2 max|u_{k-1}| >= 3)
        assert float(glob[-1]) > 2.0 and float(glob[-2]) >= 1.5


def test_forward_steps_misaligned():
    """n = 32 whose v starts 4 bytes past a 16-byte boundary: every step takes the ring kernels (scalar loads only)"""
    v = misaligned(chains(32, 2, 10.0, 37).to(DEV))
    check_forward(v, 12, 'misaligned n=32')


@pytest.mark.parametrize('n,C', [(16, 2), (40, 3), (17, 2), (32, 1)])
def test_forward_threshold_inputs(n, C):
    """n_steps = 1, v = 2 U: U holds +-0.999, +-0.9989999, +-1, +-1.999, +-2, integers, halves and positions on or
    rounding onto the volume's faces, at voxels on tile edges"""
    U = R.threshold_field(n, C, 5)
    check_forward((2.0 * U).to(DEV), 1, f'threshold n={n}')


SEG_CASES = [('IRS_SVF_SEG_FWD', 4, 40), ('IRS_SVF_SEG_FWD', 5, 40), ('IRS_SVF_SEG_FWD', 40, 40), ('IRS_SVF_SEG', 4, 17),
             ('IRS_SVF_SEG', 6, 33)]


@pytest.mark.parametrize('var,seg,n', SEG_CASES, ids=[f'{v}={s}-n{n}' for v, s, n in SEG_CASES])
def test_forward_forced_segments(monkeypatch, var, seg, n):
    monkeypatch.setenv(var, str(seg))
    v = chains(n, 2, 10.0, 41).to(DEV)
    check_forward(v, 12, f'{var}={seg} n={n}')


# ---- adjoint, one step at a time ------------------------------------------------------------------------------------------
def bump_field(n, C, base, bump, seed):
    """small smooth field plus a local Gaussian bump: |u| reaches `bump` voxels near one point only"""
    U = chains(n, C, base, seed)
    z, y, x = torch.meshgrid(torch.arange(n), torch.arange(n), torch.arange(n), indexing='ij')
    c = torch.tensor([0.62 * n, 0.55 * n, 0.4 * n])
    w = torch.exp(-((z - c[0]) ** 2 + (y - c[1]) ** 2 + (x - c[2]) ** 2) / (2 * (0.08 * n + 1.0) ** 2))
    return (U + bump * w * torch.tensor([1.0, -0.8, 0.6]).view(1, 3, 1, 1, 1)).contiguous()


def regime_field(n, C, regime, seed):
    if regime == 'small':      # max |U| < 0.999: the TMA kernel everywhere
        return chains(n, C, 0.9, seed)
    if regime == 'bump12':     # 1 <= max |U| < 2: ring tiles next to TMA tiles through the per-tile window
        return bump_field(n, C, 0.3, 1.6, seed)
    return bump_field(n, C, 0.3, 4.5, seed)   # 'bump3': global gathers and the scatter companion


def impulse_positions(n, C):
    """(chain, z, y, x) at every position class: tile interiors, x / y tile edges and corners of 32 x 8 and 32 x 16
    tiles, first / last planes of z segments of 4, 5, 8 and 10 planes, volume faces, edges and corners; chains alternate"""
    xs = sorted({0, 10, 31, 32, n - 1} & set(range(n)))
    ys = sorted({0, 5, 7, 8, 12, 15, 16, n - 1} & set(range(n)))
    zs = sorted({0, 3, 4, 5, 7, 8, 9, 10, 15, 16, 19, 20, n - 1} & set(range(n)))
    pos = []
    for i, z in enumerate(zs):
        for j, y in enumerate(ys):
            for k, x in enumerate(xs):
                if (i + j + k) % 3 == 0 or z in (0, n - 1) and y in (0, n - 1):
                    pos.append(((i + j + k) % C, z, y, x))
    return pos


def gradients(n, C, seed):
    """the incoming gradients the adjoint is driven with"""
    gen = torch.Generator().manual_seed(seed)
    dense = torch.randn(C, 3, n, n, n, generator=gen)
    z, y, x = torch.meshgrid(torch.arange(n), torch.arange(n), torch.arange(n), indexing='ij')
    mask = torch.zeros(C, 1, n, n, n, dtype=torch.bool)   # blobs with sharp edges (gradient vanishes off the mask)
    for c in range(C):
        for _ in range(5):
            ctr = torch.rand(3, generator=gen) * n
            r = 2.0 + torch.rand(1, generator=gen).item() * n / 5
            mask[c, 0] |= (z - ctr[0]) ** 2 + (y - ctr[1]) ** 2 + (x - ctr[2]) ** 2 < r * r
    imp = torch.zeros(C, 3, n, n, n)
    for c, zz, yy, xx in impulse_positions(n, C):
        imp[c, int(torch.randint(3, (1,), generator=gen)), zz, yy, xx] = torch.randn(1, generator=gen).item()
    halo = ((y % 8 == 0) | (y % 8 == 7)).view(1, 1, n, n, n)   # only rows that are halo rows of a neighbouring tile
    planes = ~(((z % 8) < 2) | ((z >= 8) & (z < 16)) | (z == n - 1)).view(1, 1, n, n, n)   # whole zero planes / segment
    return {'dense': dense, 'blobs': dense * mask, 'impulses': imp, 'halo_rows': dense * halo, 'zero_planes': dense * planes}


STEPS = [(1, 0), (2, 1), (6, 1), (12, 8), (12, 11)]
REGIMES = [('small', 2), ('small', 0), ('bump12', 2), ('bump12', 1), ('bump3', 0), ('bump3', 1), ('bump3', 2), ('bump3', 3),
           ('bump3', 8)]


def check_adjoint_step(ops, U, n_steps, k, radius_max, label, misalign=False, grads=None):
    """g_v of the public op against 1/2 A_U^T g (k >= 1) or A_v^T g with in_scale = out_scale = 1/2 (k = 0)"""
    C, _, n = U.shape[:3]
    Ud = U.to(DEV)
    hist = torch.zeros(n_steps, C, 3, n, n, n, device=DEV)
    block = torch.zeros(R.maxabs_floats(C, n, n, n, n_steps), device=DEV)
    glob, maps = R.split_maxabs(block, n_steps, C, n, n, n)
    glob[k] = R.max_abs(Ud, 1.0)
    if k == 0:
        assert n_steps == 1
        v = 2.0 * Ud
        step, out_scale, factor = R.Step(v, 0.5), 0.5, 1.0
    else:
        v = torch.zeros_like(Ud)
        hist[k - 1] = Ud
        maps[k] = R.cell_map(Ud, 1.0)
        step, out_scale, factor = R.Step(Ud, 1.0), 1.0, 0.5
    if misalign:
        v = misaligned(v)
    for name, g in (grads or gradients(n, C, 50 + k)).items():
        gd = g.to(DEV)
        g_v = ops.svf_exp_bwd(v, hist, block, gd, radius_max)
        ref, bound, _ = step.bwd(gd, out_scale)
        expect_within(g_v, factor * ref, factor * bound, f'{label} g={name}')


ADJ_CASES = [(st, rg) for st in STEPS for rg in REGIMES]


@pytest.mark.parametrize('steps,regime', ADJ_CASES, ids=[f'n40C2-{s[0]}_{s[1]}-{r[0]}-r{r[1]}' for s, r in ADJ_CASES])
def test_adjoint_step(ops, steps, regime):
    n_steps, k = steps
    U = regime_field(40, 2, regime[0], 60)
    check_adjoint_step(ops, U, n_steps, k, regime[1], f'n=40 C=2 (n_steps, k)={steps} {regime}')


RING_CASES = [((n_steps, k), rg, n, C, mis) for n, C, mis, sts, rgs in
              [(17, 2, False, [(1, 0), (2, 1), (12, 11)], [('small', 2), ('bump12', 2), ('bump3', 0), ('bump3', 3)]),
               (32, 1, True, [(1, 0), (12, 11)], [('small', 2), ('bump3', 2)])]
              for (n_steps, k) in sts for rg in rgs]


@pytest.mark.parametrize('steps,regime,n,C,mis', RING_CASES,
                         ids=[f'n{n}C{C}{"-misaligned" if m else ""}-{s[0]}_{s[1]}-{r[0]}-r{r[1]}'
                              for s, r, n, C, m in RING_CASES])
def test_adjoint_step_rings(ops, steps, regime, n, C, mis):
    """the non-TMA kernels: a row pitch the TMA unit cannot address, and a v 4 bytes past a 16-byte boundary (the ring
    kernels and svf_step_bwd_scatter_kernel load v, hist and the gradients with scalar loads only)"""
    n_steps, k = steps
    U = regime_field(n, C, regime[0], 70)
    check_adjoint_step(ops, U, n_steps, k, regime[1], f'n={n} C={C} misaligned={mis} (n_steps, k)={steps} {regime}',
                       misalign=mis)


SEGB_CASES = [('IRS_SVF_SEG_BWD', s, rg) for s in (4, 5, 40) for rg in [('small', 2), ('bump12', 2), ('bump3', 3)]] + \
             [('IRS_SVF_SEG', 4, ('bump12', 2)), ('IRS_SVF_SEG', 4, ('bump3', 0))]


@pytest.mark.parametrize('var,seg,regime', SEGB_CASES, ids=[f'{v}={s}-{r[0]}-r{r[1]}' for v, s, r in SEGB_CASES])
def test_adjoint_step_forced_segments(ops, monkeypatch, var, seg, regime):
    monkeypatch.setenv(var, str(seg))
    n = 40 if var == 'IRS_SVF_SEG_BWD' else 17
    U = regime_field(n, 2, regime[0], 80)
    for n_steps, k in ((12, 11), (12, 8), (1, 0)):
        check_adjoint_step(ops, U, n_steps, k, regime[1], f'{var}={seg} n={n} (n_steps, k)=({n_steps}, {k}) {regime}')


def test_adjoint_window_edge(ops, monkeypatch):
    """one source just below a tile's z-range moves 1.5 voxels into it: with segments of 5 planes the segment 25..29 reads
    cells down to z = 23 (cell 2), so its window must see that source and leave the one-voxel TMA kernel"""
    monkeypatch.setenv('IRS_SVF_SEG_BWD', '5')
    n, C = 40, 1
    U = chains(n, C, 0.5, 95)
    U[0, 2, 23, 20, 12] = 1.5
    g = {'dense': torch.randn(C, 3, n, n, n, generator=torch.Generator().manual_seed(96))}
    for n_steps, k in ((12, 11), (12, 8), (2, 1)):
        check_adjoint_step(ops, U, n_steps, k, 2, f'window edge (n_steps, k)=({n_steps}, {k})', grads=g)


# ---- the natural pipeline ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n,C', [(64, 2), (128, 1)])
def test_composite_twelve_steps(ops, n, C):
    """the 12-step adjoint of the kernel's own forward history against compose(): the g_u / g_work ping-pong, the scale of
    step 0 and the order of the scatter companions"""
    v = chains(n, C, 10.0, 90).to(DEV)
    hist, maxabs = ops.svf_exp_fwd(v, 12)
    assert float(maxabs[-1]) > 2.0
    g = gradients(n, C, 91)['blobs'].to(DEV)
    ref, bound = R.compose(v, hist, g, 12)
    for radius_max in (2, 8):
        g_v = ops.svf_exp_bwd(v, hist, maxabs, g, radius_max)
        expect_within(g_v, ref, bound, f'composite n={n} C={C} radius_max={radius_max}')

