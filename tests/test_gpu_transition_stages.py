"""
The Langevin + Sobolev proposal and the four LCC box passes of the SGLD transition, voxel by voxel, against the fp64
references of tests/helpers/transition_ref.py.  No voxel is exempt: every result must lie within the reference's
rounding bound.  Each stage is fed the kernel's own output of the stage before it (a, rs, ga), so errors never compound.
Every case prints max(|err| / bound) and its median, so the margin is visible.

Langevin (csrc/irs_smooth.cu irs_launch_langevin_smooth3): 3 / 5 / 7 taps with W % 4 == 0 run the fused kernel
(noise + x + y on shared-memory rows, TY rows per CTA, halo rows regenerate their Philox numbers) and a z pass; 9 taps
the vectorised four-pass sequence; 11 - 15 taps, W % 4 != 0 or a misaligned v the scalar one.  Philox noise is taken from
the unfused generator at the same (seed, iteration, chain0): langevin_sobolev(0, None, 1, []) is exactly eps in fp32.
W = 160 and W = 1216 put the end of a round of the fused kernel's in-place x pass (512 float4 units) inside a row; before a
round took whole rows, the first unit of the next round read an already smoothed left neighbour there.

LCC (csrc/irs_data.cu box_march_kernel): 32 x 8 tiles that march along z segments of box_seg_len planes; the adjoint folds
the replicate padding back onto the faces.  box_seg_len gives segments of 8 planes (D itself when D < 8) to every case of
test_lcc_passes whatever its chain count: C = 1, 2, 3 and 7 exercise grid.y there.  test_lcc_ten_plane_segments takes a
volume with enough tiles per chain that 7 chains stop the halving at 10 planes.
"""
import pytest
import torch

from tests.helpers import transition_ref as R
from tests.util import smooth_field

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def lib(built):
    from irsgmcmc_b200 import _lib
    return _lib.load()


def expect_within(out, ref, bound, what):
    nbad, at, r, med = R.worst(out.cpu(), ref.cpu(), bound.cpu())
    print(f'{what}: max |err| / bound = {r:.3g}, median {med:.3g}')
    assert nbad == 0, f'{what}: {nbad} voxels outside the bound; worst (chain, component, z, y, x) = {at} at {r:.3g} x bound'


def misaligned(t):
    """a copy of t that starts 4 bytes past a 16-byte boundary (no float4 access possible)"""
    buf = torch.zeros(t.numel() + 8, device=DEV)
    out = buf[1:1 + t.numel()].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 == 4
    return out


# ---- Langevin proposal + Sobolev smoothing -----------------------------------------------------------------------------------
def sobolev_taps(s):
    from irsgmcmc_b200.utils.functions import Sobolev_kernel_1D
    return [float(t) for t in Sobolev_kernel_1D(s, 0.5)[0]]


def check_langevin(shape, C, s, sigma_mode='shared', coef=0.9, noise='philox', chain0=0, iteration=0, misalign=False):
    from irsgmcmc_b200.utils.functions import langevin_sobolev
    g = torch.Generator().manual_seed(hash((shape, C, s)) % 1000)
    v = 2.0 * torch.randn(C, 3, *shape, generator=g)
    sigma = {'none': None, 'shared': torch.rand(1, 3, *shape, generator=g) + 0.5,
             'per_chain': torch.rand(C, 3, *shape, generator=g) + 0.5}[sigma_mode]
    taps = sobolev_taps(s) if s else []
    vd = v.to(DEV)
    if misalign:
        vd = misaligned(vd)
    sd = None if sigma is None else sigma.to(DEV)
    seed = 1234 + s
    if noise == 'explicit':
        eps = torch.randn(C, 3, *shape, generator=g)
        out = langevin_sobolev(vd, sd, coef, taps, eps=eps.to(DEV))
    else:
        eps = langevin_sobolev(torch.zeros(C, 3, *shape, device=DEV), None, 1.0, [], seed=seed, iteration=iteration,
                               chain0=chain0).cpu()
        out = langevin_sobolev(vd, sd, coef, taps, seed=seed, iteration=iteration, chain0=chain0)
    ref, bound = R.langevin_smooth(v, sigma, coef, eps, taps)
    expect_within(out, ref, bound, f'langevin {shape} C={C} s={s} sigma={sigma_mode} coef={coef} {noise} '
                                   f'chain0={chain0} iter={iteration}{" misaligned" if misalign else ""}')


LANGEVIN_SHAPES = [((5, 6, 8), 'TY=H'), ((7, 40, 16), 'ytiles'), ((4, 72, 12), 'ytiles-partial'),
                   ((3, 40, 256), 'TY24'), ((4, 40, 160), 'rows-across-rounds')]
LANGEVIN_CASES = [(shape, s, tag) for shape, tag in LANGEVIN_SHAPES for s in (1, 2, 3)] + \
                 [((5, 12, 20), s, 'vec4pass' if s == 4 else 'scalar4pass') for s in (4, 5, 6, 7)] + \
                 [((4, 9, 13), s, 'Wodd') for s in (1, 3)]


@pytest.mark.parametrize('noise', ['philox', 'explicit'])
@pytest.mark.parametrize('shape,s,tag', LANGEVIN_CASES, ids=[f'{t}-{"x".join(map(str, sh))}-s{s}'
                                                            for sh, s, t in LANGEVIN_CASES])
def test_langevin_paths(lib, shape, s, tag, noise):
    check_langevin(shape, 2, s, noise=noise, chain0=1 if noise == 'philox' else 0)


@pytest.mark.parametrize('W,path', [(1216, 'fused'), (1220, 'unfused')])
def test_langevin_widest_rows(lib, W, path):
    """W = 1216 with 7 taps is the widest row whose smallest tile (8 + 6 rows) fits in 200 KB; 1220 no longer fits.  The
    rows are wider than a round of the x pass (4 W / 512 threads), so a round ends inside a row"""
    check_langevin((2, 12, W), 1, 3, noise='philox', chain0=2, iteration=7)


@pytest.mark.parametrize('sigma_mode', ['none', 'shared', 'per_chain'])
@pytest.mark.parametrize('C,chain0,iteration', [(1, 0, 0), (3, 5, 2 ** 40 + 3)])
def test_langevin_sigma_and_counters(lib, sigma_mode, C, chain0, iteration):
    for s in (3, 5):
        check_langevin((6, 20, 24), C, s, sigma_mode, noise='philox', chain0=chain0, iteration=iteration)


@pytest.mark.parametrize('s', [2, 6])
def test_langevin_misaligned(lib, s):
    for noise in ('philox', 'explicit'):
        check_langevin((4, 10, 16), 2, s, 'per_chain', noise=noise, misalign=True)


@pytest.mark.parametrize('s', [0, 1, 3, 5])
def test_langevin_coef_zero_is_pure_smoothing(lib, s):
    check_langevin((6, 17, 32), 2, s, 'shared', coef=0.0, noise='philox')


# ---- LCC normalisation and its adjoint -----------------------------------------------------------------------------------------
def lcc_image(C, shape, seed):
    """smooth intensities plus noise, a constant slab (zero local variance: rs = 1e5) and a sharp step"""
    g = torch.Generator().manual_seed(seed)
    im = 0.5 + 0.4 * smooth_field((C, 1, *shape), 1.0, seed, passes=2) + 0.05 * torch.randn(C, 1, *shape, generator=g)
    D = shape[0]
    im[:, :, : max(1, D // 4)] = 0.25
    im[..., shape[2] // 2:] += 0.3
    return im.contiguous()


def impulse_gradient(C, shape, seed):
    """impulses at every position class: faces, edges, corners, x / y tile edges (0, 31, 32; 7, 8, 15, 16), the first and
    last planes of z segments of 8 (7, 8, 15, 16) and of 10 (9, 10, 19, 20, 29, 30) and interiors; chains alternate"""
    D, H, W = shape
    g = torch.Generator().manual_seed(seed)
    out = torch.zeros(C, 1, D, H, W)
    xs = sorted({0, 1, W // 2, 31, 32, W - 2, W - 1} & set(range(W)))
    ys = sorted({0, 1, H // 2, 7, 8, 15, 16, H - 2, H - 1} & set(range(H)))
    zs = sorted({0, 1, D // 2, 7, 8, 9, 10, 15, 16, 19, 20, 29, 30, D - 2, D - 1} & set(range(D)))
    i = 0
    for z in zs:
        for y in ys:
            for x in xs:
                out[i % C, 0, z, y, x] = torch.randn(1, generator=g).item()
                i += 1
    return out


def lcc_gradients(C, shape, seed):
    g = torch.Generator().manual_seed(seed)
    dense = torch.randn(C, 1, *shape, generator=g)
    D, H, W = shape
    z = torch.arange(D).view(D, 1, 1)
    planes = ~(((z % 8) < 2) | (z == D - 1))       # whole zero planes: a segment's first planes and the last face
    return {'dense': dense, 'impulses': impulse_gradient(C, shape, seed + 1), 'zero_planes': dense * planes}


def check_lcc(lib, C, shape, S, label):
    from irsgmcmc_b200 import _lib, ops
    im = lcc_image(C, shape, 7 * S + shape[0])
    zn, a, rs = ops.lcc_normalise(im.to(DEV), S)
    expect_within(a, *R.lcc_fwd_mean(im, S), f'{label} FWD_MEAN a')
    (rs_ref, b_rs), (z_ref, b_z) = R.lcc_fwd_var(a.cpu(), None, S)
    expect_within(rs, rs_ref, b_rs, f'{label} FWD_VAR rs')
    expect_within(zn, z_ref, b_z, f'{label} FWD_VAR z')
    D, H, W = shape
    for name, G in lcc_gradients(C, shape, 11 * S).items():
        Gd = G.to(DEV)
        work = torch.full_like(a, float('nan'))
        g_im = torch.full_like(a, float('nan'))
        _lib.check(lib.irs_lcc_normalise_bwd(_lib.ptr(Gd), _lib.ptr(a), _lib.ptr(rs), S, _lib.ptr(work),
                                             _lib.ptr(g_im), C, D, H, W, _lib.stream()))
        expect_within(work, *R.lcc_bwd_var(G, 1.0, a.cpu(), rs.cpu(), S), f'{label} g={name} BWD_VAR')
        expect_within(g_im, *R.lcc_bwd_mean(work.cpu(), S), f'{label} g={name} BWD_MEAN')


LCC_CASES = [(C, shape, S) for S in (1, 2, 3) for C, shape in
             [(2, (40, 13, 40)), (1, (20, 24, 70)), (7, (19, 16, 33)), (2, (6, 9, 13))]] + \
            [(2, (n, n, n), S) for S in (1, 2, 3) for n in range(2, 2 * S + 1)] + \
            [(1, (3, 17, 2), 3), (3, (2, 5, 64), 2)]


@pytest.mark.parametrize('C,shape,S', LCC_CASES, ids=[f'C{C}-{"x".join(map(str, sh))}-S{S}' for C, sh, S in LCC_CASES])
def test_lcc_passes(lib, C, shape, S):
    check_lcc(lib, C, shape, S, f'lcc C={C} {shape} S={S}')


def box_seg_len(C, D, H, W):
    """the z segment length the launcher picks (csrc/irs_data.cu box_seg_len)"""
    tiles = -(-W // 32) * -(-H // 8) * C
    n = D
    while n > 8 and tiles * -(-D // n) < 2 * 1184:
        n = (n + 1) // 2
    return n if n >= 8 else (D if D < 8 else 8)


def test_lcc_ten_plane_segments(lib):
    """96 x 256 planes: 7 chains make 672 tiles per segment row, so the halving stops at segments of 10 planes (2 chains
    at 8); impulses sit on their first and last planes"""
    C, shape, S = 7, (40, 96, 256), 2
    assert box_seg_len(C, *shape) == 10 and box_seg_len(2, *shape) == 8
    check_lcc(lib, C, shape, S, f'lcc C={C} {shape} S={S} segments of 10')
