"""
Average surface distance on the device (ops.average_surface_distance, utils.calc_ASD_GPU, calc_metrics) against the host
restatement utils.util.calc_ASD_host, element by element, and against a brute-force evaluation of the definition.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def pkg(built):
    import irsgmcmc_b200.utils as U
    from irsgmcmc_b200 import ops
    return U, ops


def host_asd(a, b, labels, spacing):
    """(C, L) through calc_ASD_host; a: (1 or C, 1, D, H, W), b: (C, 1, D, H, W)"""
    from irsgmcmc_b200.utils.util import calc_ASD_host
    a, b = (t.cpu().numpy() if torch.is_tensor(t) else t for t in (a, b))
    out = np.zeros((b.shape[0], len(labels)))
    for c in range(b.shape[0]):
        fa, fb = a[min(c, a.shape[0] - 1), 0], b[c, 0]
        for j, lab in enumerate(labels):
            out[c, j] = calc_ASD_host(fa == lab, fb == lab, spacing)
    return out


def assert_agree(got, want, tol=1e-6):
    got = np.asarray(got)
    assert got.shape == want.shape and got.dtype == np.float64
    assert np.array_equal(np.isinf(got), np.isinf(want)), (got, want)
    assert np.array_equal(got == 0.0, want == 0.0), (got, want)
    fin = np.isfinite(want) & (want != 0.0)
    err = np.abs(got[fin] - want[fin]) / want[fin]
    assert err.size == 0 or err.max() <= tol, (err.max(), got, want)
    return 0.0 if err.size == 0 else float(err.max())


def _grid(shape):
    return np.meshgrid(*(np.arange(n, dtype=np.float64) for n in shape), indexing='ij')


def make_case(shape=(40, 46, 53), C=3, seed=0):
    """labelled volumes (1, 1, D, H, W) and (C, 1, D, H, W) exercising every case of the definition"""
    D, H, W = shape
    zz, yy, xx = _grid(shape)

    def ellipsoid(c, r):
        return ((zz - c[0]) / r[0]) ** 2 + ((yy - c[1]) / r[1]) ** 2 + ((xx - c[2]) / r[2]) ** 2 <= 1.0

    def blobs(k):
        from tests.util import smooth_field
        f = smooth_field((1, 1, D, H, W), 1.0, seed=k, passes=4)[0, 0].numpy()
        return f > 0.35

    a = np.zeros(shape, np.int16)
    a[ellipsoid((12, 20, 18), (7, 9, 8))] = 1
    a[blobs(1 + 10 * seed)] = 2
    a[~ellipsoid((D / 2, H / 2, W / 2), (D / 2.6, H / 2.6, W / 2.6))] = 3      # touches all six faces
    a[5, 40, 3] = 4                                                             # single voxel
    a[1:4, 1:4, 1:4] = 5                                                        # two far-apart components
    a[D - 4:D - 1, H - 5:H - 2, W - 4:W - 1] = 5
    a[ellipsoid((30, 12, 40), (3, 4, 5))] = 6                                   # absent from every moving volume
    a[ellipsoid((25, 30, 30), (4, 4, 6))] = 8                                   # identical in every moving volume
    bs = []
    for c in range(C):
        b = np.zeros(shape, np.int16)
        b[ellipsoid((13 + c, 19, 19 - c), (6 + c, 9, 7))] = 1
        b[blobs(2 + c + 10 * seed)] = 2
        b[~ellipsoid((D / 2 + c, H / 2, W / 2 - c), (D / 2.4, H / 2.7, W / 2.5))] = 3
        b[7 + c, 38, 5 + 2 * c] = 4
        b[2:5, 2 + c:5 + c, 1:3] = 5
        b[D - 3:D, H - 4:H - 1, W - 6 + c:W - 2 + c] = 5
        b[ellipsoid((10, 35, 12), (3, 3, 3 + c))] = 7                           # absent from the fixed volume
        b[a == 8] = 8
        bs.append(b)
    labels = [1, 2, 3, 4, 5, 6, 7, 8, 9]                                        # 9: absent from both
    return a[None, None], np.stack(bs)[:, None], labels


@pytest.mark.parametrize('spacing', [(1.0, 1.0, 1.0), (1.0, 1.5, 2.0)])
def test_against_host_restatement(pkg, spacing):
    U, ops = pkg
    a, b, labels = make_case()
    want = host_asd(a, b, labels, spacing)
    assert np.isinf(want[:, 5:7]).all() and np.isinf(want[:, 8]).all() and (want[:, 7] == 0).all()
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    shared = ops.average_surface_distance(ta, tb, labels, spacing)
    assert shared.dtype == torch.float64 and shared.shape == (3, len(labels)) and shared.is_cuda
    assert_agree(shared.cpu().numpy(), want)
    # seg_a per chain (chain stride D*H*W) instead of shared (stride 0)
    per_chain = ops.average_surface_distance(ta.expand(3, -1, -1, -1, -1).contiguous(), tb, labels, spacing)
    assert torch.equal(per_chain, shared)
    # the drop-in helper with the reference's signature, fixed volume expanded over the chains as the Trainer passes it
    structures = {f's{l}': l for l in labels}
    got = U.calc_ASD_GPU(3, ta.expand(3, -1, -1, -1, -1), tb, structures, torch.tensor(spacing))
    assert isinstance(got, np.ndarray) and np.array_equal(got, shared.cpu().numpy())
    # per-chain fixed volumes that differ
    a2 = np.concatenate([a, b[:2]], 0)[[0, 1, 2]]
    assert_agree(ops.average_surface_distance(torch.from_numpy(a2).to(DEV), tb, labels, spacing).cpu().numpy(),
                 host_asd(a2, b, labels, spacing))


def test_more_than_32_labels(pkg):
    U, ops = pkg
    rng = np.random.default_rng(4)
    shape = (20, 22, 19)
    # 40 labels in blocks of random size, plus voxel noise
    a = np.zeros(shape, np.int16)
    for l in range(1, 41):
        z, y, x = rng.integers(0, 16, 3)
        a[z:z + rng.integers(1, 6), y:y + rng.integers(1, 7), x:x + rng.integers(1, 5)] = l
    b = np.stack([np.where(rng.random(shape) < 0.03, rng.integers(1, 42, shape), np.roll(a, c + 1, axis=c)).astype(np.int16)
                  for c in range(2)])
    labels = list(range(1, 43))
    want = host_asd(a[None, None], b[:, None], labels, (1.0, 1.5, 2.0))
    got = ops.average_surface_distance(torch.from_numpy(a[None, None]).to(DEV), torch.from_numpy(b[:, None]).to(DEV), labels,
                                       (1.0, 1.5, 2.0))
    assert_agree(got.cpu().numpy(), want)


def test_against_brute_force(pkg):
    """the shapes of tests/test_writers.py::test_average_surface_distance_against_brute_force, on the device"""
    from irsgmcmc_b200.utils.util import _label_contour
    U, ops = pkg
    n = 14
    zz, yy, xx = _grid((n, n, n))
    a = (zz - 6.0) ** 2 + (yy - 7.0) ** 2 + (xx - 6.5) ** 2 <= 16.0
    b = (zz - 7.0) ** 2 / 1.5 + (yy - 6.0) ** 2 + (xx - 7.5) ** 2 <= 14.0
    spacing = (1.0, 1.5, 2.0)
    ca, cb = _label_contour(a), _label_contour(b)
    pa = np.argwhere(ca) * np.array(spacing[::-1])
    pb = np.argwhere(cb) * np.array(spacing[::-1])
    dist = np.sqrt(((pa[:, None, :] - pb[None, :, :]) ** 2).sum(-1))
    want = 0.5 * (dist.min(1).mean() + dist.min(0).mean())
    sa = torch.from_numpy(np.where(a, 3, 0).astype(np.int16))[None, None].to(DEV)
    sb = torch.from_numpy(np.stack([np.where(b, 3, 0), np.where(a, 3, 0), np.zeros_like(a, dtype=np.int64)]).astype(np.int16))
    got = ops.average_surface_distance(sa, sb[:, None].to(DEV), [3], spacing).cpu().numpy()[:, 0]
    assert abs(got[0] - want) <= 1e-9 * want and got[1] == 0.0 and got[2] == float('inf')


def test_configuration_4_size(pkg):
    """256^3 make_pair segmentations warped by an SGLD sampler with 4 chains, all 15 structures"""
    U, ops = pkg
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    n, C = 256, 4
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=DEV)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=DEV)
    s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
    s.init_gmm(sigma_hat=0.7)
    s.step(3, use_graph=False)
    seg_w = s.warp_segmentation()
    seg_f = fixed['seg'].to(DEV)
    structures = {f's{l}': l for l in STRUCTURE_LABELS}
    got = U.calc_ASD_GPU(C, seg_f.expand(C, -1, -1, -1, -1), seg_w, structures, (1.0, 1.0, 1.0))
    want = host_asd(seg_f, seg_w, list(STRUCTURE_LABELS), (1.0, 1.0, 1.0))
    assert np.isfinite(want).all() and (want > 0).any()   # near-aligned pair: some warped structures coincide (ASD 0)
    err = assert_agree(got, want)
    print(f'256^3, {C} chains x {len(structures)} structures: max relative difference from calc_ASD_host {err:.2e}')
    ASD, DSC = U.calc_metrics(seg_f.expand(C, -1, -1, -1, -1), seg_w, structures, torch.tensor([1.0, 1.0, 1.0]), no_samples=C)
    assert np.array_equal(ASD, got) and DSC.shape == (C, len(structures))


def test_deterministic_and_independent_of_batching(pkg):
    U, ops = pkg
    a, b, labels = make_case(C=4, seed=1)
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    one = ops.average_surface_distance(ta, tb, labels, (1.0, 1.5, 2.0))
    again = ops.average_surface_distance(ta, tb, labels, (1.0, 1.5, 2.0))
    single_pairs = ops.average_surface_distance(ta, tb, labels, (1.0, 1.5, 2.0), workspace_bytes=1)   # one pair per batch
    assert torch.equal(one, again) and torch.equal(one, single_pairs)
    # more pairs than one launch group (48 boxes) in one batch
    b2 = np.concatenate([b] * 4, 0)
    many = ops.average_surface_distance(ta, torch.from_numpy(b2).to(DEV), labels, (1.0, 1.5, 2.0))
    assert torch.equal(many, one.repeat(4, 1))


def test_custom_op_matches_wrapper(pkg):
    U, ops = pkg
    a, b, labels = make_case(C=2, seed=2)
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    assert torch.equal(torch.ops.irsgmcmc.average_surface_distance(ta, tb, labels, [1.0, 1.5, 2.0]),
                       ops.average_surface_distance(ta, tb, labels, [1.0, 1.5, 2.0]))
    with pytest.raises(RuntimeError, match='unsupported'):
        ops.average_surface_distance(ta, tb, [0, 1], [1.0, 1.0, 1.0])
    with pytest.raises(RuntimeError, match='bad argument'):
        ops.average_surface_distance(ta, tb, [1], [1.0, 0.0, 1.0])


def test_run_MCMC_with_ASD(pkg, monkeypatch):
    """Trainer._run_MCMC(with_ASD=True): an ASD array (chains, structures) per kept sample, equal to calc_ASD_host on the
    segmentations the kept sample warped"""
    U, ops = pkg
    import irsgmcmc_b200.model as M
    import irsgmcmc_b200.utils.util as util
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.trainer import Trainer
    from tests.test_gpu_dropin import _reference_style_config
    n, C = 32, 2
    torch.manual_seed(5)
    fixed, moving, vp = make_pair(n)
    structures = {f's{l}': l for l in STRUCTURE_LABELS}
    seen = []
    calc_metrics = util.calc_metrics

    def recording(seg_fixed, seg_moving, *args, **kw):
        seen.append((seg_fixed.clone(), seg_moving.clone()))
        return calc_metrics(seg_fixed, seg_moving, *args, **kw)
    monkeypatch.setattr(util, 'calc_metrics', recording)
    spacing = (1.0, 1.5, 2.0)
    t = Trainer(_reference_style_config(C), fixed, moving, vp, structures_dict=structures, device=torch.device(DEV),
                im_spacing=spacing)
    gmm = M.GMM(4, 2).to(DEV)
    gmm.init_parameters(0.7)
    reg = M.RegLoss_LogNormal(w_reg=1.6, diff_op='GradientOperator', dims=(n, n, n), learnable=True).to(DEV)
    res = t._run_MCMC(gmm, reg, speed_test_iters=0, with_ASD=True)
    assert len(res['ASD']) == len(res['DSC']) == len(seen) == 3
    for asd, (sf, sw) in zip(res['ASD'], seen):
        assert asd.shape == (C, len(structures))
        assert_agree(asd, host_asd(sf, sw, list(STRUCTURE_LABELS), spacing))
