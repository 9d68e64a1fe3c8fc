"""
Hausdorff distance and its percentile on the device (ops.surface_distances, utils.calc_HD_GPU, the Trainer's with_HD) against
the host restatement utils.calc_HD_host, element by element: bit-equal for unit and dyadic spacings, where every squared
distance is exact in fp32, and within 1e-6 relative otherwise; inf and 0 exactly.  Also against brute force, for determinism
and independence of the batching, and for the ASD of the same call being average_surface_distance's to the bit.
"""
import numpy as np
import pytest
import torch

from tests.test_gpu_surface_distance import assert_agree, make_case

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
NON_DYADIC = (0.7, 1.3, 0.9)


@pytest.fixture(scope='module')
def pkg(built):
    import irsgmcmc_b200.utils as U
    from irsgmcmc_b200 import ops
    return U, ops


def host_hd(a, b, labels, spacing, q=95.0):
    """(HD, HD_q), (C, L) each, through calc_HD_host; a: (1 or C, 1, D, H, W), b: (C, 1, D, H, W)"""
    from irsgmcmc_b200.utils.util import calc_HD_host
    a, b = (t.cpu().numpy() if torch.is_tensor(t) else t for t in (a, b))
    hd, hq = np.zeros((b.shape[0], len(labels))), np.zeros((b.shape[0], len(labels)))
    for c in range(b.shape[0]):
        fa, fb = a[min(c, a.shape[0] - 1), 0], b[c, 0]
        for j, lab in enumerate(labels):
            hd[c, j], hq[c, j] = calc_HD_host(fa == lab, fb == lab, spacing, q)
    return hd, hq


def assert_hd(got, want, spacing):
    """bit-equal for unit / dyadic spacings, 1e-6 relative otherwise; inf and 0 exactly in both cases"""
    got = got.cpu().numpy() if torch.is_tensor(got) else np.asarray(got)
    err = assert_agree(got, want)
    if tuple(spacing) != NON_DYADIC:
        assert np.array_equal(got, want), (got, want)
    return err


@pytest.mark.parametrize('spacing', [(1.0, 1.0, 1.0), (1.0, 1.5, 2.0), NON_DYADIC])
@pytest.mark.parametrize('q', [95.0, 50.0, 99.0])
def test_against_host_restatement(pkg, spacing, q):
    U, ops = pkg
    a, b, labels = make_case()
    want_hd, want_q = host_hd(a, b, labels, spacing, q)
    assert np.isinf(want_hd[:, 5:7]).all() and np.isinf(want_hd[:, 8]).all() and (want_hd[:, 7] == 0).all()
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    asd, hd, hq = ops.surface_distances(ta, tb, labels, spacing, q)
    for t in (asd, hd, hq):
        assert t.dtype == torch.float64 and t.shape == (3, len(labels)) and t.is_cuda
    e1, e2 = assert_hd(hd, want_hd, spacing), assert_hd(hq, want_q, spacing)
    print(f'spacing {spacing} q {q}: max relative difference from calc_HD_host {max(e1, e2):.2e}')
    assert torch.equal(asd, ops.average_surface_distance(ta, tb, labels, spacing))
    # seg_a per chain (chain stride D*H*W) instead of shared (stride 0)
    per_chain = ops.surface_distances(ta.expand(3, -1, -1, -1, -1).contiguous(), tb, labels, spacing, q)
    assert all(torch.equal(x, y) for x, y in zip(per_chain, (asd, hd, hq)))
    # the helper with calc_ASD_GPU's signature, fixed volume expanded over the chains as the Trainer passes it
    structures = {f's{l}': l for l in labels}
    g_hd, g_q = U.calc_HD_GPU(3, ta.expand(3, -1, -1, -1, -1), tb, structures, torch.tensor(spacing), q)
    assert np.array_equal(g_hd, hd.cpu().numpy()) and np.array_equal(g_q, hq.cpu().numpy())
    # per-chain fixed volumes that differ
    a2 = np.concatenate([a, b[:2]], 0)[[0, 1, 2]]
    _, hd2, hq2 = ops.surface_distances(torch.from_numpy(a2).to(DEV), tb, labels, spacing, q)
    w_hd2, w_q2 = host_hd(a2, b, labels, spacing, q)
    assert_hd(hd2, w_hd2, spacing)
    assert_hd(hq2, w_q2, spacing)


def test_extreme_percentiles(pkg):
    """q = 100 is the Hausdorff distance itself; q = 0 is the larger of the two directed minima"""
    U, ops = pkg
    a, b, labels = make_case(seed=3)
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    for spacing in ((1.0, 1.0, 1.0), (1.0, 1.5, 2.0)):
        _, hd, h100 = ops.surface_distances(ta, tb, labels, spacing, 100.0)
        assert torch.equal(hd, h100)
        _, hd0, h0 = ops.surface_distances(ta, tb, labels, spacing, 0.0)
        assert torch.equal(hd0, hd)
        assert_hd(h0, host_hd(a, b, labels, spacing, 0.0)[1], spacing)
        fin = torch.isfinite(hd)
        assert (h0[fin] <= hd[fin]).all()


def test_more_than_32_labels(pkg):
    U, ops = pkg
    rng = np.random.default_rng(4)
    shape = (20, 22, 19)
    a = np.zeros(shape, np.int16)
    for l in range(1, 41):
        z, y, x = rng.integers(0, 16, 3)
        a[z:z + rng.integers(1, 6), y:y + rng.integers(1, 7), x:x + rng.integers(1, 5)] = l
    b = np.stack([np.where(rng.random(shape) < 0.03, rng.integers(1, 42, shape), np.roll(a, c + 1, axis=c)).astype(np.int16)
                  for c in range(2)])
    labels = list(range(1, 43))
    spacing = (1.0, 1.5, 2.0)
    want_hd, want_q = host_hd(a[None, None], b[:, None], labels, spacing)
    _, hd, hq = ops.surface_distances(torch.from_numpy(a[None, None]).to(DEV), torch.from_numpy(b[:, None]).to(DEV), labels,
                                      spacing)
    assert_hd(hd, want_hd, spacing)
    assert_hd(hq, want_q, spacing)


def test_against_brute_force(pkg):
    from irsgmcmc_b200.utils.util import _label_contour
    U, ops = pkg
    n = 14
    zz, yy, xx = np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing='ij')
    a = (zz - 6.0) ** 2 + (yy - 7.0) ** 2 + (xx - 6.5) ** 2 <= 16.0
    b = (zz - 7.0) ** 2 / 1.5 + (yy - 6.0) ** 2 + (xx - 7.5) ** 2 <= 14.0
    sa = torch.from_numpy(np.where(a, 3, 0).astype(np.int16))[None, None].to(DEV)
    sb = torch.from_numpy(np.stack([np.where(b, 3, 0), np.where(a, 3, 0), np.zeros_like(a, dtype=np.int64)]).astype(np.int16))
    for spacing in ((1.0, 1.5, 2.0), NON_DYADIC):
        ca, cb = _label_contour(a), _label_contour(b)
        pa = np.argwhere(ca) * np.array(spacing[::-1])
        pb = np.argwhere(cb) * np.array(spacing[::-1])
        dist = np.sqrt(((pa[:, None, :] - pb[None, :, :]) ** 2).sum(-1))
        for q in (95.0, 62.5):
            want_hd = max(dist.min(1).max(), dist.min(0).max())
            want_q = max(np.percentile(dist.min(1), q), np.percentile(dist.min(0), q))
            _, hd, hq = (t.cpu().numpy()[:, 0] for t in ops.surface_distances(sa, sb[:, None].to(DEV), [3], spacing, q))
            assert abs(hd[0] - want_hd) <= 1e-6 * want_hd and abs(hq[0] - want_q) <= 1e-6 * want_q
            assert hd[1] == hq[1] == 0.0 and hd[2] == hq[2] == float('inf')


def test_deterministic_and_independent_of_batching(pkg):
    U, ops = pkg
    a, b, labels = make_case(C=4, seed=1)
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    sp = (1.0, 1.5, 2.0)
    one = ops.surface_distances(ta, tb, labels, sp)
    again = ops.surface_distances(ta, tb, labels, sp)
    single_pairs = ops.surface_distances(ta, tb, labels, sp, workspace_bytes=1)   # one pair per batch
    assert all(torch.equal(x, y) and torch.equal(x, z) for x, y, z in zip(one, again, single_pairs))
    assert torch.equal(one[0], ops.average_surface_distance(ta, tb, labels, sp))
    # more pairs than one launch group (48 boxes) in one batch
    b2 = np.concatenate([b] * 4, 0)
    many = ops.surface_distances(ta, torch.from_numpy(b2).to(DEV), labels, sp)
    assert all(torch.equal(x, y.repeat(4, 1)) for x, y in zip(many, one))


def test_custom_op_matches_wrapper(pkg):
    U, ops = pkg
    a, b, labels = make_case(C=2, seed=2)
    ta, tb = torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)
    got = torch.ops.irsgmcmc.surface_distances(ta, tb, labels, [1.0, 1.5, 2.0], 90.0)
    assert all(torch.equal(x, y) for x, y in zip(got, ops.surface_distances(ta, tb, labels, [1.0, 1.5, 2.0], 90.0)))
    with pytest.raises(RuntimeError, match='unsupported'):
        ops.surface_distances(ta, tb, [0, 1], [1.0, 1.0, 1.0])
    with pytest.raises(ValueError, match='percentile'):
        ops.surface_distances(ta, tb, [1], [1.0, 1.0, 1.0], 101.0)


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
    hd, hq = U.calc_HD_GPU(C, seg_f.expand(C, -1, -1, -1, -1), seg_w, structures, (1.0, 1.0, 1.0))
    want_hd, want_q = host_hd(seg_f, seg_w, list(STRUCTURE_LABELS), (1.0, 1.0, 1.0))
    assert np.isfinite(want_hd).all() and (want_hd > 0).any()
    assert np.array_equal(hd, want_hd) and np.array_equal(hq, want_q)
    print(f'256^3, {C} chains x {len(structures)} structures: HD and HD95 bit-equal to calc_HD_host; '
          f'mean HD {hd.mean():.3f}, mean HD95 {hq.mean():.3f} voxels')


def _recording(monkeypatch, util, name):
    seen = []
    fn = getattr(util, name)

    def rec(no_samples, seg_fixed, seg_moving, *args, **kw):
        seen.append((seg_fixed[:no_samples].clone(), seg_moving[:no_samples].clone()))
        return fn(no_samples, seg_fixed, seg_moving, *args, **kw)
    monkeypatch.setattr(util, name, rec)
    return seen


def test_run_MCMC_with_HD(pkg, monkeypatch):
    """per kept sample, 'HD' / 'HD95' equal calc_HD_GPU on the segmentations that sample warped (and calc_HD_host); 'ASD',
    the posterior moments, the Dice scores and the chain states are bit-identical with the flag on and off"""
    U, ops = pkg
    import irsgmcmc_b200.utils.util as util
    from tests.test_gpu_seg_posterior import _trainer
    n, C = 32, 3
    t0 = _trainer(n, C)
    plain = t0._run_MCMC(speed_test_iters=0, with_ASD=True, with_seg_posterior=True)
    seen = _recording(monkeypatch, util, 'calc_surface_distances_GPU')
    t = _trainer(n, C)
    res = t._run_MCMC(speed_test_iters=0, with_ASD=True, with_seg_posterior=True, with_HD=True)
    assert set(res) == set(plain) | {'HD', 'HD95'}
    for key in ('mean', 'std_dev', 'im_mean', 'im_std'):
        assert torch.equal(res[key], plain[key]), key
    assert torch.equal(t.sampler.v, t0.sampler.v)
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(res['DSC'], plain['DSC']))
    assert all(np.array_equal(x, y) for x, y in zip(res['ASD'], plain['ASD']))
    # one call per kept sample, then one for the majority segmentation of the posterior
    assert len(res['HD']) == len(res['HD95']) == len(res['ASD']) == len(seen) - 1 == 6
    labels = list(t.structures_dict.values())
    for hd, hq, (sf, sw) in zip(res['HD'], res['HD95'], seen[:-1]):
        assert hd.shape == hq.shape == (C, len(labels))
        g_hd, g_q = U.calc_HD_GPU(C, sf, sw, t.structures_dict, t.im_spacing)
        assert np.array_equal(hd, g_hd) and np.array_equal(hq, g_q)
        w_hd, w_q = host_hd(sf, sw, labels, (1.0, 1.0, 1.0))
        assert np.array_equal(hd, w_hd) and np.array_equal(hq, w_q)
    P, P0 = res['seg_posterior'], plain['seg_posterior']
    assert torch.equal(P['majority'], P0['majority'])
    seg_f = t.fixed['seg'].to(DEV)
    m_hd, m_q = (x[0] for x in U.calc_HD_GPU(1, seg_f, P['majority'], t.structures_dict, t.im_spacing))
    for j, name in enumerate(t.structures_dict):
        e = P['structures'][name]
        assert set(e) == set(P0['structures'][name]) | {'HD_majority', 'HD95_majority'}
        assert e['ASD_majority'] == P0['structures'][name]['ASD_majority']
        assert e['HD_majority'] == m_hd[j] and e['HD95_majority'] == m_q[j]
    # HD alone (no ASD), another percentile: the key follows it
    res99 = _trainer(n, C)._run_MCMC(speed_test_iters=0, with_HD=True, HD_percentile=99.0)
    assert 'HD99' in res99 and 'HD95' not in res99 and isinstance(res99['ASD'], str)
    assert all(np.array_equal(x, y) for x, y in zip(res99['HD'], res['HD']))
    assert torch.equal(res99['mean'], plain['mean'])


def test_test_VI_with_HD(pkg):
    from tests.test_gpu_seg_posterior import _trainer
    U, ops = pkg
    S = 4
    t = _trainer(16, 1)
    t.config['trainer'].update(no_iters_VI=2, no_samples_VI_test=S)
    t._run_VI()
    torch.manual_seed(5)
    plain = t._test_VI(speed_test_samples=0, with_ASD=True, with_seg_posterior=True)
    torch.manual_seed(5)
    res = t._test_VI(speed_test_samples=0, with_ASD=True, with_seg_posterior=True, with_HD=True)
    assert set(res) == set(plain) | {'HD', 'HD95'}
    assert torch.equal(res['mean'], plain['mean']) and np.array_equal(res['ASD'], plain['ASD'])
    assert res['HD'].shape == res['HD95'].shape == (S, len(t.structures_dict))
    assert (res['HD95'][np.isfinite(res['HD'])] <= res['HD'][np.isfinite(res['HD'])]).all()
    P = res['seg_posterior']
    seg_f = t.fixed['seg'].to(DEV)
    m_hd, m_q = (x[0] for x in U.calc_HD_GPU(1, seg_f, P['majority'], t.structures_dict, t.im_spacing))
    for j, name in enumerate(t.structures_dict):
        assert P['structures'][name]['HD_majority'] == m_hd[j] and P['structures'][name]['HD95_majority'] == m_q[j]
    torch.manual_seed(5)
    only = t._test_VI(speed_test_samples=0, with_ASD=False, with_HD=True)
    assert np.array_equal(only['HD'], res['HD']) and np.array_equal(only['HD95'], res['HD95'])
