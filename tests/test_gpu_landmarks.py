"""
Landmark registration error and landmark posterior on the device (csrc/irs_landmark.cu): the map kernel bit-equal to the fp64
restatement on fp32 T and cross-checked against ops.warp3d of coordinate ramps, the accumulators against a two-pass mean /
covariance (chains split over launches bit-identical, permuted samples within tolerance), the finish against numpy, the
SGLDSampler integration (nothing else of the sampler changes, checkpoints) and Trainer._run_MCMC / _test_VI(with_TRE=True) on a
make_pair + make_landmarks case.
"""
import numpy as np
import pytest
import torch

from tests.helpers import landmark_ref as ref
from tests.test_landmarks import _field, _landmarks

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def ops(built):
    from irsgmcmc_b200 import ops
    return ops


def _gpu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


# ---- map ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dims,C,P', [((5, 6, 7), 3, 20), ((12, 9, 17), 64, 150), ((8, 8, 8), 1, 1), ((2, 3, 9), 3, 1),
                                      ((6, 10, 4), 3, 300)])
def test_map_bit_equal_to_restatement(ops, dims, C, P):
    """off-grid points, nodes, faces and corners on non-cubic volumes with an asymmetric field (a channel or axis swap is not
    bit-equal); P = 1 and P not a multiple of the block"""
    D, H, W = dims
    T = _field(C, D, H, W, 10)
    p, q = _landmarks(D, H, W, P, 11)
    if P == 1:
        p, q = p[:1], q[:1]
    s = (0.75, 1.25, 2.5)
    pred, tre = ops.landmark_map(_gpu(T), torch.from_numpy(p), torch.from_numpy(q), s)
    want = ref.predict(T, p)
    assert np.array_equal(pred.cpu().numpy(), want)
    assert np.array_equal(tre.cpu().numpy(), ref.tre(want, q, s))
    p2, t2 = torch.ops.irsgmcmc.landmark_map(_gpu(T), _gpu(p), _gpu(q), list(s))
    assert torch.equal(p2, pred) and torch.equal(t2, tre)
    from irsgmcmc_b200.utils import calc_TRE_GPU, calc_TRE_host
    assert np.array_equal(calc_TRE_GPU(_gpu(T), p, q, s), calc_TRE_host(T, p, q, s))


def test_nodes_against_warp3d_of_coordinate_ramps(ops):
    """an independent path: at interior grid nodes, m equals ops.warp3d of the three voxel-coordinate ramps with the same T
    (the warp samples the moving image where m says), within the warp's fp32 position arithmetic"""
    D, H, W = 10, 13, 16
    C = 3
    T = _field(C, D, H, W, 12, scale=0.02)
    T[:, 0] -= np.float32(0.05) * np.arange(W, dtype=np.float32)        # keep the positions inside the volume
    T[:, 2] += np.float32(0.02) * np.arange(D, dtype=np.float32)[:, None, None]
    Tg = _gpu(T)
    z, y, x = torch.meshgrid(*(torch.arange(n, dtype=torch.float32) for n in (D, H, W)), indexing='ij')
    rng = np.random.default_rng(13)
    nodes = np.stack([rng.integers(1, n - 1, 60) for n in (W, H, D)], -1).astype(np.float64)
    pred, _ = ops.landmark_map(Tg, nodes, nodes, (1.0, 1.0, 1.0))
    ni = nodes.astype(np.int64)
    for a, ramp in enumerate((x, y, z)):
        warped = ops.warp3d(ramp.view(1, 1, D, H, W).to(DEV).contiguous(), Tg)[:, 0].cpu().numpy()
        at = warped[:, ni[:, 2], ni[:, 1], ni[:, 0]]
        assert np.abs(pred.cpu().numpy()[..., a] - at).max() < 1e-4 * (D, H, W)[2 - a] + 1e-5, a


# ---- update and finish ------------------------------------------------------------------------------------------------------
def _samples(N, C, P, seed):
    rng = np.random.default_rng(seed)
    pred = rng.standard_normal((N, C, P, 3)) * np.array([0.5, 1.0, 2.0]) + rng.random((P, 3)) * 50
    tre = np.abs(rng.standard_normal((N, C, P))) * 2.0 + 0.1
    return pred, tre


def test_update_against_two_pass_split_and_permuted(ops):
    N, C, P = 6, 16, 150
    pred, tre = _samples(N, C, P, 20)
    acc = torch.zeros(P, 11, device=DEV, dtype=torch.float64)
    split = torch.zeros_like(acc)
    for k in range(N):
        rows = ops.landmark_update(_gpu(pred[k]), _gpu(tre[k]), k * C, acc)
        # sum, sum of squares (landmarks in index order: a sequential sum) and max per chain
        r = rows.cpu().numpy()
        assert np.array_equal(r[:, 0], np.cumsum(tre[k], 1)[:, -1])
        assert np.array_equal(r[:, 1], np.cumsum(tre[k] * tre[k], 1)[:, -1])
        assert np.array_equal(r[:, 2], tre[k].max(1))
        ops.landmark_update(_gpu(pred[k, :7]), _gpu(tre[k, :7]), k * C, split)
        ops.landmark_update(_gpu(pred[k, 7:]), _gpu(tre[k, 7:]), k * C + 7, split)
    a = acc.cpu().numpy()
    assert torch.equal(acc, split)                                       # chains split over two launches: the same bits
    flat_p, flat_t = pred.reshape(N * C, P, 3), tre.reshape(N * C, P)
    assert np.array_equal(a, ref.accumulate(flat_p, flat_t))             # the restatement's own roundings
    tp = ref.two_pass(flat_p, flat_t)
    assert np.allclose(a, tp, rtol=1e-12, atol=1e-12 * np.abs(tp[:, 3:9]).max())
    perm = np.random.default_rng(21).permutation(N * C)
    pacc = torch.zeros_like(acc)
    ops.landmark_update(_gpu(flat_p[perm]), _gpu(flat_t[perm]), 0, pacc)
    assert np.allclose(pacc.cpu().numpy(), tp, rtol=1e-12, atol=1e-12 * np.abs(tp[:, 3:9]).max())
    out = torch.ops.irsgmcmc.landmark_update(_gpu(pred[0]), _gpu(tre[0]), 0, torch.zeros_like(acc))
    assert out.shape == (C, 3)


def test_finish_against_numpy(ops):
    N, C, P = 4, 8, 130
    pred, tre = _samples(N, C, P, 30)
    flat_p, flat_t = pred.reshape(N * C, P, 3), tre.reshape(N * C, P)
    flat_p[:, 5] = flat_p[:1, 5]                                          # identical samples: zero covariance, d^2 = +inf
    rng = np.random.default_rng(31)
    q = flat_p.mean(0) + rng.standard_normal((P, 3))
    q[7] = flat_p[0, 7]
    s = (0.8, 1.0, 1.6)
    for n in (N * C, 1):
        acc = torch.zeros(P, 11, device=DEV, dtype=torch.float64)
        ops.landmark_update(_gpu(flat_p[:n]), _gpu(flat_t[:n]), 0, acc)
        out = ops.landmark_posterior(acc, n, q, s).cpu().numpy()
        want = ref.posterior(acc.cpu().numpy(), n, q, s)
        assert np.allclose(out[:, :5], want[:, :5], rtol=1e-14, atol=0)
        if n == 1:
            assert np.isnan(out[:, 5:]).all()
            continue
        assert np.isinf(out[5, 15]) and (out[5, 6:15] == 0).all()
        ok = np.arange(P) != 5
        assert np.allclose(out[ok, 5:12], want[ok, 5:12], rtol=1e-12, atol=0)
        scale = np.sqrt(np.abs(want[ok, 6:12]).max(1, keepdims=True))
        assert (np.abs(out[ok, 12:15] - want[ok, 12:15]) <= 1e-9 * scale).all()
        assert np.allclose(out[ok, 15], want[ok, 15], rtol=1e-9, atol=1e-300)
        assert torch.equal(torch.ops.irsgmcmc.landmark_posterior(acc, n, _gpu(q), list(s)).cpu(), torch.from_numpy(out))


# ---- sampler ----------------------------------------------------------------------------------------------------------------
LABELS = [10, 11, 12, 13, 16, 17, 18, 26, 49, 50, 51, 52, 53, 54, 58]


def _sampler(C, n=16, chain_offset=0, seed=0):
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    fixed, moving, vp = make_pair(n)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(hyper_mode='per_chain'), device=DEV, chain_offset=chain_offset)
    gen = torch.Generator().manual_seed(seed)
    v0 = 2.0 * torch.randn(4, 3, n, n, n, generator=gen)[chain_offset:chain_offset + C]
    s.set_state(v0, torch.full((1, 3, n, n, n), 0.5))
    s.init_gmm(sigma_hat=0.7)
    return s


def _pairs(n=16, P=40):
    from irsgmcmc_b200.data_loader.synthetic import make_landmarks
    return make_landmarks(n, no_landmarks=P)


SPACING = (1.0, 1.5, 0.8)


def test_accumulate_matches_the_kernels(ops):
    p, q = _pairs()
    a = _sampler(3)
    a.enable_landmark_posterior(p, q, SPACING)
    acc = torch.zeros(p.shape[0], 11, device=DEV, dtype=torch.float64)
    for k in range(4):
        a.step(2)
        T = a.transformation()
        pred, tre = ops.landmark_map(T, p, q, SPACING)
        rows = ops.landmark_update(pred, tre, 3 * k, acc)
        a.accumulate(transformation=T if k % 2 else None)
        assert torch.equal(a.last_landmark_stats, rows)
    assert torch.equal(a._lmpost['acc'], acc) and a._lmpost['n'] == 12
    post = a.landmark_posterior()
    assert post['n'] == 12 and torch.equal(post['table'], ops.landmark_posterior(acc, 12, q, SPACING))
    assert torch.equal(a._lmpost['acc'], acc)   # a query keeps the accumulators
    with pytest.raises(ValueError):
        a.enable_landmark_posterior(p + 20.0, q, SPACING)   # outside the 16^3 volume


def test_sampler_state_unchanged_by_the_feature(ops):
    """moments, split R-hat, label counts, Jacobian accumulators and chain states are bit-identical with the feature on and off"""
    p, q = _pairs()
    outs = []
    for on in (False, True):
        s = _sampler(4)
        s.enable_convergence_diagnostics(6)
        s.enable_segmentation_posterior(LABELS)
        s.enable_jacobian_posterior()
        if on:
            s.enable_landmark_posterior(p, q, SPACING)
        for _ in range(6):
            s.step(2)
            T = s.transformation()
            s.accumulate(seg_warped=s.warp_segmentation(transformation=T), transformation=T)
        torch.cuda.synchronize()
        outs.append((s.posterior_moments(), s.v.clone(), s.hyper.clone(), s._rhat['mean'].clone(), s._rhat['m2'].clone(),
                     s._segpost['counts'].clone(), s._jacpost['folds'].clone(), s._jacpost['mean'].clone(),
                     s._jacpost['m2'].clone()))
        if on:
            assert s._lmpost['n'] == 24
        else:
            assert not s.landmark_posterior_enabled and 'lmpost' not in s.state_dict()
    for key in ('displacement_mean', 'displacement_std', 'im_mean', 'im_std'):
        assert torch.equal(outs[0][0][key], outs[1][0][key]), key
    for x, y in zip(outs[0][1:], outs[1][1:]):
        assert torch.equal(x, y)


def test_enable_and_checkpoint_resume(ops, tmp_path):
    p, q = _pairs()
    a = _sampler(2, chain_offset=1)
    with pytest.raises(RuntimeError, match='not enabled'):
        a.landmark_posterior()
    a.enable_landmark_posterior(p, q, SPACING)
    with pytest.raises(RuntimeError, match='no accumulated'):
        a.landmark_posterior()
    for _ in range(3):
        a.step(2)
        a.accumulate()
    sd = a.state_dict()
    assert sd['lmpost']['n'] == 6 and set(sd['lmpost']) == {'fixed', 'moving', 'spacing', 'n', 'acc'}
    torch.save(sd, tmp_path / 'chains.pt')
    for _ in range(3):
        a.step(2)
        a.accumulate()
    b = _sampler(2, chain_offset=1)
    b.load_state_dict(torch.load(tmp_path / 'chains.pt'))
    assert b.landmark_posterior_enabled
    for _ in range(3):
        b.step(2)
        b.accumulate()
    torch.cuda.synchronize()
    assert torch.equal(a._lmpost['acc'], b._lmpost['acc']) and a._lmpost['n'] == b._lmpost['n'] == 12
    assert torch.equal(a.last_landmark_stats, b.last_landmark_stats)
    assert torch.equal(a.landmark_posterior()['table'].nan_to_num(), b.landmark_posterior()['table'].nan_to_num())
    c = _sampler(2, chain_offset=1)
    c.step(2)
    old = c.state_dict()
    a.load_state_dict(old)   # without the feature in the checkpoint: restarted from zero with the same landmarks
    assert a.landmark_posterior_enabled and a._lmpost['n'] == 0 and float(a._lmpost['acc'].abs().sum()) == 0.0
    a.disable_landmark_posterior()
    a.load_state_dict(old)
    assert not a.landmark_posterior_enabled


# ---- trainer ----------------------------------------------------------------------------------------------------------------
def _config(C, burn_in, samples, period):
    from tests.test_gpu_jacobian_posterior import _config as cfg
    return cfg(C, burn_in=burn_in, samples=samples, period=period)


def _trainer(n, C, burn_in, samples, period, save_dir=None, P=300, max_velocity=3.0):
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_landmarks, make_pair
    from irsgmcmc_b200.trainer import Trainer
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, max_velocity=max_velocity)
    fixed['landmarks'], moving['landmarks'] = make_landmarks(n, max_velocity=max_velocity, no_landmarks=P)
    sd = {f's{l}': l for l in STRUCTURE_LABELS}
    return Trainer(_config(C, burn_in, samples, period), fixed, moving, vp, structures_dict=sd, device=torch.device(DEV),
                   save_dir=save_dir, im_spacing=(1.0, 1.0, 1.0))


def test_run_MCMC_with_TRE(ops, tmp_path):
    from irsgmcmc_b200.logger import load_landmarks_from_disk
    # 500 transitions of 4 chains; a 10-voxel velocity gives an initial TRE of about 0.86 mm on 300 landmarks
    n, C = 64, 4
    plain = _trainer(n, C, 200, 300, 10, max_velocity=10.0)._run_MCMC(speed_test_iters=0)
    t = _trainer(n, C, 200, 300, 10, save_dir=str(tmp_path), max_velocity=10.0)
    res = t._run_MCMC(speed_test_iters=0, with_TRE=True)
    assert set(res) == set(plain) | {'TRE', 'landmark_posterior'}
    for key in ('mean', 'std_dev', 'im_mean', 'im_std'):   # the feature changes no number of the run
        assert torch.equal(res[key], plain[key]), key
    N = sum(1 for it in range(1, 501) if t._is_kept(it))
    L = res['landmark_posterior']
    assert res['TRE'].shape == L['TRE_max'].shape == L['TRE_std'].shape == (N, C) and L['n'] == N * C
    assert (L['TRE_max'] >= res['TRE']).all() and not t.sampler.landmark_posterior_enabled
    assert L['mean_TRE_of_mean'] < L['mean_initial_TRE'], (L['mean_TRE_of_mean'], L['mean_initial_TRE'])
    assert np.isclose(L['mean_expected_TRE'], res['TRE'].mean(), rtol=1e-9)
    assert all(0.0 <= L['coverage'][k] <= 1.0 for k in (50, 90, 95))
    assert L['coverage'][50] <= L['coverage'][90] <= L['coverage'][95]
    assert -1.0 <= L['uncertainty_error_spearman'] <= 1.0
    print(f"TRE: initial {L['mean_initial_TRE']:.3f} mm, of the posterior mean {L['mean_TRE_of_mean']:.3f} mm, expected "
          f"{L['mean_expected_TRE']:.3f} mm over {L['n']} samples; coverage {L['coverage']}; Spearman(sqrt tr Sigma, TRE) "
          f"{L['uncertainty_error_spearman']:.3f}; principal std median {np.median(L['principal_std'], 0).round(3).tolist()} mm")
    pts, arrays = load_landmarks_from_disk(tmp_path / 'MCMC_landmarks.vtk')
    assert np.allclose(pts, L['mean_position'], rtol=1e-6)
    assert np.allclose(arrays['expected_TRE'], L['expected_TRE'], rtol=1e-6)
    assert set(arrays) == {'covariance', 'expected_TRE', 'TRE_of_mean', 'mahalanobis2'}
    bad = _trainer(16, 1, 1, 2, 1, P=10)
    del bad.moving['landmarks']
    with pytest.raises(ValueError):
        bad._run_MCMC(speed_test_iters=0, with_TRE=True)
    bad.moving['landmarks'] = bad.fixed['landmarks'][:5]
    with pytest.raises(ValueError):
        bad._run_MCMC(speed_test_iters=0, with_TRE=True)


def test_test_VI_with_TRE(ops, tmp_path):
    from irsgmcmc_b200.logger import load_landmarks_from_disk
    S, n = 4, 16
    t = _trainer(n, 1, 2, 6, 1, save_dir=str(tmp_path), P=30)
    t.config['trainer'].update(no_iters_VI=2, no_samples_VI_test=S)
    t._run_VI()
    torch.manual_seed(5)
    plain = t._test_VI(speed_test_samples=0, with_ASD=False)
    torch.manual_seed(5)
    res = t._test_VI(speed_test_samples=0, with_ASD=False, with_TRE=True)
    assert set(res) == set(plain) | {'TRE', 'landmark_posterior'}
    assert torch.equal(res['mean'], plain['mean'])
    L = res['landmark_posterior']
    assert res['TRE'].shape == (S, 1) and L['n'] == S and L['mahalanobis2'].shape == (30,)
    pts, _ = load_landmarks_from_disk(tmp_path / 'VI_landmarks.vtk')
    assert np.allclose(pts, L['mean_position'], rtol=1e-6)
    with pytest.raises(ValueError):
        t._test_VI(no_samples=0, speed_test_samples=0, with_TRE=True)
