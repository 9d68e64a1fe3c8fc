"""
Jacobian posterior on the device: the update and finish kernels (csrc/irs_jacobian.cu) against irs_log_det_jacobian, irs_welford_update
and the numpy restatement (tests/helpers/jacobian_posterior_ref.py), the SGLDSampler integration (nothing else of the sampler
changes, checkpoints, two GPUs) and Trainer._run_MCMC / _test_VI(with_jacobian_posterior=True).
"""
import os
import socket

import numpy as np
import pytest
import torch

from tests.helpers import jacobian_posterior_ref as ref

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'eval.npz')


@pytest.fixture(scope='module')
def ops(built):
    from irsgmcmc_b200 import ops
    return ops


def _identity(C, dims):
    D, H, W = dims
    z, y, x = torch.meshgrid(*(torch.linspace(-1, 1, n) for n in (D, H, W)), indexing='ij')
    return torch.stack([x, y, z]).expand(C, 3, D, H, W).contiguous()


def _smooth(C, dims, seed, amp):
    """identity + amp x a smooth random field: no fold for small amp, folds in places for large amp"""
    g = torch.Generator().manual_seed(seed)
    D, H, W = dims
    coarse = torch.randn(C, 3, max(D // 3, 2), max(H // 3, 2), max(W // 3, 2), generator=g)
    u = torch.nn.functional.interpolate(coarse, size=dims, mode='trilinear', align_corners=True)
    return (_identity(C, dims) + amp * u).contiguous()


def _acc(dims):
    return (torch.zeros(*dims, device=DEV, dtype=torch.int32), torch.zeros(*dims, device=DEV), torch.zeros(*dims, device=DEV))


def _mask(dims, seed=0):
    return torch.rand(*dims, generator=torch.Generator().manual_seed(seed)) < 0.8


def _unaligned(t):
    """a copy of t whose storage starts 4 bytes past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 1, device=DEV, dtype=t.dtype)
    out = buf[1:].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 != 0
    return out


# ---- kernels ----------------------------------------------------------------------------------------------------------------
def test_golden_transformation(ops):
    """the reference's folding transformation (3 samples at 24^3, 826 folded voxels): folds = the golden NaN voxels; after the
    first sample the mean is log det J bit for bit where it is finite; both kernels"""
    g = np.load(GOLDEN)
    T = torch.from_numpy(g['T']).to(DEV)
    want_folds = np.isnan(g['log_det_J']).sum(0)
    assert int(want_folds.sum()) == 826
    counts, ld = ops.log_det_jacobian(T)
    mask = torch.ones(24, 24, 24, dtype=torch.bool, device=DEV)
    for layout in (lambda t: t.contiguous(), _unaligned):   # vector kernel, then scalar kernel
        folds, mean, m2 = _acc((24, 24, 24))
        stats = ops.jacobian_update(layout(T[:1]), mask, 0, folds, mean, m2)
        ok = torch.isfinite(ld[0])
        assert torch.equal(mean[ok], ld[0][ok]) and (mean[~ok] == 0).all() and (m2 == 0).all()
        assert torch.equal(folds, (~ok).int())
        assert stats[0, 1].item() == counts[0].item()
        ops.jacobian_update(layout(T[1:]), mask, 1, folds, mean, m2)
        assert np.array_equal(folds.cpu().numpy(), want_folds)


@pytest.mark.parametrize('dims', [(6, 8, 12), (5, 6, 7), (4, 6, 10)])   # W % 4 == 0: vector kernel; otherwise scalar
@pytest.mark.parametrize('C', [1, 3, 7])
def test_no_folds_equals_welford_update(ops, dims, C):
    """without folds, mean / m2 over several launches are torch.equal to irs_welford_update on the stacked log det volumes"""
    folds, mean, m2 = _acc(dims)
    wm, wm2 = torch.zeros(dims, device=DEV), torch.zeros(dims, device=DEV)
    mask = _mask(dims).to(DEV)
    count = 0
    for k in range(3):
        T = _smooth(C, dims, seed=10 * C + k, amp=0.02).to(DEV)
        _, ld = ops.log_det_jacobian(T)
        assert bool(torch.isfinite(ld).all())
        ops.jacobian_update(T, mask, count, folds, mean, m2)
        count = ops.welford_update(ld.contiguous(), count, wm, wm2)
    assert int(folds.abs().sum()) == 0
    assert torch.equal(mean, wm) and torch.equal(m2, wm2)


@pytest.mark.parametrize('dims,C,unaligned', [((8, 8, 8), 3, False), ((7, 9, 11), 7, False), ((8, 8, 8), 5, True),
                                              ((6, 5, 4), 1, False)])
def test_with_folds_against_restatement(ops, dims, C, unaligned):
    """folds exact against the non-finite voxels of irs_log_det_jacobian; moments within fp32 Welford rounding of the fp64
    two-pass statistics of the same log det values; per-sample rows against fp64 sums; an exact det == 0 and a NaN input"""
    folds, mean, m2 = _acc(dims)
    mask = _mask(dims, 3).to(DEV)
    lds, rows = [], []
    for k in range(4):
        T = _smooth(C, dims, seed=100 + k, amp=0.6)
        if k == 1:
            T[0, :, 2, 3, :] = T[0, :, 2, 3, :1]   # x differences zero along one row: det == 0 exactly there
            T[-1, 1, 1, 1, 1] = float('nan')
        T = T.to(DEV)
        _, ld = ops.log_det_jacobian(T)
        if k == 1:
            assert bool((ld[0, 2, 3] == float('-inf')).any())
        lds.append(ld.cpu().numpy())
        TT = _unaligned(T) if unaligned else T
        rows.append(ops.jacobian_update(TT, mask, k * C, folds, mean, m2).cpu().numpy())
    x = np.concatenate(lds)
    want_f, want_m, want_m2 = ref.accumulate(x)
    f = folds.cpu().numpy().reshape(-1)
    assert np.array_equal(f, want_f) and 0 < f.sum() and (f < 4 * C).any()
    ok = want_f < 4 * C
    m, s = mean.cpu().numpy().reshape(-1).astype(np.float64), m2.cpu().numpy().reshape(-1).astype(np.float64)
    scale = np.abs(x[np.isfinite(x)]).max()
    # fp32 Welford over at most 28 samples of values below `scale`: a few hundred ulps at most
    assert np.abs(m[ok] - want_m[ok]).max() <= 1e-5 * scale
    assert np.abs(s[ok] - want_m2[ok]).max() <= 1e-4 * max(float(want_m2[ok].max()), 1.0)
    assert (m[~ok] == 0).all() and (s[~ok] == 0).all()
    for k in range(4):   # counts exact, sums against fp64 over the same fp32 log det values
        want = ref.sample_stats(lds[k], mask.cpu().numpy())
        assert np.array_equal(rows[k][:, :2], want[:, :2])
        assert np.allclose(rows[k][:, 2:], want[:, 2:], rtol=1e-12, atol=1e-9)


def test_batching_is_bit_identical(ops):
    """all chains in one launch = the first 3 then the last 4 in a second launch, both kernels"""
    for dims in ((8, 8, 12), (5, 7, 9)):
        T = _smooth(7, dims, seed=7, amp=0.5).to(DEV)
        mask = _mask(dims).to(DEV)
        a, b = _acc(dims), _acc(dims)
        ra = ops.jacobian_update(T, mask, 0, *a)
        rb = torch.cat([ops.jacobian_update(T[:3].contiguous(), mask, 0, *b),
                        ops.jacobian_update(T[3:].contiguous(), mask, 3, *b)])
        for x, y in zip(a, b):
            assert torch.equal(x, y)
        assert torch.equal(ra, rb)
        assert int(a[0].sum()) > 0


def test_finish_against_restatement(ops):
    """accumulators with every count of folds 0..n (n_v = 0 and 1 included): p_fold and the integer summaries exact, the
    mean map the accumulator itself, std the fp32 expression of welford_std, the fp64 means to 1e-12"""
    dims, n = (9, 10, 12), 15
    g = np.random.default_rng(4)
    f = g.integers(0, n + 1, size=dims).astype(np.int32)
    m = np.where(f < n, g.normal(0.0, 0.3, size=dims), 0.0).astype(np.float32)
    s = np.where(f < n - 1, g.random(dims), 0.0).astype(np.float32)
    folds, mean, m2 = (torch.from_numpy(a).to(DEV) for a in (f, m, s))
    mask = _mask(dims, 4).to(DEV)
    f, m, s = f.reshape(-1), m.reshape(-1), s.reshape(-1)
    for args in ((folds, mean, m2, mask), tuple(_unaligned(t) for t in (folds, mean, m2)) + (mask,)):
        p, mo, so, summ = ops.jacobian_posterior(args[0], args[1], args[2], n, args[3])
        wp, wmo, wso, wsumm = ref.posterior(f, m, s, n, mask.cpu().numpy())
        assert np.array_equal(p.cpu().numpy().reshape(-1), wp)
        nv = n - f
        got_m, got_s = mo.cpu().numpy().reshape(-1), so.cpu().numpy().reshape(-1)
        assert np.array_equal(got_m[nv >= 1], m[nv >= 1]) and np.isnan(got_m[nv < 1]).all()
        want_s = np.sqrt(s[nv >= 2] / (nv[nv >= 2] - 1).astype(np.float32))
        assert np.array_equal(got_s[nv >= 2], want_s) and np.isnan(got_s[nv < 2]).all()
        for key in ('sum_folds', 'voxels_ever_folded', 'voxels_folded_in_majority', 'voxels_finite', 'voxels_finite_2',
                    'mask_voxels'):
            assert summ[key] == wsumm[key], key
        in_std = mask.cpu().numpy().reshape(-1)[nv >= 2]
        for key, want in (('mean_log_det_J', wsumm['mean_log_det_J']), ('mean_std_log_det_J', want_s[in_std].mean(dtype=np.float64))):
            assert abs(summ[key] - want) <= 1e-12 * max(abs(want), 1.0), key


def test_256_cubed_16_chains_make_pair(ops):
    """one kept sample of a 256^3 make_pair sampler with 16 chains against irs_log_det_jacobian + irs_welford_update"""
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    n, C = 256, 16
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=DEV)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=DEV)
    s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
    s.init_gmm(sigma_hat=0.7)
    s.enable_jacobian_posterior()
    s.step(2, use_graph=False)
    T = s.transformation()
    s.accumulate(transformation=T)
    counts, ld = ops.log_det_jacobian(T)
    j = s._jacpost
    ok = torch.isfinite(ld)
    assert torch.equal(j['folds'], (~ok).sum(0, dtype=torch.int32))
    if bool(ok.all()):
        wm, wm2 = torch.zeros(n, n, n, device=DEV), torch.zeros(n, n, n, device=DEV)
        ops.welford_update(ld, 0, wm, wm2)
        assert torch.equal(j['mean'], wm) and torch.equal(j['m2'], wm2)
    stats = s.last_jacobian_stats.cpu().numpy()
    mask = s.mask.view(n, n, n).bool()
    assert np.array_equal(stats[:, 1], (~ok & mask).sum((1, 2, 3)).cpu().numpy())
    assert np.array_equal(stats[:, 0], (ok & mask).sum((1, 2, 3)).cpu().numpy())
    ld64 = torch.where(ok & mask, ld, torch.zeros_like(ld)).double()
    assert np.allclose(stats[:, 2], ld64.sum((1, 2, 3)).cpu().numpy(), rtol=1e-10, atol=1e-6)
    post = s.jacobian_posterior()
    assert post['n'] == C and post['summary']['sum_folds'] == int((~ok & mask).sum())


# ---- sampler ----------------------------------------------------------------------------------------------------------------
LABELS = [10, 11, 12, 13, 16, 17, 18, 26, 49, 50, 51, 52, 53, 54, 58]


def _sampler(C, n=16, chain_offset=0, seed=0, device=DEV):
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    fixed, moving, vp = make_pair(n)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(hyper_mode='per_chain'), device=device, chain_offset=chain_offset)
    gen = torch.Generator().manual_seed(seed)
    v0 = 2.0 * torch.randn(4, 3, n, n, n, generator=gen)[chain_offset:chain_offset + C]
    s.set_state(v0, torch.full((1, 3, n, n, n), 0.5))
    s.init_gmm(sigma_hat=0.7)
    return s, fixed


def test_accumulate_matches_the_kernels(ops):
    """accumulate() = ops.jacobian_update on transformation(); passing transformation = computing it inside"""
    a, _ = _sampler(3)
    b, _ = _sampler(3)
    a.enable_jacobian_posterior()
    b.enable_jacobian_posterior()
    manual = _acc((16, 16, 16))
    mask = a.mask.view(16, 16, 16)
    for k in range(4):
        a.step(2)
        b.step(2)
        T = a.transformation()
        row = ops.jacobian_update(T, mask, 3 * k, *manual)
        a.accumulate()
        b.accumulate(transformation=b.transformation())
        assert torch.equal(a.last_jacobian_stats, row) and torch.equal(b.last_jacobian_stats, row)
    for name, t in zip(('folds', 'mean', 'm2'), manual):
        assert torch.equal(a._jacpost[name], t) and torch.equal(b._jacpost[name], t), name
    post = a.jacobian_posterior()
    assert post['n'] == 12 and set(post) == {'n', 'fold_probability', 'log_det_J_mean', 'log_det_J_std', 'summary'}
    assert torch.equal(a._jacpost['folds'], manual[0])   # a query keeps the accumulators: sampling can continue
    with pytest.raises(ValueError, match='transformation'):
        a.accumulate(transformation=T[:2].contiguous())


def test_sampler_state_unchanged_by_the_feature(ops):
    """pooled moments, split-R-hat accumulators, label counts and chain states are bit-identical with the feature on and off"""
    outs = []
    for on in (False, True):
        s, _ = _sampler(4)
        s.enable_convergence_diagnostics(6)
        s.enable_segmentation_posterior(LABELS)
        if on:
            s.enable_jacobian_posterior()
        for _ in range(6):
            s.step(2)
            T = s.transformation()
            s.accumulate(seg_warped=s.warp_segmentation(transformation=T), transformation=T)
        torch.cuda.synchronize()
        outs.append((s.posterior_moments(), s.v.clone(), s.hyper.clone(), s._rhat['mean'].clone(), s._rhat['m2'].clone(),
                     s._segpost['counts'].clone()))
        if on:
            assert s._jacpost['n'] == 24
        else:
            assert not s.jacobian_posterior_enabled and 'jacpost' not in s.state_dict()
    for key in ('displacement_mean', 'displacement_std', 'im_mean', 'im_std'):
        assert torch.equal(outs[0][0][key], outs[1][0][key]), key
    for x, y in zip(outs[0][1:], outs[1][1:]):
        assert torch.equal(x, y)


def test_enable_and_checkpoint_resume(ops, tmp_path):
    a, _ = _sampler(2, chain_offset=1)
    with pytest.raises(RuntimeError, match='not enabled'):
        a.jacobian_posterior()
    a.enable_jacobian_posterior()
    with pytest.raises(RuntimeError, match='no accumulated'):
        a.jacobian_posterior()
    for _ in range(3):
        a.step(2)
        a.accumulate()
    sd = a.state_dict()
    assert sd['jacpost']['n'] == 6 and set(sd['jacpost']) == {'n', 'folds', 'mean', 'm2'}
    torch.save(sd, tmp_path / 'chains.pt')
    for _ in range(3):
        a.step(2)
        a.accumulate()
    b, _ = _sampler(2, chain_offset=1)
    assert not b.jacobian_posterior_enabled
    b.load_state_dict(torch.load(tmp_path / 'chains.pt'))
    assert b.jacobian_posterior_enabled
    for _ in range(3):
        b.step(2)
        b.accumulate()
    torch.cuda.synchronize()
    for name in ('folds', 'mean', 'm2'):
        assert torch.equal(a._jacpost[name], b._jacpost[name]), name
    assert a._jacpost['n'] == b._jacpost['n'] == 12 and torch.equal(a.last_jacobian_stats, b.last_jacobian_stats)
    pa, pb = a.jacobian_posterior(), b.jacobian_posterior()
    for key in ('fold_probability', 'log_det_J_mean', 'log_det_J_std'):
        assert torch.equal(pa[key], pb[key]), key
    assert str(pa['summary']) == str(pb['summary'])   # NaN means compare equal as text
    assert torch.equal(a.v, b.v) and torch.equal(a.disp_mean, b.disp_mean)
    # a checkpoint without the feature restarts enabled accumulators from zero and leaves a disabled sampler disabled
    c, _ = _sampler(2, chain_offset=1)
    c.step(2)
    old = c.state_dict()
    assert 'jacpost' not in old
    a.load_state_dict(old)
    assert a.jacobian_posterior_enabled and a._jacpost['n'] == 0 and int(a._jacpost['folds'].abs().sum()) == 0
    a.disable_jacobian_posterior()
    a.load_state_dict(old)
    assert not a.jacobian_posterior_enabled


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world)
    s, _ = _sampler(2, chain_offset=2 * rank, device=f'cuda:{rank}')
    s.enable_jacobian_posterior()
    for _ in range(4):
        s.step(2)
        s.accumulate()
    post = s.jacobian_posterior()
    torch.save({k: (v.cpu() if torch.is_tensor(v) else v) for k, v in post.items()}, os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


def test_two_gpus_merge_equals_one_rank(ops, tmp_path):
    """4 chains over two GPUs: the merged posterior equals one GPU holding all 4 chains (folds exact, moments to fp32 merge
    rounding)"""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / 'r0.pt'), torch.load(tmp_path / 'r1.pt')
    s, _ = _sampler(4)
    s.enable_jacobian_posterior()
    for _ in range(4):
        s.step(2)
        s.accumulate()
    one = s.jacobian_posterior()
    assert r0['n'] == r1['n'] == one['n'] == 16
    assert torch.equal(r0['fold_probability'], one['fold_probability'].cpu())
    assert torch.equal(r0['log_det_J_mean'], r1['log_det_J_mean'])
    ok = torch.isfinite(one['log_det_J_mean'].cpu())
    assert torch.allclose(r0['log_det_J_mean'][ok], one['log_det_J_mean'].cpu()[ok], rtol=1e-5, atol=1e-5)
    for key in ('sum_folds', 'voxels_ever_folded', 'voxels_folded_in_majority'):
        assert r0['summary'][key] == one['summary'][key], key


# ---- trainer ----------------------------------------------------------------------------------------------------------------
def _config(C, burn_in=2, samples=6, period=1):
    return {'data_loss': {'type': 'GMM', 'args': {'no_components': 4, 's': 2}},
            'data_loss_scale_prior': {'type': 'LogScaleNormalPrior', 'args': {'loc': 0.0, 'scale': 2.3}},
            'data_loss_proportion_prior': {'type': 'DirichletPrior', 'args': {'no_classes': 4, 'alpha': 0.5}},
            'reg_loss': {'type': 'RegLoss_LogNormal', 'args': {'diff_op': 'GradientOperator', 'w_reg': 1.6, 'learnable': True}},
            'reg_loss_scale_prior': {'type': 'LogScaleNormalPrior', 'args': {'loc': 2.8, 'scale': 5.0}},
            'optimizer_SG_MCMC': {'type': 'SGD', 'args': {'lr': 0.4}},
            'optimizer_GMM': {'type': 'Adam', 'args': {'lr_log_std': 0.2, 'lr_logits': 0.2, 'lr_decay': 0.001}},
            'optimizer_reg': {'type': 'Adam', 'args': {'lr_loc': 0.01, 'lr_log_scale': 0.01, 'lr_decay': 0.001}},
            'Sobolev_grad': {'enabled': True, 's': 3, 'lambda': 0.5}, 'virtual_decimation': True,
            'trainer': {'MCMC_init': 'VI', 'no_chains': C, 'no_iters_burn_in': burn_in, 'no_samples_MCMC': samples,
                        'log_period_MCMC': period, 'uniform_noise': {'enabled': True, 'magnitude': 0.1}}}


def _trainer(n, C, save_dir=None):
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.trainer import Trainer
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n)
    sd = {f's{l}': l for l in STRUCTURE_LABELS}
    return Trainer(_config(C), fixed, moving, vp, structures_dict=sd, device=torch.device(DEV), save_dir=save_dir)


def _direct_sdlogj(paths, mask):
    """SDlogJ and the folded fraction of the log det J volumes the trainer wrote with save_sample"""
    from irsgmcmc_b200.logger import load_im_from_disk
    sd, ff = [], []
    for p in paths:
        ld, _ = load_im_from_disk(p)
        ld = ld.astype(np.float64)[mask]
        ok = np.isfinite(ld)
        sd.append(np.std(ld[ok]))
        ff.append((~ok).sum() / ld.size)
    return np.array(sd), np.array(ff)


JAC_KEYS = {'n', 'fold_probability', 'log_det_J_mean', 'log_det_J_std', 'summary', 'SDlogJ', 'folded_fraction',
            'expected_folded_voxels', 'voxels_ever_folded', 'voxels_folded_in_majority', 'mean_log_det_J', 'mean_std_log_det_J'}


def test_run_MCMC_with_jacobian_posterior(ops, tmp_path):
    from irsgmcmc_b200.logger import load_im_from_disk
    n, C = 32, 3
    plain = _trainer(n, C)._run_MCMC(speed_test_iters=0)
    assert set(plain) == {'mean', 'std_dev', 'im_mean', 'im_std', 'n', 'DSC', 'no_non_diffeomorphic_voxels', 'ASD'}
    t = _trainer(n, C, save_dir=str(tmp_path))
    res = t._run_MCMC(speed_test_iters=0, with_jacobian_posterior=True)
    assert set(res) == set(plain) | {'jacobian_posterior'}
    for key in ('mean', 'std_dev', 'im_mean', 'im_std'):   # the feature changes no number of the run
        assert torch.equal(res[key], plain[key]), key
    assert [x.tolist() for x in res['no_non_diffeomorphic_voxels']] == [x.tolist() for x in plain['no_non_diffeomorphic_voxels']]
    P = res['jacobian_posterior']
    assert set(P) == JAC_KEYS and P['n'] == 6 * C and not t.sampler.jacobian_posterior_enabled
    assert P['SDlogJ'].shape == P['folded_fraction'].shape == (6, C)
    assert P['expected_folded_voxels'] == P['summary']['sum_folds'] / P['n']
    mask = t.fixed['mask'].cpu().numpy().reshape(n, n, n).astype(bool)
    kept = [it for it in range(1, 9) if t._is_kept(it)]
    for c in range(C):
        sd, ff = _direct_sdlogj([tmp_path / f'chain_{c}_sample_{it:07}_log_det_J.nii.gz' for it in kept], mask)
        assert np.allclose(P['SDlogJ'][:, c], sd, rtol=1e-9, atol=1e-12) and np.allclose(P['folded_fraction'][:, c], ff)
    folded = sum(int(x.sum()) for x in res['no_non_diffeomorphic_voxels'])
    print('SDlogJ', np.round(P['SDlogJ'], 4).tolist(), 'expected folded voxels', P['expected_folded_voxels'],
          'folded in all samples (whole volume)', folded)
    for key, name in (('log_det_J_mean', 'log_det_J_mean'), ('log_det_J_std', 'log_det_J_std_dev'),
                      ('fold_probability', 'fold_probability')):
        im, _ = load_im_from_disk(tmp_path / f'MCMC_{name}.nii.gz')
        assert np.array_equal(im, P[key].cpu().numpy(), equal_nan=True), key


def test_test_VI_with_jacobian_posterior(ops, tmp_path):
    S, n = 4, 16
    t = _trainer(n, 1, save_dir=str(tmp_path))
    t.config['trainer'].update(no_iters_VI=2, no_samples_VI_test=S)
    t._run_VI()
    torch.manual_seed(5)
    plain = t._test_VI(speed_test_samples=0, with_ASD=False)
    torch.manual_seed(5)
    res = t._test_VI(speed_test_samples=0, with_ASD=False, with_jacobian_posterior=True)
    assert set(res) == set(plain) | {'jacobian_posterior'}
    assert torch.equal(res['mean'], plain['mean']) and res['no_non_diffeomorphic_voxels'] == plain['no_non_diffeomorphic_voxels']
    P = res['jacobian_posterior']
    assert set(P) == JAC_KEYS and P['n'] == S and P['SDlogJ'].shape == (S, 1)
    mask = t.fixed['mask'].cpu().numpy().reshape(n, n, n).astype(bool)
    sd, ff = _direct_sdlogj([tmp_path / f'sample_{i:07}_log_det_J.nii.gz' for i in range(1, S + 1)], mask)
    assert np.allclose(P['SDlogJ'][:, 0], sd, rtol=1e-9, atol=1e-12) and np.allclose(P['folded_fraction'][:, 0], ff)
    for name in ('log_det_J_mean', 'log_det_J_std_dev', 'fold_probability'):
        assert (tmp_path / f'VI_{name}.nii.gz').exists()
    with pytest.raises(ValueError):
        t._test_VI(no_samples=0, speed_test_samples=0, with_jacobian_posterior=True)
