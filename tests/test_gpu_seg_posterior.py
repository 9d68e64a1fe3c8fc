"""
Segmentation posterior on the device: the label-count and finish kernels (csrc/irs_segpost.cu) against the numpy restatement
(tests/helpers/seg_posterior_ref.py), their identities with irs_dice_counts, the SGLDSampler integration (nothing else of the
sampler changes, checkpoints) and Trainer._run_MCMC / _test_VI(with_seg_posterior=True).
"""
import numpy as np
import pytest
import torch

from tests.helpers import seg_posterior_ref as ref

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
OTHER = [0, -1, -300, 255, 256, 1000, 32767]   # never in the label lists below: the class "other"


@pytest.fixture(scope='module')
def ops(built):
    from irsgmcmc_b200 import ops
    return ops


def _segs(shape, labels, seed, p_other=0.4):
    """int16 volumes whose voxels carry one of `labels` or an "other" value"""
    g = np.random.default_rng(seed)
    values = np.asarray(labels + OTHER, dtype=np.int16)
    pick = np.where(g.random(shape) < p_other, g.integers(len(labels), len(values), shape), g.integers(0, len(labels), shape))
    return values[pick]


def _device(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _check_posterior(ops, counts, n, labels, fixed):
    """the device finish against the restatement: probabilities bit-equal, majority and summaries exact, entropy 1e-6"""
    dims = counts.shape[1:]
    prob, majority, entropy, summary = ops.label_posterior(_device(counts), n, labels, None if fixed is None else _device(fixed))
    w_prob, w_maj, w_ent, w_sum = ref.label_posterior(counts.reshape(len(labels), -1), n, labels, fixed)
    assert prob.shape == (len(labels), *dims) and majority.shape == (1, 1, *dims) and entropy.shape == (1, *dims)
    assert np.array_equal(prob.cpu().numpy().reshape(len(labels), -1), w_prob)
    assert np.array_equal(majority.cpu().numpy().reshape(-1), w_maj)
    err = float(np.abs(entropy.cpu().numpy().reshape(-1).astype(np.float64) - w_ent).max())
    assert err <= 1e-6, err
    assert np.array_equal(summary.cpu().numpy(), w_sum)
    return prob, majority, entropy, summary


# ---- kernels ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dims', [(5, 6, 7), (4, 6, 8)])   # V % 4 != 0: scalar kernels; V % 4 == 0: vector kernels
@pytest.mark.parametrize('C', [1, 3, 7])
def test_update_exact(ops, dims, C):
    labels = [10, 11, 12, 13, 16, -7, 300]
    counts = torch.zeros(len(labels), *dims, device=DEV, dtype=torch.int32)
    all_segs = []
    for k in range(3):   # several successive updates
        segs = _segs((C, 1, *dims), labels, seed=100 * C + k)
        all_segs.append(segs)
        ops.label_counts_update(_device(segs), labels, counts)
    want = ref.label_counts(np.concatenate(all_segs), labels)
    assert np.array_equal(counts.cpu().numpy().reshape(len(labels), -1), want)
    fixed = _segs((1, 1, *dims), labels, seed=7)
    _check_posterior(ops, counts.cpu().numpy(), 3 * C, labels, fixed)
    _check_posterior(ops, counts.cpu().numpy(), 3 * C, labels, None)


def test_update_unaligned_and_32_labels(ops):
    """exactly 32 labels; a segmentation buffer that is not 8-byte aligned takes the scalar kernel with the same counts"""
    dims, C = (8, 8, 8), 5
    labels = [3 * i + 1 for i in range(32)]
    segs = _segs((C, 1, *dims), labels, seed=3, p_other=0.2)
    V = int(np.prod(dims))
    buf = torch.empty(C * V + 1, device=DEV, dtype=torch.int16)
    shifted = buf[1:].view(C, 1, *dims)
    shifted.copy_(_device(segs))
    assert shifted.data_ptr() % 8 != 0
    a = torch.zeros(32, *dims, device=DEV, dtype=torch.int32)
    b = torch.zeros_like(a)
    ops.label_counts_update(shifted, labels, a)
    ops.label_counts_update(_device(segs), labels, b)
    assert torch.equal(a, b)
    assert np.array_equal(a.cpu().numpy().reshape(32, -1), ref.label_counts(segs, labels))
    _check_posterior(ops, a.cpu().numpy(), C, labels, segs[:1])
    with pytest.raises(RuntimeError, match='bad argument'):
        ops.label_counts_update(_device(segs), labels + [200], torch.zeros(33, *dims, device=DEV, dtype=torch.int32))
    with pytest.raises(RuntimeError, match='unsupported'):
        ops.label_counts_update(_device(segs), [0, 1], torch.zeros(2, *dims, device=DEV, dtype=torch.int32))
    with pytest.raises(NotImplementedError):
        ops.label_counts_update(_device(segs).int(), labels, a)


def test_batching_and_order_do_not_matter(ops):
    dims, C, labels = (6, 8, 8), 6, [10, 11, 12]
    segs = _device(_segs((C, 1, *dims), labels, seed=11))
    whole = torch.zeros(3, *dims, device=DEV, dtype=torch.int32)
    ops.label_counts_update(segs, labels, whole)
    split = torch.zeros_like(whole)
    ops.label_counts_update(segs[:2].contiguous(), labels, split)
    ops.label_counts_update(segs[2:].contiguous(), labels, split)
    perm = torch.zeros_like(whole)
    for c in torch.randperm(C).tolist():
        ops.label_counts_update(segs[c:c + 1].contiguous(), labels, perm)
    assert torch.equal(whole, split) and torch.equal(whole, perm)


def test_finish_ties(ops):
    """counts built so that classes tie: "other" keeps every tie, then the earlier label"""
    labels = [5, 9, 2]
    n = 6
    cases = [(2, 2, 0), (3, 3, 0), (1, 1, 1), (0, 3, 3), (2, 0, 2), (0, 0, 0), (6, 0, 0), (0, 2, 2), (1, 2, 2), (3, 0, 3)]
    # other = 6 - sum: (2,2,0) other 2 -> 0; (3,3,0) other 0 -> 5; (1,1,1) other 3 -> 0; (0,3,3) -> 9; (2,0,2) other 2 -> 0;
    # (0,0,0) -> 0; (6,0,0) -> 5; (0,2,2) other 2 -> 0; (1,2,2) other 1 -> 9; (3,0,3) -> 5
    want = [0, 5, 0, 9, 0, 0, 5, 0, 9, 5]
    for dims in ((1, 2, 5), (1, 1, 10), (2, 2, 4)):   # scalar and vector finish
        V = int(np.prod(dims))
        counts = np.zeros((3, V), np.int32)
        for v in range(V):
            counts[:, v] = cases[v % len(cases)]
        _, majority, _, _ = _check_posterior(ops, counts.reshape(3, *dims), n, labels, None)
        assert majority.cpu().numpy().reshape(-1).tolist() == [want[v % len(cases)] for v in range(V)]


def test_identities_with_dice_counts(ops):
    """S_l = sum over samples of |B_l| and O_l = sum of |A_l and B_l| (irs_dice_counts); identical samples: entropy 0, U = 0,
    majority = the sample restricted to the list"""
    dims, C, labels = (12, 12, 12), 5, [10, 11, 12, 13, 16]
    fixed = _device(_segs((1, 1, *dims), labels, seed=21))
    segs = _device(_segs((C, 1, *dims), labels, seed=22))
    counts = torch.zeros(len(labels), *dims, device=DEV, dtype=torch.int32)
    ops.label_counts_update(segs, labels, counts)
    _, _, _, summary = ops.label_posterior(counts, C, labels, fixed)
    dc = ops.dice_counts(fixed, segs, labels).long()   # (C, L, 3): |A|, |B|, |A and B|
    assert torch.equal(summary[:, 0], dc[:, :, 1].sum(0)) and torch.equal(summary[:, 1], dc[:, :, 2].sum(0))

    one = segs[:1].expand(C, -1, -1, -1, -1).contiguous()
    same = torch.zeros_like(counts)
    ops.label_counts_update(one, labels, same)
    _, majority, entropy, summary = ops.label_posterior(same, C, labels, fixed)
    s = one[0]
    restricted = torch.where(torch.isin(s, torch.tensor(labels, device=DEV, dtype=torch.int16)), s, torch.zeros_like(s))
    assert torch.equal(majority[0], restricted) and (entropy == 0).all() and (summary[:, 2] == 0).all()


def test_256_cubed_16_chains_make_pair(ops):
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    n, C, labels = 256, 16, list(STRUCTURE_LABELS)
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=DEV)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=DEV)
    s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
    s.init_gmm(sigma_hat=0.7)
    s.step(2, use_graph=False)
    seg_w = s.warp_segmentation()
    counts = torch.zeros(len(labels), n, n, n, device=DEV, dtype=torch.int32)
    ops.label_counts_update(seg_w, labels, counts)
    got = counts.cpu().numpy().reshape(len(labels), -1)
    assert np.array_equal(got, ref.label_counts(seg_w.cpu().numpy(), labels))
    del s, seg_w
    torch.cuda.empty_cache()
    _check_posterior(ops, got.reshape(len(labels), n, n, n), C, labels, fixed['seg'].numpy())


# ---- sampler ----------------------------------------------------------------------------------------------------------------
LABELS = [10, 11, 12, 13, 16, 17, 18, 26, 49, 50, 51, 52, 53, 54, 58]


def _sampler(C, n=16, chain_offset=0, seed=0, moving_seg=True):
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    fixed, moving, vp = make_pair(n)
    if not moving_seg:
        moving = {k: v for k, v in moving.items() if k != 'seg'}
    s = SGLDSampler(fixed, moving, C, SGLDConfig(hyper_mode='per_chain'), device=DEV, chain_offset=chain_offset)
    gen = torch.Generator().manual_seed(seed)
    v0 = 2.0 * torch.randn(4, 3, n, n, n, generator=gen)[chain_offset:chain_offset + C]
    s.set_state(v0, torch.full((1, 3, n, n, n), 0.5))
    s.init_gmm(sigma_hat=0.7)
    return s, fixed


def test_accumulate_matches_warp_segmentation(ops):
    """counts of accumulate() = counts of the warp_segmentation() outputs; passing seg_warped = warping inside"""
    a, fixed = _sampler(3)
    b, _ = _sampler(3)
    a.enable_segmentation_posterior(LABELS)
    b.enable_segmentation_posterior(LABELS)
    manual = torch.zeros(len(LABELS), 16, 16, 16, device=DEV, dtype=torch.int32)
    for _ in range(4):
        a.step(2)
        b.step(2)
        seg_a = a.warp_segmentation()
        ops.label_counts_update(seg_a, LABELS, manual)
        a.accumulate()
        b.accumulate(seg_warped=b.warp_segmentation())
    assert torch.equal(a._segpost['counts'], manual) and torch.equal(b._segpost['counts'], manual)
    assert int(manual.sum()) > 0
    post = a.segmentation_posterior(seg_fixed=fixed['seg'])
    assert post['n'] == 12 and post['labels'] == LABELS
    w_prob, w_maj, _, w_sum = ref.label_posterior(manual.cpu().numpy().reshape(len(LABELS), -1), 12, LABELS, fixed['seg'].numpy())
    assert np.array_equal(post['majority'].cpu().numpy().reshape(-1), w_maj)
    assert np.array_equal(post['summary'].cpu().numpy(), w_sum)
    assert torch.equal(a._segpost['counts'], manual)   # a query leaves the counts as they are: sampling can continue
    with pytest.raises(ValueError, match='seg_warped'):
        a.accumulate(seg_warped=seg_a[:2].contiguous())


def test_sampler_state_unchanged_by_the_feature(ops):
    """pooled moments, split-R-hat accumulators and chain states are bit-identical with the feature on and off; accumulate()
    after the segmentation warp (the Trainer's order) gives the same moments as before it"""
    outs = []
    for mode in ('off', 'on', 'off_after_warp'):
        s, _ = _sampler(4)
        s.enable_convergence_diagnostics(6)
        if mode == 'on':
            s.enable_segmentation_posterior(LABELS)
        segs = []
        for _ in range(6):
            s.step(2)
            if mode == 'off_after_warp':
                segs.append(s.warp_segmentation(transformation=s.transformation()))
                s.accumulate(seg_warped=segs[-1])
            else:
                s.accumulate()
                segs.append(s.warp_segmentation(transformation=s.transformation()))
        torch.cuda.synchronize()
        outs.append((s.posterior_moments(), s.v.clone(), s.hyper.clone(), s._rhat['mean'].clone(), s._rhat['m2'].clone(),
                     torch.stack(segs)))
    base = outs[0]
    for other in outs[1:]:
        for key in ('displacement_mean', 'displacement_std', 'im_mean', 'im_std'):
            assert torch.equal(base[0][key], other[0][key]), key
        for x, y in zip(base[1:], other[1:]):
            assert torch.equal(x, y)


def test_enable_and_checkpoint_resume(ops, tmp_path):
    s, _ = _sampler(2, moving_seg=False)
    with pytest.raises(ValueError, match='moving segmentation'):
        s.enable_segmentation_posterior(LABELS)
    a, fixed = _sampler(2, chain_offset=1)
    with pytest.raises(RuntimeError, match='not enabled'):
        a.segmentation_posterior()
    with pytest.raises(ValueError):
        a.enable_segmentation_posterior([10, 10])
    a.enable_segmentation_posterior(LABELS)
    with pytest.raises(RuntimeError, match='no accumulated'):
        a.segmentation_posterior()
    for _ in range(3):
        a.step(2)
        a.accumulate()
    sd = a.state_dict()
    assert sd['segpost']['n'] == 6 and sd['segpost']['labels'] == LABELS
    torch.save(sd, tmp_path / 'chains.pt')
    for _ in range(3):
        a.step(2)
        a.accumulate()
    b, _ = _sampler(2, chain_offset=1)
    assert not b.segmentation_posterior_enabled
    b.load_state_dict(torch.load(tmp_path / 'chains.pt'))
    assert b.segmentation_posterior_enabled
    for _ in range(3):
        b.step(2)
        b.accumulate()
    torch.cuda.synchronize()
    assert torch.equal(a._segpost['counts'], b._segpost['counts']) and a._segpost['n'] == b._segpost['n'] == 12
    pa, pb = a.segmentation_posterior(fixed['seg']), b.segmentation_posterior(fixed['seg'])
    for key in ('probability', 'majority', 'entropy', 'summary'):
        assert torch.equal(pa[key], pb[key]), key
    assert torch.equal(a.v, b.v) and torch.equal(a.disp_mean, b.disp_mean)
    # a checkpoint without the feature restarts enabled counts from zero and leaves a disabled sampler disabled
    c, _ = _sampler(2, chain_offset=1)
    c.step(2)
    old = c.state_dict()
    assert 'segpost' not in old
    a.load_state_dict(old)
    assert a.segmentation_posterior_enabled and a._segpost['n'] == 0 and int(a._segpost['counts'].abs().sum()) == 0
    a.disable_segmentation_posterior()
    a.load_state_dict(old)
    assert not a.segmentation_posterior_enabled


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


def _trainer(n, C, structures=True, save_dir=None):
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.trainer import Trainer
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n)
    sd = {f's{l}': l for l in STRUCTURE_LABELS} if structures else None
    return Trainer(_config(C), fixed, moving, vp, structures_dict=sd, device=torch.device(DEV), save_dir=save_dir)


def test_run_MCMC_with_seg_posterior(ops, tmp_path):
    from irsgmcmc_b200.logger import load_im_from_disk
    from irsgmcmc_b200.utils.util import calc_ASD_GPU, calc_DSC_GPU
    n, C = 32, 3
    plain = _trainer(n, C)._run_MCMC(speed_test_iters=0)
    assert set(plain) == {'mean', 'std_dev', 'im_mean', 'im_std', 'n', 'DSC', 'no_non_diffeomorphic_voxels', 'ASD'}
    t = _trainer(n, C, save_dir=str(tmp_path))
    res = t._run_MCMC(speed_test_iters=0, with_ASD=True, with_seg_posterior=True)
    assert set(res) == set(plain) | {'seg_posterior'}
    for key in ('mean', 'std_dev', 'im_mean', 'im_std'):   # the feature changes no number of the run
        assert torch.equal(res[key], plain[key]), key
    assert res['n'] == plain['n'] == 6 * C
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(res['DSC'], plain['DSC']))
    assert [x.tolist() for x in res['no_non_diffeomorphic_voxels']] == [x.tolist() for x in plain['no_non_diffeomorphic_voxels']]
    P = res['seg_posterior']
    assert set(P) == {'labels', 'n', 'probability', 'majority', 'entropy', 'summary', 'structures'} and P['n'] == 6 * C
    assert P['probability'].shape == (15, n, n, n) and P['majority'].dtype == torch.int16
    assert not t.sampler.segmentation_posterior_enabled
    seg_f = t.fixed['seg'].to(DEV)
    dsc = calc_DSC_GPU(1, seg_f, P['majority'], t.structures_dict)[0]
    asd = calc_ASD_GPU(1, seg_f, P['majority'], t.structures_dict, t.im_spacing)[0]
    summary = P['summary'].cpu().numpy()
    got, want = [], []
    for j, (name, lab) in enumerate(t.structures_dict.items()):
        e = P['structures'][name]
        assert set(e) == {'expected_volume', 'uncertain_voxels', 'soft_DSC', 'DSC_majority', 'ASD_majority'}
        F = int((t.fixed['seg'] == lab).sum())
        got.append([e['DSC_majority'], e['ASD_majority'], e['expected_volume'], e['uncertain_voxels'], e['soft_DSC']])
        want.append([dsc[j], asd[j], summary[j, 0] / P['n'], summary[j, 2], 2.0 * summary[j, 1] / (summary[j, 0] + P['n'] * F)])
    assert np.array_equal(np.array(got, dtype=np.float64), np.array(want, dtype=np.float64), equal_nan=True)
    mean_dsc = np.nanmean(np.stack(res['DSC']), axis=(0, 1))
    print('soft DSC', [round(P['structures'][k]['soft_DSC'], 3) for k in t.structures_dict],
          'mean per-sample DSC', np.round(mean_dsc, 3).tolist())
    maj, _ = load_im_from_disk(tmp_path / 'MCMC_seg_majority.nii.gz')
    ent, _ = load_im_from_disk(tmp_path / 'MCMC_seg_entropy.nii.gz')
    assert maj.dtype == np.int16 and np.array_equal(maj, P['majority'][0, 0].cpu().numpy())
    assert ent.dtype == np.float32 and np.array_equal(ent, P['entropy'][0].cpu().numpy())
    with pytest.raises(ValueError, match='structures_dict'):
        _trainer(n, C, structures=False)._run_MCMC(speed_test_iters=0, with_seg_posterior=True)


def test_test_VI_with_seg_posterior(ops, tmp_path):
    S = 4
    t = _trainer(16, 1, save_dir=str(tmp_path))
    t.config['trainer'].update(no_iters_VI=2, no_samples_VI_test=S)
    t._run_VI()
    torch.manual_seed(5)
    plain = t._test_VI(speed_test_samples=0, with_ASD=False)
    torch.manual_seed(5)
    res = t._test_VI(speed_test_samples=0, with_ASD=False, with_seg_posterior=True)
    assert set(res) == set(plain) | {'seg_posterior'}
    assert torch.equal(res['mean'], plain['mean']) and np.array_equal(res['DSC'], plain['DSC'], equal_nan=True)
    P = res['seg_posterior']
    assert P['n'] == S and P['majority'].shape == (1, 1, 16, 16, 16)
    assert 'ASD_majority' not in next(iter(P['structures'].values()))
    assert (tmp_path / 'VI_seg_majority.nii.gz').exists() and (tmp_path / 'VI_seg_entropy.nii.gz').exists()
    with pytest.raises(ValueError):
        t._test_VI(no_samples=0, speed_test_samples=0, with_seg_posterior=True)
