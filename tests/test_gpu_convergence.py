"""
Convergence diagnostics on the device: the split-R-hat kernels (csrc/irs_diagnostics.cu) against fp64 torch / numpy
restatements, the SGLDSampler integration (pooled moments untouched, sharding, checkpoints) and Trainer._run_MCMC(with_R_hat).
"""
import os
import socket

import numpy as np
import pytest
import torch

from tests.util import rel

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def pkg(built):
    from irsgmcmc_b200 import _lib, ops
    from irsgmcmc_b200.utils import diagnostics
    return ops, _lib, diagnostics


def _half_count(k, N):
    """the sampler's rule: (half, draws already in it) of kept sample k of N, None for the middle one of an odd N"""
    n = N // 2
    if k < n:
        return 0, k
    if k >= N - n:
        return 1, k - (N - n)
    return None


def _feed(ops, draws):
    """draws (N, C, 4, D, H, W) fp64 -> (mean, m2) (2, C, 4, D, H, W) through ops.split_welford_update, one sample at a time"""
    N, C = draws.shape[:2]
    mean = torch.zeros(2, *draws.shape[1:], device=DEV)
    m2 = torch.zeros_like(mean)
    for k in range(N):
        hc = _half_count(k, N)
        x = draws[k].float().to(DEV)
        if hc is not None:
            ops.split_welford_update(x[:, :3].contiguous(), x[:, 3:].contiguous(), hc[0], hc[1], mean, m2)
    return mean, m2


def _sequences(draws):
    N = draws.shape[0]
    n = N // 2
    return torch.stack((draws[:n], draws[N - n:])), n   # (2, n, C, 4, ...)


@pytest.mark.parametrize('dims,N', [((6, 7, 8), 9), ((5, 5, 5), 8)])   # float4 and scalar update paths; odd and even N
def test_update_and_rhat_against_fp64(pkg, dims, N):
    ops, _, diag = pkg
    C = 3
    g = torch.Generator().manual_seed(N)
    draws = (torch.randn(N, C, 4, *dims, generator=g, dtype=torch.float64) * 0.7 +
             0.3 * torch.randn(1, C, 4, *dims, generator=g, dtype=torch.float64))
    mean, m2 = _feed(ops, draws)
    seq, n = _sequences(draws)
    want_mean = seq.mean(1)                                      # (2, C, 4, ...)
    want_m2 = ((seq - want_mean[:, None]) ** 2).sum(1)
    assert rel(mean, want_mean) < 1e-5 and rel(m2, want_m2) < 1e-5, (rel(mean, want_mean), rel(m2, want_m2))

    mask = torch.rand(dims, generator=g) > 0.3
    V = int(np.prod(dims))
    rhat, summary, M = ops.split_rhat(mean.view(2 * C, 4, *dims), m2.view(2 * C, 4, *dims), n, mask.to(DEV))
    assert M == 2 * C and rhat.shape == (4, *dims)
    # numpy split_rhat of the stored draws, element by element (it splits the chains itself, dropping an odd N's middle)
    d = draws.numpy().reshape(N, C, 4 * V)
    want = np.array([diag.split_rhat(d[:, :, e].T) for e in range(4 * V)]).reshape(4, *dims)
    err = float(np.abs(rhat.cpu().numpy() - want).max())
    print(f'split R-hat {dims} N={N}: max |device - numpy| = {err:.3e}')
    assert err <= 1e-4
    # the middle sample of an odd N is not folded in
    if N % 2:
        changed = draws.clone()
        changed[N // 2] += 100.0
        m_b, m2_b = _feed(ops, changed)
        assert torch.equal(m_b, mean) and torch.equal(m2_b, m2)
    # mask summaries
    r = torch.from_numpy(want).float()
    for k in range(4):
        inside = r[k][mask]
        assert abs(summary[k, 0].item() - float(inside.max())) < 1e-4
        assert int(summary[k, 1]) == int((rhat[k].cpu()[mask] > 1.01).sum())
        assert int(summary[k, 2]) == int((rhat[k].cpu()[mask] > 1.1).sum())
    # the custom op is the same computation
    r_op, s_op = torch.ops.irsgmcmc.split_rhat(mean.view(2 * C, 4, *dims), m2.view(2 * C, 4, *dims), n, mask.to(DEV))
    assert torch.equal(r_op, rhat) and torch.equal(s_op, summary)


def test_edge_rules(pkg):
    ops = pkg[0]
    M, n, dims = 4, 5, (2, 2, 4)
    mean = torch.zeros(M, 1, *dims, device=DEV)
    m2 = torch.zeros_like(mean)
    mean.view(M, -1)[:, 1] = torch.arange(M, device=DEV, dtype=torch.float32)   # element 1: W = 0 < B
    m2.view(M, -1)[:, 2] = 1.0                                                  # element 2: B = 0, W > 0 -> sqrt((n-1)/n)
    rhat, summary, _ = ops.split_rhat(mean, m2, n, torch.ones(dims, dtype=torch.bool, device=DEV))
    flat = rhat.view(-1).cpu()
    assert flat[0] == 1.0 and flat[3] == 1.0 and flat[1] == float('inf')
    assert abs(float(flat[2]) - ((n - 1) / n) ** 0.5) < 1e-7
    assert summary[0, 0].item() == float('inf') and int(summary[0, 1]) == 1 == int(summary[0, 2])
    with pytest.raises(ValueError):
        ops.split_rhat(mean, m2, 1, torch.ones(dims, dtype=torch.bool, device=DEV))


def test_iid_and_shifted_chains(pkg):
    ops = pkg[0]
    C, N, dims = 8, 400, (16, 16, 16)                      # M = 16 sequences of n = 200
    g = torch.Generator(device=DEV).manual_seed(5)
    mean = torch.zeros(2, C, 4, *dims, device=DEV)
    m2 = torch.zeros_like(mean)
    shifted_mean, shifted_m2 = torch.zeros_like(mean), torch.zeros_like(mean)
    shift = torch.arange(C, device=DEV, dtype=torch.float32).view(C, 1, 1, 1, 1)
    for k in range(N):
        half, cnt = _half_count(k, N)
        x = torch.randn(C, 4, *dims, generator=g, device=DEV)
        ops.split_welford_update(x[:, :3].contiguous(), x[:, 3:].contiguous(), half, cnt, mean, m2)
        y = x + shift
        ops.split_welford_update(y[:, :3].contiguous(), y[:, 3:].contiguous(), half, cnt, shifted_mean, shifted_m2)
    mask = torch.ones(dims, dtype=torch.bool, device=DEV)
    rhat, _, M = ops.split_rhat(mean.view(2 * C, 4, *dims), m2.view(2 * C, 4, *dims), N // 2, mask)
    inside = ((rhat >= 0.97) & (rhat <= 1.03)).float().mean().item()
    print(f'iid chains: {100 * inside:.3f} % of R-hat in [0.97, 1.03], max {rhat.max().item():.4f}')
    assert M == 16 and inside >= 0.99
    rs, summary, _ = ops.split_rhat(shifted_mean.view(2 * C, 4, *dims), shifted_m2.view(2 * C, 4, *dims), N // 2, mask)
    assert rs.min().item() > 1.5 and int(summary[:, 2].sum()) == rs.numel()


# ---- sampler ----------------------------------------------------------------------------------------------------------------
def _sampler(C, n=16, chain_offset=0, mode='per_chain', seed=0, **kw):
    from irsgmcmc_b200.sampler import SGLDSampler, SGLDConfig
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    fixed, moving, vp = make_pair(n)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(hyper_mode=mode, **kw), device=DEV, chain_offset=chain_offset)
    gen = torch.Generator().manual_seed(seed)
    v0 = 0.5 * torch.randn(4, 3, n, n, n, generator=gen)[chain_offset:chain_offset + C]
    s.set_state(v0, torch.full((1, 3, n, n, n), 0.5))
    s.init_gmm(sigma_hat=0.7)
    return s


def test_pooled_moments_and_states_unchanged(pkg):
    outs = []
    for on in (False, True):
        s = _sampler(4, mode='reference')
        if on:
            s.enable_convergence_diagnostics(6)
        for _ in range(6):
            s.step(2)
            s.accumulate()
        torch.cuda.synchronize()
        outs.append((s.posterior_moments(), s.v.clone(), s.hyper.clone()))
        if on:
            with pytest.raises(RuntimeError, match='sample 7'):
                s.accumulate()
            d = s.convergence_diagnostics()
            assert d['displacement'].shape == (3, 16, 16, 16) and d['im'].shape == (1, 16, 16, 16) and d['M'] == 8
            assert d['n'] == 3 and len(d['mask']['displacement']['max']) == 3 and len(d['mask']['im']['n_above_1.1']) == 1
    (a, va, ha), (b, vb, hb) = outs
    assert torch.equal(va, vb) and torch.equal(ha, hb)
    for key in ('displacement_mean', 'displacement_std', 'im_mean', 'im_std'):
        assert torch.equal(a[key], b[key]), key
    assert a['n'] == b['n'] == 24


def test_needs_all_samples(pkg):
    s = _sampler(2)
    with pytest.raises(RuntimeError, match='not enabled'):
        s.convergence_diagnostics()
    with pytest.raises(ValueError):
        s.enable_convergence_diagnostics(3)
    s.enable_convergence_diagnostics(5)
    for _ in range(4):
        s.step(1)
        s.accumulate()
    with pytest.raises(RuntimeError, match='4 accumulated'):
        s.convergence_diagnostics()
    s.step(1)
    s.accumulate()
    assert s.convergence_diagnostics()['n'] == 2


def test_sharded_partials_match_one_sampler(pkg):
    """two samplers of 2 chains (chain_offset 0 and 2), their partial sums added as the all-reduce would, against one sampler of
    4 chains.  The shards accumulate the 4-chain sampler's samples of their chains (copied into their output buffers), so the
    comparison is of the diagnostics alone, not of transitions run with other launch shapes."""
    ops, L, _ = pkg
    N, n = 6, 16
    whole = _sampler(4)
    shards = [_sampler(2, chain_offset=o) for o in (0, 2)]
    for s in [whole] + shards:
        s.enable_convergence_diagnostics(N)
    for _ in range(N):
        whole.step(2)
        whole.accumulate()
        for o, s in zip((0, 2), shards):
            s.displacement.copy_(whole.displacement[o:o + 2])
            s.im_warped.copy_(whole.im_warped[o:o + 2])
            s.accumulate()
    want = whole.convergence_diagnostics()
    lib, E, V = L.load(), 4 * n ** 3, n ** 3
    views = [(s._rhat['mean'].view(4, E), s._rhat['m2'].view(4, E)) for s in shards]
    sums = torch.zeros(2, E, device=DEV, dtype=torch.float64)
    for m, m2 in views:
        part = torch.empty(2, E, device=DEV, dtype=torch.float64)
        L.check(lib.irs_split_rhat_sums(L.ptr(m), L.ptr(m2), 4, E, N // 2, L.ptr(part), L.stream()))
        sums += part
    sb = torch.zeros(E, device=DEV, dtype=torch.float64)
    for m, _ in views:
        part = torch.empty(E, device=DEV, dtype=torch.float64)
        L.check(lib.irs_split_rhat_between(L.ptr(m), 4, E, L.ptr(sums[0]), 8, L.ptr(part), L.stream()))
        sb += part
    rhat = torch.empty(4, V, device=DEV)
    summary = torch.empty(4, 3, device=DEV, dtype=torch.float64)
    partials = torch.empty(L.RHAT_PARTIALS_DOUBLES, device=DEV, dtype=torch.float64)
    counters = torch.empty(4, device=DEV, dtype=torch.int32)
    L.check(lib.irs_split_rhat_finish(L.ptr(sums[1]), L.ptr(sb), 8, N // 2, L.ptr(whole.mask), 4, V, L.ptr(rhat),
                                      L.ptr(partials), L.ptr(counters), L.ptr(summary), L.stream()))
    got = rhat.view(4, n, n, n)
    err = max(float((got[:3] - want['displacement']).abs().max()), float((got[3:] - want['im']).abs().max()))
    print('sharded vs one sampler: max |R-hat difference| =', err)
    assert err <= 1e-6


def test_power_chains_started_far_apart(pkg):
    """chains started from velocity fields far apart with a tiny step have not mixed: max R-hat in the mask > 1.1"""
    n, C, N = 16, 4, 8
    s = _sampler(C, mode='per_chain', tau=1e-4)
    v = torch.stack([torch.full((3, n, n, n), 1.5 * (c - 1.5)) for c in range(C)])
    s.set_state(v, torch.full((1, 3, n, n, n), 0.5))
    s.enable_convergence_diagnostics(N)
    for _ in range(N):
        s.step(1)
        s.accumulate()
    d = s.convergence_diagnostics()
    print('power test: max R-hat in the mask', d['mask']['displacement']['max'], d['mask']['im']['max'])
    assert max(d['mask']['displacement']['max']) > 1.1 and sum(d['mask']['displacement']['n_above_1.1']) > 0


def test_checkpoint_resume_with_diagnostics(pkg, tmp_path):
    a = _sampler(2, chain_offset=1, mode='per_chain')
    a.enable_convergence_diagnostics(7)
    for _ in range(3):
        a.step(2)
        a.accumulate()
    torch.save(a.state_dict(), tmp_path / 'chains.pt')
    for _ in range(4):
        a.step(2)
        a.accumulate()
    b = _sampler(2, chain_offset=1, mode='per_chain')
    assert not b.diagnostics_enabled
    b.load_state_dict(torch.load(tmp_path / 'chains.pt'))
    assert b.diagnostics_enabled
    for _ in range(4):
        b.step(2)
        b.accumulate()
    torch.cuda.synchronize()
    da, db = a.convergence_diagnostics(), b.convergence_diagnostics()
    assert torch.equal(a._rhat['mean'], b._rhat['mean']) and torch.equal(a._rhat['m2'], b._rhat['m2'])
    assert torch.equal(da['displacement'], db['displacement']) and torch.equal(da['im'], db['im']) and da['mask'] == db['mask']
    assert torch.equal(a.disp_mean, b.disp_mean) and torch.equal(a.v, b.v)


def test_resume_from_checkpoint_without_diagnostics(pkg, tmp_path):
    a = _sampler(2, mode='per_chain')
    a.step(2)
    a.accumulate()
    sd = a.state_dict()
    assert 'rhat' not in sd
    torch.save(sd, tmp_path / 'old.pt')
    a.step(2)
    a.accumulate()
    for enabled in (False, True):
        b = _sampler(2, mode='per_chain')
        if enabled:   # diagnostics enabled here restart from zero kept samples
            b.enable_convergence_diagnostics(4)
            b.step(1)
            b.accumulate()
        b.load_state_dict(torch.load(tmp_path / 'old.pt'))
        assert b.diagnostics_enabled == enabled and (not enabled or b._rhat['k'] == 0)
        b.step(2)
        b.accumulate()
        torch.cuda.synchronize()
        assert torch.equal(a.v, b.v) and torch.equal(a.disp_mean, b.disp_mean) and torch.equal(a.im_m2, b.im_m2)


# ---- trainer ----------------------------------------------------------------------------------------------------------------
def _config(C, burn_in=2, samples=8, period=1):
    return {'data_loss': {'type': 'GMM', 'args': {'no_components': 4, 's': 2}},
            'reg_loss': {'type': 'RegLoss_LogNormal', 'args': {'diff_op': 'GradientOperator', 'w_reg': 1.6, 'learnable': True}},
            'optimizer_SG_MCMC': {'type': 'SGD', 'args': {'lr': 0.4}},
            'Sobolev_grad': {'enabled': True, 's': 3, 'lambda': 0.5}, 'virtual_decimation': True,
            'trainer': {'MCMC_init': 'VI', 'no_chains': C, 'no_iters_burn_in': burn_in, 'no_samples_MCMC': samples,
                        'log_period_MCMC': period, 'uniform_noise': {'enabled': True, 'magnitude': 0.1}}}


def _trainer(n, C, save_dir=None, device=DEV):
    from irsgmcmc_b200.trainer import Trainer, sampler_config_from_json
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n)
    cfg = _config(C)
    from irsgmcmc_b200.sampler import SGLDConfig
    sc = SGLDConfig(**dict(sampler_config_from_json(cfg).__dict__, hyper_mode='per_chain'))
    return Trainer(cfg, fixed, moving, vp, device=torch.device(device), save_dir=save_dir, sampler_config=sc)


def _check_R_hat(R, n, M):
    assert R['displacement'].shape == (3, n, n, n) and R['im'].shape == (1, n, n, n) and R['M'] == M and R['n'] == 4
    assert torch.isfinite(R['displacement']).all() and (R['displacement'] > 0).all()
    assert set(R['mask']) == {'displacement', 'im'} and len(R['mask']['displacement']['max']) == 3
    assert set(R['traces']) == {'data', 'reg', 'alpha', 'reg_energy'}
    for q in R['traces'].values():
        assert set(q) == {'R_hat', 'ESS'} and q['R_hat'] > 0


def test_run_MCMC_with_R_hat(pkg, tmp_path):
    n, C = 32, 4
    plain = _trainer(n, C)._run_MCMC(speed_test_iters=0)
    assert set(plain) == {'mean', 'std_dev', 'im_mean', 'im_std', 'n', 'DSC', 'no_non_diffeomorphic_voxels', 'ASD'}
    t = _trainer(n, C, save_dir=str(tmp_path))
    res = t._run_MCMC(speed_test_iters=0, with_R_hat=True)
    assert set(res) == set(plain) | {'R_hat'}
    _check_R_hat(res['R_hat'], n, 2 * C)
    print('trainer R-hat mask summary', res['R_hat']['mask'], 'traces', res['R_hat']['traces'])
    for key in ('mean', 'std_dev', 'im_mean', 'im_std'):   # the diagnostics change no number of the run
        assert torch.equal(res[key], plain[key]), key
    assert res['n'] == plain['n'] == 8 * C and not t.sampler.diagnostics_enabled
    from irsgmcmc_b200.logger import load_field_from_disk, load_im_from_disk
    f, _ = load_field_from_disk(tmp_path / 'MCMC_R_hat_displacement.vtk')
    im, _ = load_im_from_disk(tmp_path / 'MCMC_R_hat_im.nii.gz')
    assert np.array_equal(f, res['R_hat']['displacement'].cpu().numpy())
    assert np.array_equal(im, res['R_hat']['im'][0].cpu().numpy())
    # drop-in modules cannot mirror per-chain parameters
    with pytest.raises(NotImplementedError):
        t._push_hyper(object(), None)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n, C, out_dir):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world)
    res = _trainer(n, C, device=f'cuda:{rank}')._run_MCMC(speed_test_iters=0, with_R_hat=True)
    R = res['R_hat']
    torch.save({'disp': R['displacement'].cpu(), 'im': R['im'].cpu(), 'M': R['M'], 'mask': R['mask'], 'traces': R['traces']},
               os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


def test_run_MCMC_with_R_hat_two_gpus(pkg, tmp_path):
    """4 chains over two GPUs: every rank gets the same maps and summaries over all 8 sequences"""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    n, C = 32, 4
    mp.spawn(_worker, args=(2, _free_port(), n, C, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / 'r0.pt'), torch.load(tmp_path / 'r1.pt')
    assert r0['M'] == r1['M'] == 2 * C
    assert torch.equal(r0['disp'], r1['disp']) and torch.equal(r0['im'], r1['im'])
    assert r0['mask'] == r1['mask'] and r0['traces'] == r1['traces']
    one = _trainer(n, C)._run_MCMC(speed_test_iters=0, with_R_hat=True)['R_hat']
    assert float((one['displacement'].cpu() - r0['disp']).abs().max()) < 1e-3
