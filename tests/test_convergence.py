"""
Convergence diagnostics, what can be checked without a GPU:
 - utils.diagnostics.split_rhat / ess against a brute-force loop restatement of BDA3 sections 11.4-11.5, their edge rules, and
   their statistics on iid and AR(1) chains;
 - argument validation of the split-R-hat entry points of the C ABI;
 - the schema / fake implementation of irsgmcmc::split_rhat and its refusal of CPU tensors;
 - parallel.split_rhat_totals over a world-size-2 gloo group against the single-process combination.
"""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from irsgmcmc_b200.utils.diagnostics import ess, split_rhat


# ---- brute-force restatements (plain loops) ----------------------------------------------------------------------------
def _split(draws):
    draws = [list(map(float, c)) for c in draws]
    N = len(draws[0])
    n = N // 2
    return [c[:n] for c in draws] + [c[N - n:] for c in draws], n


def _mean(xs):
    return sum(xs) / len(xs)


def _var(xs):
    m = _mean(xs)
    return sum((x - m) ** 2 for x in xs) / (len(xs) - 1)


def brute_rhat(draws):
    seqs, n = _split(draws)
    W = _mean([_var(s) for s in seqs])
    B_n = _var([_mean(s) for s in seqs])
    if W == 0.0:
        return 1.0 if B_n == 0.0 else math.inf
    return math.sqrt(((n - 1) / n * W + B_n) / W)


def brute_ess(draws):
    seqs, n = _split(draws)
    M = len(seqs)
    var_plus = (n - 1) / n * _mean([_var(s) for s in seqs]) + _var([_mean(s) for s in seqs])
    rho = []
    for t in range(n):
        V = 0.0
        for s in seqs:
            V += sum((s[i + t] - s[i]) ** 2 for i in range(n - t)) / (n - t)
        rho.append(1.0 - V / M / (2.0 * var_plus))
    total, prev, k = 0.0, math.inf, 0
    while k + 1 < n:
        p = rho[k] + rho[k + 1]
        if p <= 0.0:
            break
        p = min(p, prev)
        total += p
        prev = p
        k += 2
    return M * n / (-1.0 + 2.0 * total)


def _ar1(rng, chains, N, rho):
    x = np.empty((chains, N))
    x[:, 0] = rng.standard_normal(chains) / math.sqrt(1 - rho ** 2)
    e = rng.standard_normal((chains, N))
    for i in range(1, N):
        x[:, i] = rho * x[:, i - 1] + e[:, i]
    return x


@pytest.mark.parametrize('shape,shift,rho', [((4, 40), 0.0, 0.0), ((3, 41), 0.0, 0.6), ((2, 30), 2.0, 0.0), ((5, 9), 0.3, -0.4)])
def test_split_rhat_and_ess_match_brute_force(shape, shift, rho):
    rng = np.random.default_rng(sum(shape))
    x = _ar1(rng, shape[0], shape[1], rho) + shift * np.arange(shape[0])[:, None]
    assert abs(split_rhat(x) - brute_rhat(x)) < 1e-12 * brute_rhat(x)
    assert abs(ess(x) - brute_ess(x)) < 1e-9 * abs(brute_ess(x))


def test_edge_rules():
    same = np.full((3, 10), 2.5)
    assert split_rhat(same) == 1.0 == brute_rhat(same)
    assert math.isnan(ess(same))
    per_chain_constant = np.repeat(np.arange(3.0)[:, None], 10, axis=1)   # W = 0 < B
    assert split_rhat(per_chain_constant) == math.inf == brute_rhat(per_chain_constant)
    # odd N: the middle draw belongs to neither half
    x = np.random.default_rng(0).standard_normal((2, 9))
    y = x.copy()
    y[:, 4] = 1e6
    assert split_rhat(x) == split_rhat(y) and ess(x) == ess(y)
    with pytest.raises(ValueError):
        split_rhat(np.zeros((2, 3)))
    with pytest.raises(ValueError):
        ess(np.zeros(8))


def test_iid_chains():
    rng = np.random.default_rng(1)
    chains, N = 8, 1000
    rh, es = [], []
    for _ in range(20):
        x = rng.standard_normal((chains, N))
        rh.append(split_rhat(x))
        es.append(ess(x))
    assert all(abs(r - 1.0) < 0.02 for r in rh), rh
    # the estimate of M n = 8000 independent draws: its Monte-Carlo spread is a few per cent
    assert 0.85 * chains * N < np.mean(es) < 1.15 * chains * N and min(es) > 0.7 * chains * N, es
    shifted = rng.standard_normal((chains, N)) + 0.5 * np.arange(chains)[:, None]
    assert split_rhat(shifted) > 1.1


def test_ar1_ess_near_analytic():
    rng = np.random.default_rng(2)
    chains, N, rho = 4, 20000, 0.5
    x = _ar1(rng, chains, N, rho)
    want = chains * N * (1 - rho) / (1 + rho)
    got = ess(x)
    assert abs(got - want) < 0.1 * want, (got, want)
    assert abs(split_rhat(x) - 1.0) < 0.01


# ---- C ABI ---------------------------------------------------------------------------------------------------------------
def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call: null pointers, n < 2, M < 2, a half index outside {0, 1}, too many components"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    f = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    upd = lib.irs_split_welford_update
    assert upd(f, f, 2, 64, 2, 0.0, f, f, None) == -1
    assert upd(f, f, 2, 64, -1, 0.0, f, f, None) == -1
    assert upd(None, f, 2, 64, 0, 0.0, f, f, None) == -1
    assert upd(f, f, 2, 64, 0, 0.0, f, None, None) == -1
    assert upd(f, f, 0, 64, 0, 0.0, f, f, None) == -1
    assert upd(f, f, 2, 64, 1, -1.0, f, f, None) == -1
    sums = lib.irs_split_rhat_sums
    assert sums(f, f, 4, 64, 1, f, None) == -1
    assert sums(f, None, 4, 64, 5, f, None) == -1
    assert sums(f, f, 0, 64, 5, f, None) == -1
    btw = lib.irs_split_rhat_between
    assert btw(f, 4, 64, f, 1, f, None) == -1
    assert btw(f, 4, 64, None, 8, f, None) == -1
    assert btw(f, 9, 64, f, 8, f, None) == -1   # more local sequences than in total
    fin = lib.irs_split_rhat_finish
    assert fin(f, f, 8, 1, f, 4, 16, f, f, f, f, None) == -1
    assert fin(f, f, 1, 5, f, 4, 16, f, f, f, f, None) == -1
    assert fin(f, f, 8, 5, f, 5, 16, f, f, f, f, None) == -1
    assert fin(f, f, 8, 5, None, 4, 16, f, f, f, f, None) == -1
    assert fin(f, f, 8, 5, f, 4, 16, f, f, f, None, None) == -1


# ---- custom op -------------------------------------------------------------------------------------------------------------
def test_fake_implementation_and_cpu_refusal(built):
    import irsgmcmc_b200  # noqa: F401
    from irsgmcmc_b200 import torch_ops
    from torch._subclasses.fake_tensor import FakeTensorMode
    assert 'split_rhat' in torch_ops.OPS
    with FakeTensorMode():
        mean = torch.empty(6, 4, 8, 9, 10, device='cuda')
        mask = torch.empty(8, 9, 10, device='cuda', dtype=torch.bool)
        rhat, summary = torch.ops.irsgmcmc.split_rhat(mean, mean, 5, mask)
        assert rhat.shape == (4, 8, 9, 10) and rhat.dtype == torch.float32 and rhat.device.type == 'cuda'
        assert summary.shape == (4, 3) and summary.dtype == torch.float64
    m = torch.zeros(4, 1, 6, 6, 6)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        torch.ops.irsgmcmc.split_rhat(m, m, 3, torch.ones(6, 6, 6, dtype=torch.bool))
    from irsgmcmc_b200 import ops
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.split_rhat(m, m, 3, torch.ones(6, 6, 6, dtype=torch.bool))


# ---- the collective phases over gloo ------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _partials(mean, m2, n):
    """torch restatement of the two local kernels: (sums (2, E), between(s1, M))"""
    sums = torch.stack((mean.sum(0), (m2 / (n - 1)).sum(0)))
    return sums, lambda s1, M: ((mean - s1 / M) ** 2).sum(0)


def _worker(rank, world, port, mean, m2, n, counts, out_dir):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from irsgmcmc_b200 import parallel
    o = sum(counts[:rank])
    sums, between = _partials(mean[o:o + counts[rank]], m2[o:o + counts[rank]], n)
    M, tot, sb = parallel.split_rhat_totals(counts[rank], sums, between)
    torch.save({'M': M, 'sums': tot, 'sb': sb}, os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


@pytest.mark.parametrize('counts', [(5, 4), (1, 1)])
def test_split_rhat_totals_world_size_2(tmp_path, counts):
    torch.manual_seed(0)
    M, E, n = sum(counts), 37, 6
    mean = torch.randn(M, E, dtype=torch.float64) + torch.arange(M, dtype=torch.float64)[:, None] * 0.1
    m2 = torch.rand(M, E, dtype=torch.float64) * (n - 1)
    mp.spawn(_worker, args=(2, _free_port(), mean, m2, n, counts, str(tmp_path)), nprocs=2, join=True)
    from irsgmcmc_b200 import parallel
    sums, between = _partials(mean, m2, n)
    M1, want_sums, want_sb = parallel.split_rhat_totals(M, sums, between)   # single process: the local combination
    assert M1 == M
    rs = [torch.load(tmp_path / f'r{r}.pt') for r in (0, 1)]
    for r in rs:
        assert r['M'] == M
        assert torch.allclose(r['sums'], want_sums, rtol=1e-12, atol=1e-12)
        assert torch.allclose(r['sb'], want_sb, rtol=1e-12, atol=1e-12)
    assert torch.equal(rs[0]['sums'], rs[1]['sums']) and torch.equal(rs[0]['sb'], rs[1]['sb'])
