"""
Jacobian posterior, what can be checked without a GPU:
 - the numpy restatement the GPU tests compare the kernels with (tests/helpers/jacobian_posterior_ref.py) against plain loops over
   the definitions, with voxels that fold in some samples, in every sample and in none, and NaN / -inf / +inf log det values;
 - its log det J against loops and against the reference's folded voxels of the golden transformation;
 - argument validation of irs_jacobian_update / irs_jacobian_posterior (refused before any CUDA call);
 - parallel.merge_jacobian_moments over a world-size-2 gloo group against one process holding all samples.
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

from tests.helpers import jacobian_posterior_ref as ref

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'eval.npz')


def _lds(N, V, seed):
    """(N, V) log det values: voxel 0 folds in every sample, voxel 1 in none, the others at random (NaN, -inf, +inf)"""
    g = np.random.default_rng(seed)
    x = g.normal(0.0, 0.3, size=(N, V))
    bad = g.random((N, V)) < 0.3
    x[bad] = g.choice([np.nan, -np.inf, np.inf], size=int(bad.sum()))
    x[:, 0] = np.nan
    x[:, 1] = g.normal(0.0, 0.3, size=N)
    return x


def _brute(x, mask):
    N, V = x.shape
    folds, mean, m2 = [], [], []
    for v in range(V):
        vals = [float(x[j, v]) for j in range(N) if math.isfinite(x[j, v])]
        folds.append(N - len(vals))
        m = sum(vals) / len(vals) if vals else 0.0
        mean.append(m)
        m2.append(sum((a - m) ** 2 for a in vals))
    p, mo, so = [], [], []
    for v in range(V):
        nv = N - folds[v]
        p.append(np.float32(folds[v]) / np.float32(N))
        mo.append(mean[v] if nv >= 1 else float('nan'))
        so.append(math.sqrt(m2[v] / (nv - 1)) if nv >= 2 else float('nan'))
    inm = [v for v in range(V) if mask[v]]
    summ = {'sum_folds': sum(folds[v] for v in inm), 'voxels_ever_folded': sum(1 for v in inm if folds[v] > 0),
            'voxels_folded_in_majority': sum(1 for v in inm if 2 * folds[v] > N),
            'voxels_finite': sum(1 for v in inm if N - folds[v] >= 1), 'voxels_finite_2': sum(1 for v in inm if N - folds[v] >= 2),
            'mask_voxels': len(inm)}
    f1 = [mo[v] for v in inm if N - folds[v] >= 1]
    f2 = [so[v] for v in inm if N - folds[v] >= 2]
    summ['mean_log_det_J'] = sum(f1) / len(f1) if f1 else float('nan')
    summ['mean_std_log_det_J'] = sum(f2) / len(f2) if f2 else float('nan')
    stats = []
    for j in range(N):
        fin = [float(x[j, v]) for v in inm if math.isfinite(x[j, v])]
        stats.append([len(fin), len(inm) - len(fin), sum(fin), sum(a * a for a in fin)])
    return folds, mean, m2, p, mo, so, summ, stats


@pytest.mark.parametrize('N,V,seed', [(7, 40, 0), (2, 13, 1), (1, 9, 2), (12, 30, 3)])
def test_restatement_matches_loops(N, V, seed):
    x = _lds(N, V, seed)
    mask = np.random.default_rng(seed + 10).random(V) < 0.7
    mask[:2] = True
    folds, mean, m2 = ref.accumulate(x)
    p, mo, so, summ = ref.posterior(folds, mean, m2, N, mask)
    bf, bm, bm2, bp, bmo, bso, bsumm, bstats = _brute(x, mask)
    assert folds.dtype == np.int32 and folds.tolist() == bf
    assert folds[0] == N and folds[1] == 0
    assert np.allclose(mean, bm, rtol=0, atol=1e-12) and np.allclose(m2, bm2, rtol=0, atol=1e-12)
    assert p.dtype == np.float32 and np.array_equal(p, np.asarray(bp, np.float32))
    assert np.allclose(mo, bmo, rtol=0, atol=1e-12, equal_nan=True) and np.allclose(so, bso, rtol=0, atol=1e-12, equal_nan=True)
    for key in ('sum_folds', 'voxels_ever_folded', 'voxels_folded_in_majority', 'voxels_finite', 'voxels_finite_2', 'mask_voxels'):
        assert summ[key] == bsumm[key], key
    for key in ('mean_log_det_J', 'mean_std_log_det_J'):
        assert math.isclose(summ[key], bsumm[key], rel_tol=1e-12, abs_tol=1e-12) or \
            (math.isnan(summ[key]) and math.isnan(bsumm[key])), key
    stats = np.stack([ref.sample_stats(x[j:j + 1], mask)[0] for j in range(N)])
    assert np.allclose(stats, bstats, rtol=1e-12, atol=1e-12)


def test_no_folds_is_plain_welford_statistics():
    x = np.random.default_rng(5).normal(size=(6, 20))
    folds, mean, m2 = ref.accumulate(x)
    assert (folds == 0).all() and np.allclose(mean, x.mean(0)) and np.allclose(m2, ((x - x.mean(0)) ** 2).sum(0))
    _, _, std, summ = ref.posterior(folds, mean, m2, 6, np.ones(20, bool))
    assert np.allclose(std, x.std(0, ddof=1)) and summ['sum_folds'] == 0 and summ['voxels_ever_folded'] == 0


def test_sdlogj_is_population_std():
    x = np.random.default_rng(6).normal(size=(3, 50))
    x[1, :5] = np.nan
    mask = np.ones(50, bool)
    s = ref.sample_stats(x, mask)
    want = [np.std(r[np.isfinite(r)]) for r in x]
    assert np.allclose(ref.sdlogj(s), want, rtol=1e-12) and s[1, 1] == 5


def test_log_det_j_against_loops_and_golden():
    g = np.random.default_rng(7)
    C, D, H, W = 2, 3, 4, 5
    T = g.normal(size=(C, 3, D, H, W))
    ld = ref.log_det_j(T)
    for c in range(C):
        for z in range(D):
            for y in range(H):
                for x in range(W):
                    ix, iy, iz = min(x, W - 2), min(y, H - 2), min(z, D - 2)
                    J = np.empty((3, 3))
                    for ch in range(3):
                        f = T[c, ch]
                        J[0, ch] = (f[z, y, ix + 1] - f[z, y, ix]) * (W - 1) / 2
                        J[1, ch] = (f[z, iy + 1, x] - f[z, iy, x]) * (H - 1) / 2
                        J[2, ch] = (f[iz + 1, y, x] - f[iz, y, x]) * (D - 1) / 2
                    det = np.linalg.det(J)
                    want = math.log(det) if det > 0 else float('nan')
                    got = ld[c, z, y, x]
                    assert (math.isnan(want) and not math.isfinite(got)) or math.isclose(got, want, rel_tol=1e-9, abs_tol=1e-9)
    gold = np.load(GOLDEN)
    ld = ref.log_det_j(gold['T'])
    folds, _, _ = ref.accumulate(ld)
    assert int((~np.isfinite(ld)).sum()) == int(np.isnan(gold['log_det_J']).sum()) == 826
    assert np.array_equal(~np.isfinite(ld), np.isnan(gold['log_det_J']))
    assert int(folds.sum()) == 826


# ---- C ABI ---------------------------------------------------------------------------------------------------------------
def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call (-1, or -2 for sizes the library does not support): null pointers, C < 1, a dimension
    < 2, count_before < 0 or past 2^24 samples; n outside 1..2^24, V < 1"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    f = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    names = ('T', 'mask', 'C', 'D', 'H', 'W', 'count', 'folds', 'mean', 'm2', 'stats', 'partials', 'counters')
    good = dict(T=f, mask=f, C=2, D=4, H=4, W=4, count=0.0, folds=f, mean=f, m2=f, stats=f, partials=f, counters=f)
    upd = lambda **kw: lib.irs_jacobian_update(*[kw.get(k, good[k]) for k in names], None)
    for key in ('T', 'mask', 'folds', 'mean', 'm2', 'stats', 'partials', 'counters'):
        assert upd(**{key: None}) == -1, key
    assert upd(C=0) == -1 and upd(D=1) == -1 and upd(W=1) == -1
    assert upd(C=70000) == -2 and upd(D=2048, H=2048, W=2048) == -2
    assert upd(count=-1.0) == -1 and upd(count=float('nan')) == -1 and upd(count=float(2 ** 24 - 1)) == -1
    pnames = ('folds', 'mean', 'm2', 'n', 'V', 'mask', 'p', 'mo', 'so', 'partials', 'counters', 'summary')
    pgood = dict(folds=f, mean=f, m2=f, n=3, V=64, mask=f, p=f, mo=f, so=f, partials=f, counters=f, summary=f)
    post = lambda **kw: lib.irs_jacobian_posterior(*[kw.get(k, pgood[k]) for k in pnames], None)
    for key in ('folds', 'mean', 'm2', 'mask', 'p', 'mo', 'so', 'partials', 'counters', 'summary'):
        assert post(**{key: None}) == -1, key
    assert post(n=0) == -1 and post(n=2 ** 24 + 1) == -1 and post(V=0) == -1


def test_ops_refuse_cpu_tensors(built):
    from irsgmcmc_b200 import ops
    T = torch.zeros(1, 3, 4, 4, 4)
    folds, mean, m2 = torch.zeros(4, 4, 4, dtype=torch.int32), torch.zeros(4, 4, 4), torch.zeros(4, 4, 4)
    mask = torch.ones(4, 4, 4, dtype=torch.bool)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.jacobian_update(T, mask, 0, folds, mean, m2)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.jacobian_posterior(folds, mean, m2, 1, mask)


# ---- the merge over gloo -------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _local(x):
    """fp32 accumulators as the device keeps them"""
    folds, mean, m2 = ref.accumulate(x)
    return torch.from_numpy(folds), torch.from_numpy(mean.astype(np.float32)), torch.from_numpy(m2.astype(np.float32))


def _worker(rank, world, port, parts, out_dir):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from irsgmcmc_b200 import parallel
    folds, mean, m2 = (t.view(3, 4, 5) for t in _local(parts[rank]))
    before = (folds.clone(), mean.clone(), m2.clone())
    n, f, m, s = parallel.merge_jacobian_moments(len(parts[rank]), folds, mean, m2)
    kept = all(torch.equal(a, b) for a, b in zip(before, (folds, mean, m2)))
    torch.save({'n': n, 'folds': f, 'mean': m, 'm2': s, 'kept': kept}, os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


def test_merge_jacobian_moments_world_size_2(tmp_path):
    x = _lds(13, 60, 11)
    x[:, 2] = np.nan            # folds on every sample of both ranks
    x[:8, 3] = np.nan           # every sample of rank 0 folds, rank 1 has finite ones
    parts = [x[:8], x[8:]]
    mp.spawn(_worker, args=(2, _free_port(), parts, str(tmp_path)), nprocs=2, join=True)
    folds, mean, m2 = ref.accumulate(x)
    for r in (0, 1):
        res = torch.load(tmp_path / f'r{r}.pt')
        assert res['n'] == 13 and res['kept']
        assert res['folds'].dtype == torch.int32 and res['folds'].shape == (3, 4, 5)
        assert np.array_equal(res['folds'].numpy().reshape(-1), folds)
        ok = folds < 13
        # fp32 accumulators and an fp32 merge: a few ulps of the values and of sum (x - mean)^2
        assert np.allclose(res['mean'].numpy().reshape(-1)[ok], mean[ok], rtol=1e-6, atol=1e-6)
        assert np.allclose(res['m2'].numpy().reshape(-1)[ok], m2[ok], rtol=1e-5, atol=1e-5)
        assert (res['mean'].numpy().reshape(-1)[~ok] == 0).all() and (res['m2'].numpy().reshape(-1)[~ok] == 0).all()
    from irsgmcmc_b200 import parallel
    f, m, s = _local(x)
    n, f2, m2_, s2 = parallel.merge_jacobian_moments(13, f, m, s)   # no process group: copies of the local accumulators
    assert n == 13 and torch.equal(f2, f) and torch.equal(m2_, m) and torch.equal(s2, s) and f2.data_ptr() != f.data_ptr()
