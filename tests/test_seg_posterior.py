"""
Segmentation posterior, what can be checked without a GPU:
 - the numpy restatement the GPU tests compare the kernels with (tests/helpers/seg_posterior_ref.py) against plain loops over
   the definitions, ties included;
 - argument validation of irs_label_counts_update / irs_label_posterior (refused before any CUDA call);
 - the schemas and fake implementations of irsgmcmc::label_counts_update / ::label_posterior and their refusal of CPU tensors;
 - parallel.merge_label_counts over a world-size-2 gloo group against the sum of the local counts.
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

from tests.helpers import seg_posterior_ref as ref


# ---- the numpy restatement against loops -----------------------------------------------------------------------------------
def brute(segs, labels, seg_fixed):
    """per voxel, straight from the definitions"""
    N, V = len(segs), segs[0].size
    flat = [np.asarray(s).reshape(-1) for s in segs]
    fixed = np.asarray(seg_fixed).reshape(-1)
    L = len(labels)
    counts = [[0] * V for _ in range(L)]
    for s in flat:
        for v in range(V):
            for l in range(L):
                if int(s[v]) == labels[l]:
                    counts[l][v] += 1
    majority, entropy = [], []
    for v in range(V):
        other = N - sum(counts[l][v] for l in range(L))
        best, lab = other, 0                       # "other" first: it keeps every tie
        for l in range(L):
            if counts[l][v] > best:               # then the earlier label keeps a tie
                best, lab = counts[l][v], labels[l]
        majority.append(lab)
        h = 0.0
        for c in [other] + [counts[l][v] for l in range(L)]:
            if c:
                h -= c / N * math.log(c / N)
        entropy.append(h)
    summary = []
    for l in range(L):
        summary.append([sum(counts[l]), sum(counts[l][v] for v in range(V) if int(fixed[v]) == labels[l]),
                        sum(1 for v in range(V) if 0 < counts[l][v] < N)])
    return counts, majority, entropy, summary


@pytest.mark.parametrize('N,labels,seed', [(5, [3, 7, 11], 0), (4, [2, -5], 1), (6, [1, 2, 3, 4], 2), (1, [9], 3)])
def test_restatement_matches_loops(N, labels, seed):
    rng = np.random.default_rng(seed)
    values = np.array(labels + [0, 0, -1, 300, 1000], dtype=np.int16)   # "other": 0, negative, > 255, not in the list
    segs = values[rng.integers(0, len(values), size=(N, 3, 4, 5))]
    fixed = values[rng.integers(0, len(values), size=(3, 4, 5))]
    counts = ref.label_counts(segs, labels)
    prob, majority, entropy, summary = ref.label_posterior(counts, N, labels, fixed)
    bc, bm, be, bs = brute(segs, labels, fixed)
    assert counts.dtype == np.int32 and counts.tolist() == bc
    assert majority.dtype == np.int16 and majority.tolist() == bm
    assert np.allclose(entropy, be, rtol=0, atol=1e-12)
    assert summary.dtype == np.int64 and summary.tolist() == bs
    assert prob.dtype == np.float32 and np.array_equal(prob, np.float32(counts) / np.float32(N))


def test_ties():
    labels = [4, 8, 2]
    # voxel 0: other 2, label 4 2 -> other;  voxel 1: 4 and 8 twice each -> 4 (earlier);  voxel 2: 8 and 2 twice each -> 8;
    # voxel 3: all four distinct classes once -> other;  voxel 4: 2 three times -> 2
    segs = np.array([[0, 4, 8, 0, 2], [0, 4, 8, 4, 2], [4, 8, 2, 8, 2], [4, 8, 2, 2, 9]], dtype=np.int16)
    counts = ref.label_counts(segs, labels)
    _, majority, entropy, summary = ref.label_posterior(counts, 4, labels, None)
    assert majority.tolist() == [0, 4, 8, 0, 2] == brute(segs, labels, np.zeros(5))[1]
    assert abs(entropy[3] - math.log(4)) < 1e-12 and abs(entropy[0] - math.log(2)) < 1e-12
    assert summary[:, 1].tolist() == [0, 0, 0]   # no fixed segmentation: O = 0


def test_identical_samples():
    labels = [5, 6]
    seg = np.array([5, 6, 0, 7, -5, 6], dtype=np.int16)
    counts = ref.label_counts([seg] * 3, labels)
    _, majority, entropy, summary = ref.label_posterior(counts, 3, labels, seg)
    assert majority.tolist() == [5, 6, 0, 0, 0, 6] and (entropy == 0).all()
    assert summary.tolist() == [[3, 3, 0], [6, 6, 0]]


# ---- C ABI ---------------------------------------------------------------------------------------------------------------
def _labels(*v):
    return (ctypes.c_int * len(v))(*v)


def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call: null pointers, n_labels outside 1..32, C < 1, V < 1, n < 1, duplicate labels (-1);
    label 0 in the list (-2)"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    f = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    lab = _labels(3, 7, 11)
    upd = lib.irs_label_counts_update
    assert upd(None, 2, 64, lab, 3, f, None) == -1
    assert upd(f, 2, 64, lab, 3, None, None) == -1
    assert upd(f, 2, 64, None, 3, f, None) == -1
    assert upd(f, 0, 64, lab, 3, f, None) == -1
    assert upd(f, 2, 0, lab, 3, f, None) == -1
    assert upd(f, 2, 64, lab, 0, f, None) == -1
    assert upd(f, 2, 64, _labels(*range(1, 34)), 33, f, None) == -1
    assert upd(f, 2, 64, _labels(3, 7, 3), 3, f, None) == -1
    assert upd(f, 2, 64, _labels(3, 40000), 2, f, None) == -1       # not an int16 value
    assert upd(f, 2, 64, _labels(3, 0, 5), 3, f, None) == -2
    post = lib.irs_label_posterior
    args = lambda **kw: [kw.get(k, d) for k, d in (('counts', f), ('labels', lab), ('L', 3), ('n', 4), ('V', 64),
                                                    ('fixed', None), ('prob', f), ('maj', f), ('ent', f), ('summ', f))]
    assert post(*args(counts=None), None) == -1
    for key in ('prob', 'maj', 'ent', 'summ', 'labels'):
        assert post(*args(**{key: None}), None) == -1, key
    assert post(*args(n=0), None) == -1
    assert post(*args(n=2 ** 31), None) == -1   # more segmentations than int32 counts can hold
    assert post(*args(V=0), None) == -1
    assert post(*args(L=0), None) == -1 and post(*args(L=33, labels=_labels(*range(1, 34))), None) == -1
    assert post(*args(labels=_labels(2, 2), L=2), None) == -1
    assert post(*args(labels=_labels(0, 2), L=2), None) == -2


# ---- custom ops ------------------------------------------------------------------------------------------------------------
def test_ops_schemas_fakes_and_cpu_refusal(built):
    import irsgmcmc_b200  # noqa: F401
    from irsgmcmc_b200 import ops, torch_ops
    from torch._subclasses.fake_tensor import FakeTensorMode
    assert {'label_counts_update', 'label_posterior'} <= set(torch_ops.OPS) and len(torch_ops.OPS) == 25
    upd, post = torch.ops.irsgmcmc.label_counts_update.default, torch.ops.irsgmcmc.label_posterior.default
    mutated = [a.name for a in upd._schema.arguments if a.alias_info is not None and a.alias_info.is_write]
    assert mutated == ['counts'] and str(upd._schema).endswith('-> ()')
    assert 'Tensor? seg_fixed' in str(post._schema) and '(Tensor, Tensor, Tensor, Tensor)' in str(post._schema)
    with FakeTensorMode():
        seg = torch.empty(3, 1, 6, 7, 8, device='cuda', dtype=torch.int16)
        counts = torch.empty(5, 6, 7, 8, device='cuda', dtype=torch.int32)
        assert torch.ops.irsgmcmc.label_counts_update(seg, [1, 2, 3, 4, 5], counts) is None
        prob, majority, entropy, summary = torch.ops.irsgmcmc.label_posterior(counts, 9, [1, 2, 3, 4, 5], seg[:1])
        assert prob.shape == (5, 6, 7, 8) and prob.dtype == torch.float32 and prob.device.type == 'cuda'
        assert majority.shape == (1, 1, 6, 7, 8) and majority.dtype == torch.int16
        assert entropy.shape == (1, 6, 7, 8) and entropy.dtype == torch.float32
        assert summary.shape == (5, 3) and summary.dtype == torch.int64
    seg, counts = torch.zeros(2, 1, 4, 4, 4, dtype=torch.int16), torch.zeros(2, 4, 4, 4, dtype=torch.int32)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        torch.ops.irsgmcmc.label_counts_update(seg, [1, 2], counts)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        torch.ops.irsgmcmc.label_posterior(counts, 2, [1, 2], None)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.label_counts_update(seg, [1, 2], counts)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.label_posterior(counts, 2, [1, 2])


# ---- the all-reduce over gloo --------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, counts, ns, out_dir):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from irsgmcmc_b200 import parallel
    local = counts[rank].clone()
    n, total = parallel.merge_label_counts(ns[rank], local)
    torch.save({'n': n, 'total': total, 'local_after': local}, os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


def test_merge_label_counts_world_size_2(tmp_path):
    g = torch.Generator().manual_seed(0)
    ns = (12, 5)
    counts = torch.stack([torch.randint(0, n + 1, (3, 5, 6, 7), generator=g, dtype=torch.int32) for n in ns])
    mp.spawn(_worker, args=(2, _free_port(), counts, ns, str(tmp_path)), nprocs=2, join=True)
    rs = [torch.load(tmp_path / f'r{r}.pt') for r in (0, 1)]
    for r, res in enumerate(rs):
        assert res['n'] == sum(ns)
        assert res['total'].dtype == torch.int32 and res['total'].shape == (3, 5, 6, 7)
        assert torch.equal(res['total'], counts.sum(0, dtype=torch.int32))
        assert torch.equal(res['local_after'], counts[r])   # the local counts stay as they are
    from irsgmcmc_b200 import parallel
    n, total = parallel.merge_label_counts(7, counts[0])     # no process group: a copy of the local counts
    assert n == 7 and torch.equal(total, counts[0]) and total.data_ptr() != counts[0].data_ptr()
