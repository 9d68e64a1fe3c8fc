"""
Hausdorff distance and its percentile on the device (irsgmcmc_b200/csrc/irs_surface.cu, irs_select.cuh), what can be checked
without a GPU:
 - the selection arithmetic (csrc/irs_select.cuh: percentile ranks, radix digit step, numpy's interpolation) compiled for the
   host, bit for bit against np.percentile of the square-rooted keys;
 - the host restatement utils.calc_HD_host against brute force over all pairs of contour voxels;
 - argument validation of the C ABI, the op's fake implementation and the refusal of CPU tensors.
"""
import ctypes
import subprocess

import numpy as np
import pytest
import torch

from tests.test_surface_distance import CSRC

HARNESS = r'''
#include "irs_select.cuh"
extern "C" double percentile_of_keys(const float* keys, unsigned int n, double q) { return irs_percentile_of_keys(keys, n, q); }
'''

QS = (0.0, 50.0, 95.0, 99.0, 100.0)


@pytest.fixture(scope='module')
def sel(tmp_path_factory):
    from irsgmcmc_b200 import build
    d = tmp_path_factory.mktemp('select')
    src, out = d / 'select_harness.cu', d / 'libselect_harness.so'
    src.write_text(HARNESS)
    cmd = [build._nvcc(), '-shared', '-O2', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-Xcompiler', '-fPIC',
           '-diag-suppress', '20013,550', '-I', CSRC, str(src), '-o', str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = ctypes.CDLL(str(out))
    lib.percentile_of_keys.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_double]
    lib.percentile_of_keys.restype = ctypes.c_double
    return lib


def _check(sel, keys, q):
    keys = np.ascontiguousarray(keys, dtype=np.float32)
    got = sel.percentile_of_keys(keys.ctypes.data_as(ctypes.c_void_p), keys.size, q)
    want = float(np.percentile(np.sqrt(keys.astype(np.float64)), q))
    assert got == want, (keys.size, q, got, want)   # bit for bit, 0 == -0 aside (no negative keys)


def test_selection_matches_numpy_percentile(sel):
    rng = np.random.default_rng(0)
    lists = [np.array([7.0]), np.array([0.0]), np.array([2.0, 5.0]), np.array([5.0, 2.0]), np.zeros(100), np.full(37, 9.0),
             np.array([0.0, 0.0, 1.0]), np.array([3.0, 3.0, 3.0, 1e5])]
    for n in (3, 10, 101, 1000, 4099, 60000):
        lists.append(rng.integers(0, 3 * 60 ** 2, n).astype(np.float32))                 # integer squared distances
        lists.append(rng.integers(0, 4, n).astype(np.float32))                           # heavy ties
        lists.append(np.where(rng.random(n) < 0.9, 0.0, rng.integers(1, 50, n)).astype(np.float32))   # mostly on the contour
        lists.append((rng.random(n) * 1e4).astype(np.float32))                           # non-dyadic spacings: any fp32
        lists.append((rng.integers(0, 2000, n) * 2.25 + rng.integers(0, 40, n) * 4.0).astype(np.float32))   # spacing (1.5, 2)
    for keys in lists:
        for q in QS + tuple(rng.random(3) * 100.0):
            _check(sel, keys, float(q))


def test_selection_ranks_at_exact_and_near_boundaries(sel):
    """q where (n - 1) q / 100 lands on an integer, just below one and at g = 0.5, where numpy switches its formula"""
    rng = np.random.default_rng(1)
    for n in (2, 3, 5, 21, 201):
        keys = rng.integers(0, 500, n).astype(np.float32)
        for q in (100.0 * k / (n - 1) for k in range(n)):
            _check(sel, keys, q)
            _check(sel, keys, np.nextafter(q, 0.0))
        for k in range(n - 1):
            _check(sel, keys, 100.0 * (k + 0.5) / (n - 1))


def _brute_hd(a, b, spacing, q):
    from irsgmcmc_b200.utils.util import _label_contour
    ca, cb = _label_contour(a), _label_contour(b)
    pa = np.argwhere(ca) * np.array(spacing[::-1])
    pb = np.argwhere(cb) * np.array(spacing[::-1])
    dist = np.sqrt(((pa[:, None, :] - pb[None, :, :]) ** 2).sum(-1))
    d_ab, d_ba = dist.min(1), dist.min(0)
    return max(d_ab.max(), d_ba.max()), max(np.percentile(d_ab, q), np.percentile(d_ba, q))


@pytest.mark.parametrize('spacing', [(1.0, 1.0, 1.0), (1.0, 1.5, 2.0), (0.7, 1.3, 0.9)])
def test_calc_HD_host_against_brute_force(spacing):
    from irsgmcmc_b200.utils import calc_HD_host
    n = 14
    zz, yy, xx = np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing='ij')
    a = (zz - 6.0) ** 2 + (yy - 7.0) ** 2 + (xx - 6.5) ** 2 <= 16.0
    b = (zz - 7.0) ** 2 / 1.5 + (yy - 6.0) ** 2 + (xx - 7.5) ** 2 <= 14.0
    c = np.zeros_like(a)
    c[1:3, 1:4, 2:4] = True
    c[10:13, 11:13, 9:12] = True                       # two far-apart components
    edge = np.zeros_like(a)
    edge[:, :5, :] = True                              # touches five faces of the volume
    for x, y in ((a, b), (a, c), (c, b), (edge, a), (a, a)):
        for q in QS + (37.5,):
            hd, hd_q = calc_HD_host(x, y, spacing, q)
            want_hd, want_q = _brute_hd(x, y, spacing, q)
            assert abs(hd - want_hd) <= 1e-12 * max(want_hd, 1.0) and abs(hd_q - want_q) <= 1e-12 * max(want_q, 1.0)
    assert calc_HD_host(a, a, spacing) == (0.0, 0.0)
    assert calc_HD_host(a, np.zeros_like(a), spacing) == (float('inf'), float('inf'))
    # q = 100 is the Hausdorff distance itself
    hd, hd_100 = calc_HD_host(a, c, spacing, 100.0)
    assert hd == hd_100


def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call: percentile outside [0, 100] or NaN, label 0, bad spacing, a pair range past the table,
    a workspace one float short of 2 * box voxels + |A| + |B|, missing outputs"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    boxes = (ctypes.c_int * 8)(0, 0, 0, 7, 7, 7, 5, 6)
    ok = (ctypes.c_int * 1)(3)

    def sd(labels=ok, spacing=(1.0, 1.0, 1.0), q=95.0, begin=0, end=1, ws_floats=1 << 20, hd=fake, hd_q=fake):
        return lib.irs_surface_distances(fake, 0, fake, labels, 1, boxes, _lib.host_floats(spacing), q, begin, end, fake,
                                         ws_floats, fake, fake, fake, hd, hd_q, 1, 8, 8, 8, None)
    for q in (-1.0, 100.5, float('nan'), float('inf'), -0.0001):
        assert sd(q=q) == -1, q
    assert sd(labels=(ctypes.c_int * 1)(0)) == -2
    for sp in ([0.0, 1.0, 1.0], [1.0, -1.0, 1.0], [1.0, 1.0, float('nan')], [1.0, float('inf'), 1.0]):
        assert sd(spacing=sp) == -1, sp
    assert sd(begin=0, end=2) == -1                              # past the (C, n_labels) table
    assert sd(ws_floats=2 * 8 ** 3 + 5 + 6 - 1) == -3             # 2 floats per box voxel + |A| + |B|
    assert sd(hd=None) == -1 and sd(hd_q=None) == -1
    assert _lib.SD_COUNTERS == 3 * _lib.ASD_MAX_BOXES


def test_fake_implementation_and_cpu_refusal(built):
    import irsgmcmc_b200  # noqa: F401
    from torch._subclasses.fake_tensor import FakeTensorMode
    op = torch.ops.irsgmcmc.surface_distances
    assert str(op.default._schema).startswith('irsgmcmc::surface_distances(')
    assert str(op.default._schema).endswith('-> (Tensor, Tensor, Tensor)')
    with FakeTensorMode():
        a = torch.empty(1, 1, 8, 9, 10, device='cuda', dtype=torch.int16)
        b = torch.empty(3, 1, 8, 9, 10, device='cuda', dtype=torch.int16)
        outs = op(a, b, [1, 2, 5, 7], [1.0, 1.5, 2.0], 99.0)
        assert len(outs) == 3
        for out in outs:
            assert out.shape == (3, 4) and out.dtype == torch.float64 and out.device.type == 'cuda'
    seg = torch.ones(2, 1, 6, 6, 6, dtype=torch.int16)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        op(seg, seg, [1], [1.0, 1.0, 1.0], 95.0)
    from irsgmcmc_b200.utils import calc_HD_GPU
    with pytest.raises(NotImplementedError):
        calc_HD_GPU(2, seg, seg, {'a': 1}, (1.0, 1.0, 1.0))
    with pytest.raises(NotImplementedError):
        calc_HD_GPU(2, seg.float(), seg.float(), {'a': 1}, (1.0, 1.0, 1.0))
