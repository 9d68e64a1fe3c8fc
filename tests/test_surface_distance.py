"""
Average surface distance on the device (irsgmcmc_b200/csrc/irs_surface.cu), what can be checked without a GPU:
 - the line arithmetic of the exact Euclidean distance transform (csrc/irs_edt.cuh) compiled for the host, against brute force
   and, composed over three axes, against scipy's exact transform;
 - the op's schema / fake implementation, refusal of CPU tensors, argument validation of the C ABI.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'irsgmcmc_b200', 'csrc')

HARNESS = r'''
#include <vector>
#include "irs_edt.cuh"
extern "C" void edt_sites(float* d, long long ds, int n, float w) { irs_edt_sites_1d(d, ds, n, w); }
extern "C" void edt_envelope(float* d, long long ds, int n, float w) {
    std::vector<int> v(n > 0 ? n : 1);
    std::vector<float> fv(n > 0 ? n : 1), zb(n > 0 ? n : 1);
    irs_edt_envelope_1d(d, ds, n, w, v.data(), fv.data(), zb.data(), 1);
}
'''

WEIGHTS = (1.0, 1.5 ** 2, 2.0 ** 2)


@pytest.fixture(scope='module')
def edt(tmp_path_factory):
    from irsgmcmc_b200 import build
    d = tmp_path_factory.mktemp('edt')
    src, out = d / 'edt_harness.cu', d / 'libedt_harness.so'
    src.write_text(HARNESS)
    cmd = [build._nvcc(), '-shared', '-O2', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-Xcompiler', '-fPIC',
           '-diag-suppress', '20013,550', '-I', CSRC, str(src), '-o', str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = ctypes.CDLL(str(out))
    for name in ('edt_sites', 'edt_envelope'):
        getattr(lib, name).argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_float]
        getattr(lib, name).restype = None
    return lib


def _run(fn, line, w):
    a = np.ascontiguousarray(line, dtype=np.float32).copy()
    fn(a.ctypes.data_as(ctypes.c_void_p), 1, a.size, w)
    return a


def _brute(f, w):
    """min_j f(j) + w (i - j)^2 in float64 (+inf when every f(j) is +inf)"""
    i = np.arange(f.size, dtype=np.float64)
    return (f.astype(np.float64)[None, :] + w * (i[:, None] - i[None, :]) ** 2).min(1)


def test_two_sweep_rows_against_brute_force(edt):
    rng = np.random.default_rng(0)
    patterns = [np.zeros(17, bool), np.eye(1, 17, 9, dtype=bool)[0], np.ones(17, bool), np.eye(1, 1, 0, dtype=bool)[0],
                np.zeros(1, bool), np.eye(1, 40, 0, dtype=bool)[0], np.eye(1, 40, 39, dtype=bool)[0]]
    patterns += [rng.random(n) < p for n in (2, 7, 33, 64, 250) for p in (0.02, 0.2, 0.7)]
    for sites in patterns:
        f = np.where(sites, 0.0, np.inf)
        for w in WEIGHTS:
            got = _run(edt.edt_sites, f, w)
            want = _brute(f, w)
            # w k^2 for these weights is exactly representable: no rounding at all
            assert np.array_equal(got, want.astype(np.float32)), (sites.astype(int), w)


def test_envelope_against_brute_force(edt):
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 9, 31, 64, 200):
        for w in WEIGHTS:
            for p_inf in (0.0, 0.5, 0.95, 1.0):
                # integer inputs: every value the pass forms is exact in fp32, so the result must be exact too
                f = np.where(rng.random(n) < p_inf, np.inf, rng.integers(0, 4 * n, n).astype(np.float64))
                got = _run(edt.edt_envelope, f, w)
                assert np.array_equal(got, _brute(f, w).astype(np.float32)), (n, w, p_inf)
                # arbitrary reals: fp32 rounding only
                f = np.where(rng.random(n) < p_inf, np.inf, (rng.random(n) * 3 * n).astype(np.float32).astype(np.float64))
                got = _run(edt.edt_envelope, f, w)
                want = _brute(f, w)
                fin = np.isfinite(want)
                assert np.array_equal(np.isfinite(got), fin)
                assert np.all(np.abs(got[fin] - want[fin]) <= 1e-6 * np.maximum(want[fin], 1.0)), (n, w, p_inf)


def test_separable_transform_matches_scipy(edt):
    """the three passes as irs_surface.cu chains them (sites along W, envelopes along H then D, weights spacing^2 with the
    spacing given as (x, y, z)) reproduce scipy's exact Euclidean distance transform"""
    from scipy import ndimage
    rng = np.random.default_rng(2)
    spacing = (1.0, 1.5, 2.0)
    for shape, p in (((9, 11, 13), 0.03), ((6, 5, 7), 0.3), ((5, 6, 4), 0.0), ((4, 4, 4), 1.0)):
        sites = rng.random(shape) < p
        if p == 0.0:
            sites[2, 3, 1] = True
        vol = np.where(sites, 0.0, np.inf).astype(np.float32)
        D, H, W = shape
        fp = vol.ctypes.data_as(ctypes.c_void_p).value
        for z in range(D):
            for y in range(H):
                edt.edt_sites(fp + 4 * (z * H + y) * W, 1, W, spacing[0] ** 2)
        for z in range(D):
            for x in range(W):
                edt.edt_envelope(fp + 4 * (z * H * W + x), W, H, spacing[1] ** 2)
        for y in range(H):
            for x in range(W):
                edt.edt_envelope(fp + 4 * (y * W + x), H * W, D, spacing[2] ** 2)
        want = ndimage.distance_transform_edt(~sites, sampling=spacing[::-1]) ** 2
        assert np.allclose(vol, want, rtol=1e-6, atol=0), shape


def test_fake_implementation_and_cpu_refusal(built):
    import irsgmcmc_b200  # noqa: F401
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        a = torch.empty(1, 1, 8, 9, 10, device='cuda', dtype=torch.int16)
        b = torch.empty(3, 1, 8, 9, 10, device='cuda', dtype=torch.int16)
        out = torch.ops.irsgmcmc.average_surface_distance(a, b, [1, 2, 5, 7], [1.0, 1.5, 2.0])
        assert out.shape == (3, 4) and out.dtype == torch.float64 and out.device.type == 'cuda'
    seg = torch.ones(2, 1, 6, 6, 6, dtype=torch.int16)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        torch.ops.irsgmcmc.average_surface_distance(seg, seg, [1], [1.0, 1.0, 1.0])
    from irsgmcmc_b200.utils import calc_ASD_GPU
    with pytest.raises(NotImplementedError):
        calc_ASD_GPU(2, seg, seg, {'a': 1}, (1.0, 1.0, 1.0))
    with pytest.raises(NotImplementedError):
        calc_ASD_GPU(2, seg.float(), seg.float(), {'a': 1}, (1.0, 1.0, 1.0))


def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call: label 0, label counts out of 1..32, non-positive or non-finite spacing"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    lab = (ctypes.c_int * 2)(1, 0)
    assert lib.irs_surface_boxes(fake, 0, fake, lab, 2, fake, 1, 8, 8, 8, None) == -2
    assert lib.irs_surface_boxes(fake, 0, fake, lab, 0, fake, 1, 8, 8, 8, None) == -1
    assert lib.irs_surface_boxes(fake, 0, fake, (ctypes.c_int * 33)(*range(1, 34)), 33, fake, 1, 8, 8, 8, None) == -1
    boxes = (ctypes.c_int * 8)(0, 0, 0, 7, 7, 7, 5, 5)
    ok = (ctypes.c_int * 1)(3)

    def asd(labels, spacing, begin=0, end=1, ws_floats=1 << 20):
        return lib.irs_average_surface_distance(fake, 0, fake, labels, 1, boxes, _lib.host_floats(spacing), begin, end, fake,
                                                ws_floats, fake, fake, fake, 1, 8, 8, 8, None)
    assert asd((ctypes.c_int * 1)(0), [1.0, 1.0, 1.0]) == -2
    for sp in ([0.0, 1.0, 1.0], [1.0, -1.0, 1.0], [1.0, 1.0, float('nan')], [1.0, float('inf'), 1.0]):
        assert asd(ok, sp) == -1, sp
    assert asd(ok, [1.0, 1.0, 1.0], begin=0, end=2) == -1                 # past the (C, n_labels) table
    assert asd(ok, [1.0, 1.0, 1.0], ws_floats=2 * 8 ** 3 - 1) == -3      # 2 floats per box voxel
