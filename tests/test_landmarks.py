"""
Landmark registration error and landmark posterior (irsgmcmc_b200/csrc/irs_landmark.cuh, irs_landmark.cu), what can be checked
without a GPU:
 - the numpy restatement (tests/helpers/landmark_ref.py, utils.calc_TRE_host) against plain loops;
 - the kernels' per-landmark arithmetic (csrc/irs_landmark.cuh) compiled for the host by this module: predicted positions and TREs bit-equal
   to the restatement, the accumulators bit-equal to its Welford recurrence, eigenvalues and Mahalanobis distances against
   np.linalg within 1e-9 relative, NaN rows for one sample and +inf for a singular covariance;
 - argument validation of the C ABI, the op schemas, fake implementations and the refusal of CPU tensors;
 - parallel.merge_landmark_moments over a world-size-2 gloo group against one pooled accumulation;
 - make_landmarks: phi(q) reproduces p through an independent warp of coordinate ramps; make_pair is unchanged;
 - the host summaries (coverage, rank correlation) and the VTK writer.
"""
import ctypes
import hashlib
import os
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.helpers import landmark_ref as ref

P_ = lambda a: a.ctypes.data_as(ctypes.c_void_p)
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'irsgmcmc_b200', 'csrc')

# what landmark_map_kernel, landmark_update_kernel and landmark_posterior_kernel run per thread, in plain loops on the CPU
HARNESS = r'''
#include "irs_landmark.cuh"
extern "C" {
// pred (C,P,3), tre (C,P) for T (C,3,D,H,W), p / q (P,3), spacing (3)
void emul_landmark_map(const float* T, const double* p, const double* q, const double* s, double* pred, double* tre, int C,
                       int P, int D, int H, int W) {
    const size_t V = (size_t)D * H * W;
    for (int c = 0; c < C; ++c)
        for (int i = 0; i < P; ++i) {
            double* m = pred + 3 * ((size_t)c * P + i);
            irs_landmark_predict(T + (size_t)c * 3 * V, D, H, W, p + 3 * i, m);
            tre[(size_t)c * P + i] = irs_landmark_tre(m, q + 3 * i, s);
        }
}
// the accumulators (P, 11) after the samples pred (N,P,3) / tre (N,P) in order
void emul_landmark_accumulate(const double* pred, const double* tre, int N, int P, double* acc) {
    for (int k = 0; k < N; ++k)
        for (int i = 0; i < P; ++i)
            irs_landmark_welford(acc + (size_t)IRS_LANDMARK_ACC * i, (double)(k + 1), pred + 3 * ((size_t)k * P + i),
                                 tre[(size_t)k * P + i]);
}
void emul_landmark_finish(const double* acc, double n, const double* q, const double* s, double* out, int P) {
    for (int i = 0; i < P; ++i)
        irs_landmark_finish(acc + (size_t)IRS_LANDMARK_ACC * i, n, q + 3 * i, s, out + (size_t)IRS_LANDMARK_COLS * i);
}
// eigenvalues (descending) and r^T S^-1 r of n symmetric 3x3 (xx, xy, xz, yy, yz, zz)
void emul_sym3(const double* S, const double* r, double* ev, double* d2, int n) {
    for (int k = 0; k < n; ++k) {
        irs_sym3_eigen(S + 6 * k, ev + 3 * k);
        d2[k] = irs_sym3_mahalanobis2(S + 6 * k, r + 3 * k);
    }
}
}
'''


@pytest.fixture(scope='module')
def emul(tmp_path_factory):
    """irs_landmark.cuh built for the host with nvcc's host compiler (no FMA contraction on x86-64 without -mfma)"""
    from irsgmcmc_b200 import build
    d = tmp_path_factory.mktemp('landmark')
    src, out = d / 'landmark_harness.cu', d / 'liblandmark_harness.so'
    src.write_text(HARNESS)
    cmd = [build._nvcc(), '-shared', '-O2', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-Xcompiler', '-fPIC',
           '-diag-suppress', '20013,550', '-I', CSRC, str(src), '-o', str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return ctypes.CDLL(str(out))


def _field(C, D, H, W, seed, scale=0.3):
    """an asymmetric fp32 transformation: identity grid + different random offsets per channel and axis"""
    rng = np.random.default_rng(seed)
    lin = [np.linspace(-1, 1, n, dtype=np.float32) for n in (W, H, D)]
    z, y, x = np.meshgrid(lin[2], lin[1], lin[0], indexing='ij')
    base = np.stack((x, y, z)).astype(np.float32)
    T = base[None] + (scale * rng.standard_normal((C, 3, D, H, W))).astype(np.float32)
    T[:, 0] += np.float32(0.05) * np.arange(W, dtype=np.float32)   # channel- and axis-specific drifts
    T[:, 2] -= np.float32(0.02) * np.arange(D, dtype=np.float32)[:, None, None]
    return np.ascontiguousarray(T)


def _landmarks(D, H, W, P, seed):
    """off-grid points, nodes, faces (0 and n - 1 on each axis) and the eight corners"""
    rng = np.random.default_rng(seed)
    hi = np.array([W - 1, H - 1, D - 1], dtype=np.float64)
    pts = [rng.random((P, 3)) * hi, rng.integers(0, hi + 1, (6, 3)).astype(np.float64)]
    for a in range(3):
        for v in (0.0, hi[a]):
            x = rng.random(3) * hi
            x[a] = v
            pts.append(x[None])
    pts.append(np.array([[i * hi[0], j * hi[1], k * hi[2]] for i in (0, 1) for j in (0, 1) for k in (0, 1)]))
    p = np.ascontiguousarray(np.concatenate(pts))
    q = np.ascontiguousarray(p + rng.standard_normal(p.shape) * 2.0)
    return p, q


def _emul_map(emul, T, p, q, s):
    C, _, D, H, W = T.shape
    P = p.shape[0]
    pred, tre = np.empty((C, P, 3)), np.empty((C, P))
    emul.emul_landmark_map(P_(T), P_(p), P_(q), P_(np.asarray(s, dtype=np.float64)), P_(pred), P_(tre), C, P, D, H, W)
    return pred, tre


# ---- the restatement against loops -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dims', [(5, 6, 7), (4, 4, 4), (2, 3, 9)])
def test_restatement_matches_loops(dims):
    D, H, W = dims
    T = _field(3, D, H, W, 0)
    p, q = _landmarks(D, H, W, 20, 1)
    s = (0.7, 1.3, 2.1)
    pred = ref.predict(T, p)
    assert np.array_equal(pred, ref.predict_loops(T, p))
    assert np.array_equal(ref.tre(pred, q, s), ref.tre_loops(pred, q, s))
    from irsgmcmc_b200.utils import calc_TRE_host
    assert np.array_equal(calc_TRE_host(torch.from_numpy(T), torch.from_numpy(p), torch.from_numpy(q), s), ref.tre(pred, q, s))
    # at a node the prediction is T there in voxel units, and the identity grid gives back the point itself
    acc = ref.accumulate(pred, ref.tre(pred, q, s))
    tp = ref.two_pass(pred, ref.tre(pred, q, s))
    assert np.allclose(acc, tp, rtol=1e-12, atol=1e-12 * np.abs(tp).max())


def test_identity_transformation_maps_landmarks_to_themselves():
    D, H, W = 5, 6, 7
    T = _field(1, D, H, W, 0, scale=0.0)
    T[:, 0] -= np.float32(0.05) * np.arange(W, dtype=np.float32)
    T[:, 2] += np.float32(0.02) * np.arange(D, dtype=np.float32)[:, None, None]
    nodes = np.array([[0, 0, 0], [6, 5, 4], [3, 2, 1]], dtype=np.float64)
    assert np.allclose(ref.predict(T, nodes)[0], nodes, atol=2e-6)


# ---- the device arithmetic built for the host ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('dims,C', [((5, 6, 7), 3), ((9, 4, 2), 1), ((8, 8, 8), 4)])
def test_emulated_map_is_bit_equal_to_restatement(emul, dims, C):
    D, H, W = dims
    T = _field(C, D, H, W, 2)
    p, q = _landmarks(D, H, W, 33, 3)
    s = (0.9, 1.1, 2.5)
    pred, tre = _emul_map(emul, T, p, q, s)
    want = ref.predict(T, p)
    assert np.array_equal(pred, want)
    assert np.array_equal(tre, ref.tre(want, q, s))
    # a swap of the channels or axes would not be bit-equal: the field is asymmetric
    assert not np.array_equal(pred, ref.predict(np.ascontiguousarray(T[:, ::-1]), p))


def test_emulated_map_clamps_every_coordinate(emul):
    """NaN, +-inf and far-outside coordinates read the nearest edge cell (the kernel's clamp) and never outside T"""
    T = _field(2, 3, 4, 5, 4)
    p = np.array([[np.nan, 1.0, 1.0], [np.inf, -np.inf, 0.5], [-7.0, 100.0, 2.0], [4.0, 3.0, 2.0]])
    q = np.zeros_like(p)
    pred, _ = _emul_map(emul, T, p, q, (1.0, 1.0, 1.0))
    assert np.isfinite(pred[:, 2:]).all()
    assert np.array_equal(pred[:, 2:], ref.predict(T, p[2:]))


def test_emulated_accumulators_and_finish(emul):
    rng = np.random.default_rng(5)
    N, P = 37, 19
    pred = rng.standard_normal((N, P, 3)) * np.array([1.0, 2.0, 0.5]) + 20.0
    pred[:, 0] = pred[:1, 0]                                  # identical samples: zero covariance
    tre = np.abs(rng.standard_normal((N, P))) * 3.0
    acc = np.zeros((P, 11))
    emul.emul_landmark_accumulate(P_(np.ascontiguousarray(pred)), P_(np.ascontiguousarray(tre)), N, P, P_(acc))
    assert np.array_equal(acc, ref.accumulate(pred, tre))
    tp = ref.two_pass(pred, tre)
    assert np.allclose(acc, tp, rtol=1e-12, atol=1e-12 * np.abs(tp).max())
    q = np.ascontiguousarray(pred.mean(0) + rng.standard_normal((P, 3)))
    s = np.array([0.8, 1.2, 1.5])
    for n, a in ((N, acc), (1, ref.accumulate(pred[:1], tre[:1]))):
        out = np.empty((P, 16))
        emul.emul_landmark_finish(P_(a), ctypes.c_double(n), P_(q), P_(s), P_(out), P)
        want = ref.posterior(a, n, q, s)
        if n == 1:
            assert np.isnan(out[:, 5:]).all() and np.isnan(want[:, 5:]).all()
            assert np.allclose(out[:, :5], want[:, :5], rtol=1e-15, atol=0)
            continue
        assert np.isinf(out[0, 15]) and np.isinf(want[0, 15])         # the zero covariance of landmark 0
        assert (out[0, 12:15] == 0).all() and (out[0, 6:12] == 0).all()
        scale = np.abs(want[1:, 6:12]).max(1, keepdims=True)
        assert np.allclose(out[1:, 6:12], want[1:, 6:12], rtol=1e-12, atol=0)
        assert (np.abs(out[1:, 12:15] - want[1:, 12:15]) <= 1e-9 * np.sqrt(scale)).all()
        assert np.allclose(out[1:, 15], want[1:, 15], rtol=1e-9, atol=0)
        assert np.allclose(out[:, :6], want[:, :6], rtol=1e-14, atol=0)


def _sym6(S):
    return np.array([S[0, 0], S[0, 1], S[0, 2], S[1, 1], S[1, 2], S[2, 2]])


def _rotation(rng):
    Q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    return Q


def test_emulated_eigenvalues_and_mahalanobis(emul):
    """well separated, nearly repeated (pairs and triples, from 1e-3 down to 1e-12 relative), repeated, diagonal and scaled
    spectra in random orientations: eigenvalues within 1e-9 of the largest, d^2 within 1e-9 relative; exactly singular
    matrices give +inf"""
    rng = np.random.default_rng(6)
    spectra = [(3.0, 2.0, 1.0), (1.0, 1.0, 1.0), (5.0, 1.0, 1.0), (5.0, 5.0, 1.0), (2.0, 1e-6, 1e-7)]
    for rel in (1e-3, 1e-6, 1e-9, 1e-12):
        spectra += [(3.0, 1.0 + rel, 1.0), (3.0 + rel, 3.0, 1.0), (2.0 + 2 * rel, 2.0 + rel, 2.0)]
    mats, rs = [], []
    for lam in spectra:
        for scale in (1.0, 1e-4, 1e4):
            for _ in range(4):
                Q = _rotation(rng)
                S = Q @ np.diag(np.array(lam) * scale) @ Q.T
                mats.append(_sym6((S + S.T) / 2))
                rs.append(rng.standard_normal(3) * np.sqrt(scale))
        mats.append(_sym6(np.diag(lam)))                  # diagonal: sorted as it is
        rs.append(rng.standard_normal(3))
    S6, R = np.ascontiguousarray(mats), np.ascontiguousarray(rs)
    ev, d2 = np.empty((len(S6), 3)), np.empty(len(S6))
    emul.emul_sym3(P_(S6), P_(R), P_(ev), P_(d2), len(S6))
    for k in range(len(S6)):
        S = S6[k][[0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(3, 3)
        want = np.linalg.eigvalsh(S)[::-1]
        assert np.all(np.abs(ev[k] - want) <= 1e-9 * np.abs(want).max()), (k, ev[k], want)
        assert ev[k][0] >= ev[k][1] >= ev[k][2]
        if want[-1] > 1e-6 * want[0]:   # well enough conditioned for a 1e-9 check of the solve
            wd = float(R[k] @ np.linalg.solve(S, R[k]))
            assert abs(d2[k] - wd) <= 1e-9 * abs(wd), (k, d2[k], wd)
    singular = np.ascontiguousarray([_sym6(np.diag([2.0, 1.0, 0.0])), _sym6(np.zeros((3, 3))),
                                     _sym6(np.array([[1.0, 1.0, 0.0], [1.0, 1.0, 0.0], [0.0, 0.0, 3.0]])),
                                     _sym6(np.diag([-1.0, 2.0, 3.0]))])
    ev, d2 = np.empty((4, 3)), np.empty(4)
    emul.emul_sym3(P_(singular), P_(np.ones((4, 3))), P_(ev), P_(d2), 4)
    assert np.isinf(d2).all() and (d2 > 0).all()
    assert np.allclose(ev[2], [3.0, 2.0, 0.0], atol=1e-15)


# ---- the C ABI, the ops and their schemas --------------------------------------------------------------------------------------
def test_abi_argument_validation_without_gpu(built):
    """rejected before any CUDA call: null pointers, C < 1, P < 1, a dimension < 2, bad spacing, counts outside [0, 2^53]"""
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    f = ctypes.c_void_p(256)   # never dereferenced: every call below is refused first
    sp = lambda *v: (ctypes.c_double * 3)(*v)
    names = ('T', 'C', 'D', 'H', 'W', 'p', 'q', 'P', 's', 'pred', 'tre')
    good = dict(T=f, C=2, D=4, H=5, W=6, p=f, q=f, P=3, s=sp(1.0, 1.0, 1.0), pred=f, tre=f)
    mp_ = lambda **kw: lib.irs_landmark_map(*[kw.get(k, good[k]) for k in names], None)
    for key in ('T', 'p', 'q', 's', 'pred', 'tre'):
        assert mp_(**{key: None}) == -1, key
    assert mp_(C=0) == -1 and mp_(P=0) == -1 and mp_(D=1) == -1 and mp_(H=1) == -1 and mp_(W=1) == -1
    for bad in ((0.0, 1.0, 1.0), (1.0, -1.0, 1.0), (1.0, 1.0, float('nan')), (float('inf'), 1.0, 1.0)):
        assert mp_(s=sp(*bad)) == -1, bad
    unames = ('pred', 'tre', 'C', 'P', 'count', 'acc', 'stats')
    ugood = dict(pred=f, tre=f, C=2, P=3, count=0.0, acc=f, stats=f)
    up = lambda **kw: lib.irs_landmark_update(*[kw.get(k, ugood[k]) for k in unames], None)
    for key in ('pred', 'tre', 'acc', 'stats'):
        assert up(**{key: None}) == -1, key
    assert up(C=0) == -1 and up(P=0) == -1
    assert up(count=-1.0) == -1 and up(count=float('nan')) == -1 and up(count=0.5) == -1 and up(count=2.0 ** 53 - 1) == -1
    pnames = ('acc', 'q', 'P', 'n', 's', 'out')
    pgood = dict(acc=f, q=f, P=3, n=2, s=sp(1.0, 2.0, 3.0), out=f)
    po = lambda **kw: lib.irs_landmark_posterior(*[kw.get(k, pgood[k]) for k in pnames], None)
    for key in ('acc', 'q', 's', 'out'):
        assert po(**{key: None}) == -1, key
    assert po(P=0) == -1 and po(n=0) == -1 and po(n=2 ** 53 + 2) == -1 and po(s=sp(1.0, 0.0, 1.0)) == -1
    assert _lib.LANDMARK_ACC == 11 and _lib.LANDMARK_COLS == 16


def test_ops_check_landmarks_and_refuse_cpu_tensors(built):
    from irsgmcmc_b200 import ops
    from irsgmcmc_b200.utils import calc_TRE_GPU
    p, q = torch.tensor([[1.0, 2.0, 3.0]]), torch.tensor([[0.0, 0.0, 0.0]])
    dims = (4, 5, 6)
    ops.check_landmarks(p, q, dims)
    for bad in ([[5.01, 1.0, 1.0]], [[1.0, 4.5, 1.0]], [[1.0, 1.0, 3.5]], [[-1e-9, 1.0, 1.0]], [[float('nan'), 1.0, 1.0]]):
        with pytest.raises(ValueError):
            ops.check_landmarks(torch.tensor(bad), q, dims)
    with pytest.raises(ValueError):
        ops.check_landmarks(p, torch.tensor([[float('inf'), 0.0, 0.0]]), dims)
    with pytest.raises(ValueError):
        ops.check_landmarks(p, torch.zeros(2, 3), dims)
    with pytest.raises(ValueError):
        ops.landmark_spacing((1.0, 0.0, 1.0))
    T = torch.zeros(1, 3, 4, 5, 6)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.landmark_map(T, p, q, (1.0, 1.0, 1.0))
    acc = torch.zeros(1, 11, dtype=torch.float64)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.landmark_update(torch.zeros(1, 1, 3, dtype=torch.float64), torch.zeros(1, 1, dtype=torch.float64), 0, acc)
    with pytest.raises(RuntimeError, match='CUDA'):
        ops.landmark_posterior(acc, 1, q, (1.0, 1.0, 1.0))
    with pytest.raises(NotImplementedError):
        calc_TRE_GPU(T, p, q, (1.0, 1.0, 1.0))


def test_op_schemas_and_fakes(built):
    import irsgmcmc_b200  # noqa: F401
    from irsgmcmc_b200 import torch_ops
    from torch._subclasses.fake_tensor import FakeTensorMode
    ns = torch.ops.irsgmcmc
    assert str(ns.landmark_map.default._schema) == ('irsgmcmc::landmark_map(Tensor T, Tensor fixed_landmarks, Tensor '
                                                    'moving_landmarks, float[] spacing) -> (Tensor, Tensor)')
    assert str(ns.landmark_update.default._schema) == ('irsgmcmc::landmark_update(Tensor pred, Tensor tre, SymInt count_before, '
                                                       'Tensor(a3!) acc) -> Tensor')
    assert str(ns.landmark_posterior.default._schema) == ('irsgmcmc::landmark_posterior(Tensor acc, SymInt n, Tensor '
                                                          'moving_landmarks, float[] spacing) -> Tensor')
    assert len(torch_ops.OPS) == 25 and not any(name.startswith('landmark') for name in torch_ops.OPS)
    with FakeTensorMode():
        T = torch.empty(5, 3, 8, 9, 10, device='cuda')
        p = torch.empty(7, 3, device='cuda', dtype=torch.float64)
        pred, tre = ns.landmark_map(T, p, p, [1.0, 1.0, 2.0])
        assert pred.shape == (5, 7, 3) and tre.shape == (5, 7) and pred.dtype == tre.dtype == torch.float64
        acc = torch.empty(7, 11, device='cuda', dtype=torch.float64)
        stats = ns.landmark_update(pred, tre, 10, acc)
        assert stats.shape == (5, 3) and stats.dtype == torch.float64 and stats.device.type == 'cuda'
        out = ns.landmark_posterior(acc, 15, p, [1.0, 1.0, 2.0])
        assert out.shape == (7, 16) and out.dtype == torch.float64
    T = torch.zeros(1, 3, 4, 4, 4)
    with pytest.raises(NotImplementedError, match="'CPU' backend"):
        ns.landmark_map(T, torch.zeros(1, 3, dtype=torch.float64), torch.zeros(1, 3, dtype=torch.float64), [1.0, 1.0, 1.0])


# ---- the merge over gloo ------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, parts, out_dir):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from irsgmcmc_b200 import parallel
    pred, tre = parts[rank]
    acc = torch.from_numpy(ref.accumulate(pred, tre)) if len(tre) else torch.zeros(pred.shape[1], 11, dtype=torch.float64)
    before = acc.clone()
    n, merged = parallel.merge_landmark_moments(len(tre), acc)
    torch.save({'n': n, 'acc': merged, 'kept': torch.equal(acc, before)}, os.path.join(out_dir, f'r{rank}.pt'))
    dist.destroy_process_group()


@pytest.mark.parametrize('split', [9, 0])
def test_merge_landmark_moments_world_size_2(tmp_path, split):
    rng = np.random.default_rng(7)
    N, P = 23, 6
    pred = rng.standard_normal((N, P, 3)) * 3.0 + 40.0
    tre = np.abs(rng.standard_normal((N, P))) + 1.0
    parts = [(pred[:split], tre[:split]), (pred[split:], tre[split:])]
    mp.spawn(_worker, args=(2, _free_port(), parts, str(tmp_path)), nprocs=2, join=True)
    want = ref.two_pass(pred, tre)
    for r in (0, 1):
        res = torch.load(tmp_path / f'r{r}.pt')
        assert res['n'] == N and res['kept']
        got = res['acc'].numpy()
        assert np.allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max())
    from irsgmcmc_b200 import parallel
    acc = torch.from_numpy(ref.accumulate(pred, tre))
    n, same = parallel.merge_landmark_moments(N, acc)   # no process group: a copy of the local accumulators
    assert n == N and torch.equal(same, acc) and same.data_ptr() != acc.data_ptr()


# ---- synthetic ground truth ------------------------------------------------------------------------------------------------------
def _digest(*dicts):
    h = hashlib.sha256()
    for d in dicts:
        for k in sorted(d):
            h.update(k.encode())
            h.update(d[k].contiguous().numpy().tobytes())
    return h.hexdigest()


def test_make_pair_unchanged():
    """make_pair, which the golden tests and the benchmark depend on, gives the bits it gave before make_landmarks shared its
    velocity draw"""
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    assert _digest(*make_pair(16)) == '5517517f06c2cbc04cb1f975e6aaf27f4c5566a952641800eb8eb961cbfa0084'
    assert _digest(*make_pair(24, seed=5, max_velocity=2.0)) == '745b3bf967ab51b839ceb04e42e639736cda64946f2248a240c4fcedd51209b5'


def test_make_landmarks_correspondence():
    """phi(q) = p, checked through F.grid_sample of the fixed voxel-coordinate ramps with make_pair's grid (the warp that builds
    the moving image): what the moving image holds at q is what the fixed image holds at p"""
    import torch.nn.functional as F
    from irsgmcmc_b200.data_loader import synthetic
    n, seed = 32, 3
    p, q = synthetic.make_landmarks(n, seed=seed, no_landmarks=120)
    assert p.shape == q.shape == (120, 3) and p.dtype == q.dtype == torch.float64
    assert (q == q.round()).all() and (p >= 1.0).all() and (p <= n - 2.0).all()
    assert len({tuple(x) for x in q.tolist()}) == 120
    _, moving, _ = synthetic.make_pair(n, seed=seed)
    qi = q.long()
    assert moving['mask'][0, 0, qi[:, 2], qi[:, 1], qi[:, 0]].all()
    _, _, v = synthetic._texture_and_velocity(n, seed, 3.0, 'cpu')
    grid = synthetic._exp_velocity(v)
    ramp = torch.arange(n, dtype=torch.float32)
    ramps = torch.stack((ramp.view(1, 1, n).expand(n, n, n), ramp.view(1, n, 1).expand(n, n, n),
                         ramp.view(n, 1, 1).expand(n, n, n))).unsqueeze(0)
    warped = F.grid_sample(ramps, grid, mode='bilinear', padding_mode='border', align_corners=True)[0]
    at_q = warped[:, qi[:, 2], qi[:, 1], qi[:, 0]].T.double()
    assert torch.allclose(at_q, p, atol=1e-4), (at_q - p).abs().max()
    p2, q2 = synthetic.make_landmarks(n, seed=seed, no_landmarks=120)
    assert torch.equal(p, p2) and torch.equal(q, q2)
    with pytest.raises(ValueError):
        synthetic.make_landmarks(8, no_landmarks=10 ** 6)


# ---- host summaries and the writer --------------------------------------------------------------------------------------------------
def test_posterior_summary_and_vtk_round_trip(tmp_path):
    from scipy import stats
    from irsgmcmc_b200.logger import load_landmarks_from_disk, save_landmarks_to_disk
    from irsgmcmc_b200.utils import landmark_posterior_summary
    rng = np.random.default_rng(8)
    P = 40
    table = np.zeros((P, 16))
    table[:, :3] = rng.random((P, 3)) * 10
    table[:, 3] = rng.random(P) * 4
    table[:, 4] = table[:, 3] + 0.5
    table[:, 6:12] = np.array([2.0, 0.1, 0.0, 1.0, 0.0, 3.0]) * (1 + rng.random((P, 1)))
    table[:, 15] = np.linspace(0.0, 10.0, P)
    table[-1, 15] = np.inf
    p = rng.random((P, 3)) * 10
    q = p + 1.0
    s = (1.0, 2.0, 0.5)
    out = landmark_posterior_summary(torch.from_numpy(table), p, q, s)
    for level in (50, 90, 95):
        assert out['coverage'][level] == np.mean(table[:, 15] <= stats.chi2.ppf(level / 100, 3))
    assert np.allclose(out['initial_TRE'], np.sqrt(1 + 4 + 0.25))
    assert out['mean_TRE_of_mean'] == pytest.approx(table[:, 3].mean())
    spread = np.sqrt(table[:, 6] + table[:, 9] + table[:, 11])
    assert out['uncertainty_error_spearman'] == pytest.approx(stats.spearmanr(spread, table[:, 3])[0])
    table[:, 5:] = np.nan   # one sample: no covariance
    out1 = landmark_posterior_summary(table, p, q, s)
    assert all(np.isnan(v) for v in out1['coverage'].values()) and np.isnan(out1['uncertainty_error_spearman'])
    path = tmp_path / 'lm.vtk'
    cov = rng.random((P, 6))
    save_landmarks_to_disk(path, p, cov, {'a': table[:, 3], 'b': np.full(P, np.nan)})
    pts, arrays = load_landmarks_from_disk(path)
    assert np.allclose(pts, p.astype(np.float32))
    assert np.allclose(arrays['covariance'], cov[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(P, 3, 3).astype(np.float32))
    assert np.allclose(arrays['a'], table[:, 3].astype(np.float32)) and np.isnan(arrays['b']).all()
    assert path.read_bytes().startswith(b'# vtk DataFile Version 3.0\n') and b'DATASET POLYDATA' in path.read_bytes()
