"""
Landmark posterior kernels per kept sample at 256^3 x 16 chains and 64^3 x 1024 chains, 300 landmarks: what the sampler adds
to accumulate() with the feature on, next to the transformation T it consumes.

Prints one JSON line (and writes it to --out) with, per configuration and per call (CUDA events around --reps calls after
warm-up, mean; the median of --rounds rounds that alternate the three measurements):
  map_update_ms    irs_landmark_map + irs_landmark_update for all C chains (the two launches accumulate() adds)
  map_ms           irs_landmark_map alone (the rest of map_update_ms is the in-order chain loop of the update)
  T_ms             irs_svf_outputs: T = identity + normalised displacement for the C chains (what accumulate() reads)
  finish_ms        irs_landmark_posterior of the P landmarks
  map_update_over_T
The displacement is random (0.5 voxel std) and the landmarks uniform inside the volume.  T (3.2 GB in both configurations)
exceeds the 126 MB L2; the landmark buffers (C P 32 bytes) fit in it.  The GPU name and power limit are read in the same run.

usage: python tools/bench_landmarks.py [--reps 20] [--rounds 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_jacobian_posterior import gpu_info, timed  # noqa: E402


def run(n, C, P, reps, rounds, dev):
    from irsgmcmc_b200 import _lib
    lib = _lib.load()
    st = _lib.stream()
    g = torch.Generator(device=dev).manual_seed(0)
    u = 0.5 * torch.randn(C, 3, n, n, n, device=dev, generator=g)
    lin = [torch.linspace(-1, 1, n, device=dev) for _ in range(3)]
    T = torch.empty_like(u)
    p = torch.rand(P, 3, device=dev, dtype=torch.float64, generator=g) * (n - 1)
    q = p + torch.randn(P, 3, device=dev, dtype=torch.float64, generator=g)
    sp = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    pred = torch.empty(C, P, 3, device=dev, dtype=torch.float64)
    tre = torch.empty(C, P, device=dev, dtype=torch.float64)
    acc = torch.zeros(P, _lib.LANDMARK_ACC, device=dev, dtype=torch.float64)
    stats = torch.empty(C, 3, device=dev, dtype=torch.float64)
    out = torch.empty(P, _lib.LANDMARK_COLS, device=dev, dtype=torch.float64)
    state = {'n': 0}

    def make_T():
        _lib.check(lib.irs_svf_outputs(_lib.ptr(u), *(_lib.ptr(x) for x in lin), _lib.ptr(T), None, C, n, n, n, st))

    def lm_map():
        _lib.check(lib.irs_landmark_map(_lib.ptr(T), C, n, n, n, _lib.ptr(p), _lib.ptr(q), P, sp, _lib.ptr(pred),
                                        _lib.ptr(tre), st))

    def map_update():
        lm_map()
        _lib.check(lib.irs_landmark_update(_lib.ptr(pred), _lib.ptr(tre), C, P, float(state['n']), _lib.ptr(acc),
                                           _lib.ptr(stats), st))
        state['n'] += C

    def finish():
        _lib.check(lib.irs_landmark_posterior(_lib.ptr(acc), _lib.ptr(q), P, max(state['n'], 1), sp, _lib.ptr(out), st))

    make_T()
    mu, mp_, tt, fin = [], [], [], []
    for r in range(rounds):
        w = 3 if r == 0 else 1
        mu.append(timed(map_update, reps, w))
        mp_.append(timed(lm_map, reps, w))
        tt.append(timed(make_T, reps, w))
        fin.append(timed(finish, reps, w))
    med = lambda xs: sorted(xs)[len(xs) // 2]
    m_u, m_m, t_ms, f_ms = med(mu), med(mp_), med(tt), med(fin)
    torch.cuda.synchronize()
    return {'volume': [n, n, n], 'chains': C, 'landmarks': P, 'map_update_ms': round(m_u, 4), 'map_ms': round(m_m, 4),
            'T_ms': round(t_ms, 4), 'finish_ms': round(f_ms, 4), 'map_update_over_T': round(m_u / t_ms, 4),
            'samples_accumulated': state['n'], 'acc_finite': bool(torch.isfinite(acc).all()),
            'statistic': f'median of {rounds} alternated rounds of the mean over {reps} calls'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_landmarks.py measures the CUDA kernels: no CUDA device')
    dev = 'cuda:0'
    configs = []
    for n, C in ((256, 16), (64, 1024)):
        configs.append(run(n, C, 300, args.reps, args.rounds, dev))
        torch.cuda.empty_cache()
    rec = {'tool': 'bench_landmarks', **gpu_info(), 'configs': configs}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
