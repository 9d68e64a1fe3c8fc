"""
Jacobian posterior kernels at 256^3 x 16 chains and 64^3 x 1024 chains: the transformation is the identity plus a smooth random
displacement (a few percent of the voxels fold), generated on the device.

Prints one JSON line (and writes it to --out) with, per configuration and per call (CUDA events around --reps launches after
warm-up, mean; the median of --rounds rounds that alternate the kernels):
  update_ms        ops.jacobian_update of the C transformations into the accumulators (folds, mean, m2) + per-chain sums
  log_det_ms       ops.log_det_jacobian of the same T (the existing kernel, which writes a (C,D,H,W) volume)
  finish_ms        ops.jacobian_posterior: the three maps and the mask summaries
  *_bytes / *_TBps the bytes the algorithm has to move, from shapes, over the time:
                   update = read T (12 B per chain and voxel) + mask (1 B) + read and write the accumulators (12 B each way);
                   log_det = read T + write log det J (4 B per chain and voxel);
                   finish = read the accumulators (12 B) and the mask (1 B) + write three fp32 maps (12 B)
T (3.2 GB in both configurations) exceeds the 126 MB L2.  The GPU name and power limit are read in the same run.

usage: python tools/bench_jacobian_posterior.py [--reps 20] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(','))
        return {'gpu': name, 'power_limit': power, 'sm_clock_max': clock}
    except Exception as exc:   # the numbers are still reported, with the reason the card could not be read
        return {'gpu': torch.cuda.get_device_name(0), 'power_limit': f'unavailable ({type(exc).__name__})'}


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def transformation(C, n, dev, seed=0):
    """identity + a smooth random field, (C,3,n,n,n) fp32 on the device: N(0,1) on a grid of m^3 points 8 voxels apart,
    trilinearly interpolated and scaled by 1 / m, so that its gradient in normalised units is about N(0, 1/2)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    lin = torch.linspace(-1, 1, n, device=dev)
    z, y, x = torch.meshgrid(lin, lin, lin, indexing='ij')
    T = torch.empty(C, 3, n, n, n, device=dev)
    m = max(n // 8, 2)
    amp = 1.0 / m
    for c in range(C):   # one chain at a time: the interpolation's temporaries stay small
        u = torch.nn.functional.interpolate(torch.randn(1, 3, m, m, m, device=dev, generator=g), size=(n, n, n),
                                            mode='trilinear', align_corners=True)[0]
        T[c, 0], T[c, 1], T[c, 2] = x + amp * u[0], y + amp * u[1], z + amp * u[2]
    return T


def run(n, C, reps, rounds, dev):
    from irsgmcmc_b200 import ops
    V = n ** 3
    T = transformation(C, n, dev)
    mask = torch.ones(n, n, n, device=dev, dtype=torch.bool)
    folds = torch.zeros(n, n, n, device=dev, dtype=torch.int32)
    mean, m2 = torch.zeros(n, n, n, device=dev), torch.zeros(n, n, n, device=dev)
    scratch = ops.jacobian_scratch(C, dev)
    state = {'count': 0}

    def update():
        ops.jacobian_update(T, mask, state['count'], folds, mean, m2, scratch)
        state['count'] += C

    upd, ldj, fin = [], [], []
    for r in range(rounds):
        upd.append(timed(update, reps, 3 if r == 0 else 1))
        ldj.append(timed(lambda: ops.log_det_jacobian(T), reps, 3 if r == 0 else 1))
        fin.append(timed(lambda: ops.jacobian_posterior(folds, mean, m2, state['count'], mask), reps, 3 if r == 0 else 1))
    med = lambda xs: sorted(xs)[len(xs) // 2]
    counts, _ = ops.log_det_jacobian(T, want_log_det=False)
    update_ms, log_det_ms, finish_ms = med(upd), med(ldj), med(fin)
    update_bytes = 12 * C * V + V + 24 * V
    log_det_bytes = 12 * C * V + 4 * C * V
    finish_bytes = 12 * V + V + 12 * V
    return {'volume': [n, n, n], 'chains': C, 'folded_fraction': round(float(counts.sum()) / (C * V), 5),
            'update_ms': round(update_ms, 4), 'update_bytes': update_bytes, 'update_TBps': round(update_bytes / update_ms / 1e9, 3),
            'log_det_ms': round(log_det_ms, 4), 'log_det_bytes': log_det_bytes,
            'log_det_TBps': round(log_det_bytes / log_det_ms / 1e9, 3), 'update_over_log_det': round(update_ms / log_det_ms, 3),
            'finish_ms': round(finish_ms, 4), 'finish_bytes': finish_bytes, 'finish_TBps': round(finish_bytes / finish_ms / 1e9, 3),
            'statistic': f'median of {rounds} alternated rounds of the mean over {reps} launches'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_jacobian_posterior.py measures the CUDA kernels: no CUDA device')
    dev = 'cuda:0'
    configs = []
    for n, C in ((256, 16), (64, 1024)):
        configs.append(run(n, C, args.reps, args.rounds, dev))
        torch.cuda.empty_cache()
    rec = {'tool': 'bench_jacobian_posterior', **gpu_info(), 'configs': configs}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
