"""
Convergence diagnostics on one GPU: the per-kept-sample split-Welford update and the final split R-hat at the sizes the sampler
runs many chains (64 chains at 128^3, 16 at 256^3), and what the update adds to a kept sample of the SGLD sampler.

Prints one JSON line (and writes it to --out) with, per (chains, size):
  update_ms / update_TBps      ops.split_welford_update of one sample of every chain (CUDA events, mean over --reps after
                               warm-up); bytes = the algorithm's: read the sample (4 V floats per chain), read and write mean
                               and M2 of its sequence (4 x 4 V floats)
  pooled_update_ms / _TBps     the pooled Welford update of the same sample (irs_welford_update, what accumulate() always runs)
  rhat_ms / rhat_TBps          ops.split_rhat over the 2 C sequences (three kernels + allocations); bytes = read mean / M2 of all
                               sequences twice and once, the fp64 sums and the maps
and, for --kept-chains chains at --kept-size, the time of a kept sample (one transition + accumulate()) with the diagnostics off
and on, alternated.  The working sets exceed the 126 MB L2.  The GPU name and power limit are read in the same run.

usage: python tools/bench_rhat.py [--reps 20] [--out profiles/rhat_bench.json]
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


def kernels(C, n, reps):
    from irsgmcmc_b200 import ops
    V = n ** 3
    dev = 'cuda:0'
    g = torch.Generator(device=dev).manual_seed(0)
    disp = torch.randn(C, 3, n, n, n, device=dev, generator=g)
    im = torch.rand(C, 1, n, n, n, device=dev, generator=g)
    mean = torch.zeros(2, C, 4, n, n, n, device=dev)
    m2 = torch.zeros_like(mean)
    half = [0]

    def update():
        ops.split_welford_update(disp, im, half[0], 10, mean, m2)
        half[0] ^= 1
    upd = timed(update, reps)
    pm, pm2 = torch.zeros(3, n, n, n, device=dev), torch.zeros(3, n, n, n, device=dev)
    im_m, im_m2 = torch.zeros(1, n, n, n, device=dev), torch.zeros(1, n, n, n, device=dev)

    def pooled():
        ops.welford_update(disp, 10, pm, pm2)
        ops.welford_update(im, 10, im_m, im_m2)
    pool = timed(pooled, reps)
    # a plausible state for the R-hat: every sequence holds 50 draws around its own mean
    mean.copy_(torch.randn_like(mean) * 0.1)
    m2.copy_(torch.rand_like(m2) * 49.0)
    mask = torch.ones(n, n, n, device=dev, dtype=torch.bool)
    rh = timed(lambda: ops.split_rhat(mean.view(2 * C, 4, n, n, n), m2.view(2 * C, 4, n, n, n), 50, mask), max(3, reps // 4), 1)
    M, E = 2 * C, 4 * V
    upd_bytes = C * V * (16 + 32 + 32)
    pool_bytes = C * V * 16 + V * 4 * 16
    rhat_bytes = 2 * M * E * 4 + 2 * E * 8 + (M * E * 4 + E * 8 + E * 8) + (2 * E * 8 + V + E * 4)
    del disp, im, mean, m2
    torch.cuda.empty_cache()
    return {'chains': C, 'size': n, 'accumulator_GB': round(64 * C * V / 1e9, 2),
            'update_ms': round(upd, 4), 'update_TBps': round(upd_bytes / upd / 1e9, 3),
            'pooled_update_ms': round(pool, 4), 'pooled_update_TBps': round(pool_bytes / pool / 1e9, 3),
            'rhat_ms': round(rh, 3), 'rhat_TBps': round(rhat_bytes / rh / 1e9, 3)}


def kept_sample(C, n, reps):
    """a kept sample of the sampler (one transition + accumulate()) with the diagnostics off / on, alternated"""
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    from irsgmcmc_b200.data_loader.synthetic import make_pair
    fixed, moving, vp = make_pair(n)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(hyper_mode='per_chain'), device='cuda:0')
    torch.manual_seed(0)
    s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
    s.init_gmm(sigma_hat=0.7)
    s.step(2)
    off, on = [], []
    for _ in range(reps):
        for diag, out in ((False, off), (True, on)):
            if diag:
                s.enable_convergence_diagnostics(4)
            else:
                s.disable_convergence_diagnostics()
            out.append(timed(lambda: (s.step(1), s.accumulate()), 1, 0))
    s.disable_convergence_diagnostics()
    off_ms, on_ms = sorted(off)[len(off) // 2], sorted(on)[len(on) // 2]
    return {'chains': C, 'size': n, 'kept_sample_ms_off': round(off_ms, 3), 'kept_sample_ms_on': round(on_ms, 3),
            'slowdown': round(on_ms / off_ms, 4), 'reps': reps, 'statistic': 'median'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--sizes', default='64x128,16x256', help='chains x size, comma separated')
    ap.add_argument('--kept-chains', type=int, default=64)
    ap.add_argument('--kept-size', type=int, default=128)
    ap.add_argument('--kept-reps', type=int, default=8, help='kept samples timed with the diagnostics off and with them on')
    ap.add_argument('--out', default=os.path.join('profiles', 'rhat_bench.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rhat.py measures the CUDA kernels: no CUDA device')
    res = dict(gpu_info())
    res['kernels'] = [kernels(int(c), int(n), args.reps) for c, n in (x.split('x') for x in args.sizes.split(','))]
    res['kept_sample'] = kept_sample(args.kept_chains, args.kept_size, args.kept_reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
