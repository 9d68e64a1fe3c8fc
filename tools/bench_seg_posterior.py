"""
Segmentation posterior at the shape of configuration 4 (BASELINE.json: 256^3 with segmentations): the 15 structures of a
make_pair segmentation warped by an SGLD sampler of C chains after a few transitions.

Prints one JSON line (and writes it to --out) with, per call (CUDA events around --reps launches after warm-up, mean):
  update_ms        ops.label_counts_update of the C warped segmentations into the (15, V) counts
  warp_ms          the nearest-neighbour warp of the moving segmentation that produces them (irs_warp3d_nearest_i16)
  finish_ms        ops.label_posterior with the fixed segmentation: probabilities, majority, entropy, summaries
  *_bytes / *_TBps the bytes the algorithm has to move (from shapes and the counts actually touched) over the time:
                   update = read C V int16 + read and write every counts element some chain carries (4 B each way);
                   warp = read T (3 C V fp32) + write C V int16 (+ the gathered labels, at least C V int16);
                   finish = read L V int32 + write L V fp32 + V int16 + V fp32 + read V int16 of the fixed segmentation
and the segmentation work of one kept sample (transformation + nearest warp + Dice counts), without and with the update,
alternated, median over --kept-reps.  The counts (1.0 GB) and segmentations (134 MB) exceed the 126 MB L2.  The GPU name and
power limit are read in the same run.

usage: python tools/bench_seg_posterior.py [--size 256] [--chains 16] [--reps 50] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--size', type=int, default=256)
    ap.add_argument('--chains', type=int, default=16)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--kept-reps', type=int, default=21)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_seg_posterior.py measures the CUDA kernels: no CUDA device')
    from irsgmcmc_b200 import ops
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    dev, n, C, labels = 'cuda:0', args.size, args.chains, list(STRUCTURE_LABELS)
    V, L = n ** 3, len(labels)
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=dev)
    s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=dev)
    s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
    s.init_gmm(sigma_hat=0.7)
    s.step(3, use_graph=False)
    T = s.transformation()
    seg_w = s.warp_segmentation(transformation=T)
    seg_f = fixed['seg'].to(dev)
    counts = torch.zeros(L, n, n, n, device=dev, dtype=torch.int32)

    ops.label_counts_update(seg_w, labels, counts)
    touched = int((counts > 0).sum())          # counts elements one update reads and writes
    update_ms = timed(lambda: ops.label_counts_update(seg_w, labels, counts), args.reps)
    warp_ms = timed(lambda: s.warp_segmentation(transformation=T), args.reps)
    n_acc = (1 + 3 + args.reps) * C   # segmentations in the counts: the first update, the warm-up and the timed ones
    finish_ms = timed(lambda: ops.label_posterior(counts, n_acc, labels, seg_f), args.reps)

    def kept(with_update):
        T_k = s.transformation()
        w = s.warp_segmentation(transformation=T_k)
        ops.dice_counts(seg_f, w, labels)
        if with_update:
            ops.label_counts_update(w, labels, counts)
    for flag in (False, True):
        timed(lambda: kept(flag), 1, 3)
    off, on = [], []
    for _ in range(args.kept_reps):
        off.append(timed(lambda: kept(False), 1, 0))
        on.append(timed(lambda: kept(True), 1, 0))
    med = lambda xs: sorted(xs)[len(xs) // 2]

    update_bytes = 2 * C * V + 8 * touched
    warp_bytes = 12 * C * V + 2 * C * V + 2 * C * V
    finish_bytes = 4 * L * V + 4 * L * V + 2 * V + 4 * V + 2 * V
    rec = {'tool': 'bench_seg_posterior', 'volume': [n, n, n], 'chains': C, 'labels': L, 'reps': args.reps, **gpu_info(),
           'counts_GB': round(4 * L * V / 1e9, 3), 'touched_fraction': round(touched / (L * V), 4),
           'update_ms': round(update_ms, 4), 'update_bytes': update_bytes, 'update_TBps': round(update_bytes / update_ms / 1e9, 3),
           'warp_ms': round(warp_ms, 4), 'warp_bytes': warp_bytes, 'warp_TBps': round(warp_bytes / warp_ms / 1e9, 3),
           'update_over_warp': round(update_ms / warp_ms, 3),
           'finish_ms': round(finish_ms, 4), 'finish_bytes': finish_bytes, 'finish_TBps': round(finish_bytes / finish_ms / 1e9, 3),
           'kept_sample_seg_ms_off': round(med(off), 4), 'kept_sample_seg_ms_on': round(med(on), 4),
           'kept_sample_statistic': f'median of {args.kept_reps}, alternated'}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
