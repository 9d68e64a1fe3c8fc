"""
Average surface distance at the shape of configuration 4 (BASELINE.json: 256^3 with segmentations, per-sample Dice / ASD):
make_pair segmentations warped by an SGLD sampler after a few transitions, the 15 structures of the synthetic pair, C chains.

Prints one JSON line with, per C:
  call_ms      calc_ASD_GPU, the whole call with its one host synchronisation (CUDA events, mean over --reps after warm-up)
  kernels_ms   the library's kernels of one call alone (torch.profiler in a separate pass, device time per call)
  metrics_ms   calc_metrics (Dice + ASD) end to end
  max_rel_diff largest relative difference from calc_ASD_host over all (sample, structure) pairs
and calc_ASD_host on one sample (all structures) for the ratio, the GPU name and its power limit read in the same run.

usage: python tools/bench_asd.py [--size 256] [--chains 1 16] [--reps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KERNELS = ('surface_box', 'edt_rows', 'edt_envelope', 'asd_reduce', 'fill_kernel')


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(','))
        return {'gpu': name, 'power_limit': power, 'sm_clock_max': clock}
    except Exception as exc:   # the numbers are still reported, with the reason the card could not be read
        return {'gpu': torch.cuda.get_device_name(0), 'power_limit': f'unavailable ({type(exc).__name__})'}


def kernel_ms(fn, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        if any(k in e.key for k in KERNELS):
            total += getattr(e, 'device_time_total', None) or getattr(e, 'cuda_time_total', 0.0)
    return total / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--size', type=int, default=256)
    ap.add_argument('--chains', type=int, nargs='+', default=[1, 16])
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_asd.py measures the CUDA kernels: no CUDA device')
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    from irsgmcmc_b200.utils.util import calc_ASD_GPU, calc_ASD_host, calc_metrics
    dev, n = 'cuda:0', args.size
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=dev)
    structures = {f's{l}': l for l in STRUCTURE_LABELS}
    spacing = (1.0, 1.0, 1.0)
    seg_f = fixed['seg'].to(dev)
    rec = {'tool': 'bench_asd', 'volume': [n, n, n], 'structures': len(structures), 'spacing': spacing, 'reps': args.reps,
           **gpu_info(), 'runs': []}
    host_one_s = None
    for C in args.chains:
        s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=dev)
        s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
        s.init_gmm(sigma_hat=0.7)
        s.step(3, use_graph=False)
        seg_w = s.warp_segmentation()
        seg_fc = seg_f.expand(C, -1, -1, -1, -1)
        torch.cuda.synchronize()

        def asd():
            return calc_ASD_GPU(C, seg_fc, seg_w, structures, spacing)
        for _ in range(3):
            dev_asd = asd()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            asd()
        e1.record()
        torch.cuda.synchronize()
        call_ms = e0.elapsed_time(e1) / args.reps
        calc_metrics(seg_fc, seg_w, structures, spacing, no_samples=C)
        e0.record()
        for _ in range(args.reps):
            calc_metrics(seg_fc, seg_w, structures, spacing, no_samples=C)
        e1.record()
        torch.cuda.synchronize()
        metrics_ms = e0.elapsed_time(e1) / args.reps
        k_ms = kernel_ms(asd, args.reps)
        a, b = seg_f.cpu().numpy()[0, 0], seg_w.cpu().numpy()
        host = np.zeros((C, len(structures)))
        for c in range(C):
            t0 = time.perf_counter()
            for j, lab in enumerate(STRUCTURE_LABELS):
                host[c, j] = calc_ASD_host(a == lab, b[c, 0] == lab, spacing)
            if host_one_s is None:
                host_one_s = time.perf_counter() - t0
        fin = np.isfinite(host) & (host != 0)
        same_special = bool(np.array_equal(np.isinf(dev_asd), np.isinf(host)) and np.array_equal(dev_asd == 0, host == 0))
        rel = float((np.abs(dev_asd[fin] - host[fin]) / host[fin]).max()) if fin.any() else 0.0
        rec['runs'].append({'chains': C, 'call_ms': call_ms, 'kernels_ms': k_ms, 'metrics_ms': metrics_ms,
                            'max_rel_diff_vs_host': rel, 'inf_and_zero_match_host': same_special,
                            'mean_asd_voxels': float(dev_asd[np.isfinite(dev_asd)].mean())})
        del s
        torch.cuda.empty_cache()
    rec['host_one_sample_s'] = host_one_s
    for r in rec['runs']:
        r['speedup_vs_host_one_sample'] = host_one_s * 1e3 / r['call_ms']
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
