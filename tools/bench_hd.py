"""
Hausdorff distance and HD95 at the shape of configuration 4 (BASELINE.json: 256^3 with segmentations): make_pair segmentations
warped by an SGLD sampler after a few transitions, the 15 structures of the synthetic pair, C chains.

Prints one JSON line with, per C:
  sd_call_ms / asd_call_ms   ops.surface_distances (ASD + HD + HD95) and ops.average_surface_distance (ASD alone), whole calls
                             with their host synchronisation, alternated in the same run: median over --rounds of the mean of
                             --reps calls (CUDA events)
  kernels_ms                 device time per call of each library kernel of surface_distances (torch.profiler, separate pass),
                             and of the reduction of average_surface_distance for the difference the lists make
  max_rel_diff_hd / _hd95    largest relative difference from calc_HD_host over all (sample, structure) pairs, and whether
                             they are bit-equal (unit spacing: they must be)
  longest_list               contour voxels of the largest structure: the longest list one CTA of hd_select_kernel selects in
and calc_HD_host on one sample (all structures), the GPU name and its power limit read in the same run.  'large_lists' times one
pair with the longest lists a structure can give at this size (the complement of an ellipsoid, touching all six faces).

usage: python tools/bench_hd.py [--size 256] [--chains 1 16] [--reps 10] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_asd import gpu_info  # noqa: E402

KERNELS = ('surface_box', 'edt_rows', 'edt_envelope', 'asd_reduce', 'hd_select', 'fill_kernel')


def kernel_table(fn, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                name = k + ('<true>' if '<true>' in e.key else '<false>' if '<false>' in e.key else '')
                t = getattr(e, 'device_time_total', None) or getattr(e, 'cuda_time_total', 0.0)
                out[name] = out.get(name, 0.0) + t / 1e3 / reps
    return out


def timed(fn, reps):
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
    ap.add_argument('--chains', type=int, nargs='+', default=[1, 16])
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_hd.py measures the CUDA kernels: no CUDA device')
    from irsgmcmc_b200 import ops
    from irsgmcmc_b200.data_loader.synthetic import STRUCTURE_LABELS, make_pair
    from irsgmcmc_b200.sampler import SGLDConfig, SGLDSampler
    from irsgmcmc_b200.utils.util import _label_contour, calc_HD_host
    dev, n = 'cuda:0', args.size
    torch.manual_seed(0)
    fixed, moving, vp = make_pair(n, device=dev)
    labels = list(STRUCTURE_LABELS)
    spacing = (1.0, 1.0, 1.0)
    seg_f = fixed['seg'].to(dev)
    rec = {'tool': 'bench_hd', 'volume': [n, n, n], 'structures': len(labels), 'spacing': spacing, 'percentile': 95.0,
           'reps': args.reps, 'rounds': args.rounds, **gpu_info(), 'runs': []}
    host_one_s = None
    for C in args.chains:
        s = SGLDSampler(fixed, moving, C, SGLDConfig(), device=dev)
        s.set_state(0.5 * torch.randn(C, 3, n, n, n), torch.exp(0.5 * vp['log_var']))
        s.init_gmm(sigma_hat=0.7)
        s.step(3, use_graph=False)
        seg_w = s.warp_segmentation()
        torch.cuda.synchronize()

        def sd():
            return ops.surface_distances(seg_f, seg_w, labels, spacing, 95.0)

        def asd():
            return ops.average_surface_distance(seg_f, seg_w, labels, spacing)
        for _ in range(3):
            dev_asd, dev_hd, dev_q = (t.cpu().numpy() for t in sd())
            asd()
        assert np.array_equal(dev_asd, asd().cpu().numpy())
        t_sd, t_asd = [], []
        for _ in range(args.rounds):   # alternated, so that both see the same state of the machine
            t_sd.append(timed(sd, args.reps))
            t_asd.append(timed(asd, args.reps))
        k_sd, k_asd = kernel_table(sd, args.reps), kernel_table(asd, args.reps)
        a, b = seg_f.cpu().numpy()[0, 0], seg_w.cpu().numpy()
        host_hd, host_q = np.zeros((C, len(labels))), np.zeros((C, len(labels)))
        longest = 0
        for c in range(C):
            t0 = time.perf_counter()
            for j, lab in enumerate(labels):
                host_hd[c, j], host_q[c, j] = calc_HD_host(a == lab, b[c, 0] == lab, spacing)
            if host_one_s is None:
                host_one_s = time.perf_counter() - t0
            for lab in labels:
                longest = max(longest, int(_label_contour(a == lab).sum()), int(_label_contour(b[c, 0] == lab).sum()))

        def rel(got, want):
            fin = np.isfinite(want) & (want != 0)
            return float((np.abs(got[fin] - want[fin]) / want[fin]).max()) if fin.any() else 0.0
        run = {'chains': C, 'sd_call_ms': float(np.median(t_sd)), 'asd_call_ms': float(np.median(t_asd)),
               'sd_call_ms_all': t_sd, 'asd_call_ms_all': t_asd, 'kernels_ms_surface_distances': k_sd,
               'kernels_ms_average_surface_distance': k_asd,
               'max_rel_diff_hd': rel(dev_hd, host_hd), 'max_rel_diff_hd95': rel(dev_q, host_q),
               'bit_equal_to_host': bool(np.array_equal(dev_hd, host_hd) and np.array_equal(dev_q, host_q)),
               'longest_list': longest, 'mean_hd_voxels': float(dev_hd.mean()), 'mean_hd95_voxels': float(dev_q.mean())}
        run['sd_over_asd'] = run['sd_call_ms'] / run['asd_call_ms']
        rec['runs'].append(run)
        del s
        torch.cuda.empty_cache()
    rec['host_one_sample_s'] = host_one_s
    # the longest lists a structure can give: the complement of an ellipsoid touches all six faces (about 4e5 contour voxels at
    # 256^3), against the same shape shifted by a few voxels -- does the single selection CTA per list make a tail?
    zz, yy, xx = (torch.arange(n, device=dev, dtype=torch.float64).view(*sh) for sh in ((-1, 1, 1), (1, -1, 1), (1, 1, -1)))

    def outside(c, r):
        return ((zz - c[0]) / r[0]) ** 2 + ((yy - c[1]) / r[1]) ** 2 + ((xx - c[2]) / r[2]) ** 2 > 1.0
    big_a = (3 * outside((n / 2, n / 2, n / 2), (n / 2.6,) * 3)).to(torch.int16)[None, None].contiguous()
    big_b = (3 * outside((n / 2 + 3, n / 2, n / 2 - 2), (n / 2.4, n / 2.7, n / 2.5))).to(torch.int16)[None, None].contiguous()

    def big_sd():
        return ops.surface_distances(big_a, big_b, [3], spacing, 95.0)

    def big_asd():
        return ops.average_surface_distance(big_a, big_b, [3], spacing)
    for _ in range(3):
        _, g_hd, g_q = (float(t.item()) for t in big_sd())
        big_asd()
    t_sd, t_asd = [], []
    for _ in range(args.rounds):
        t_sd.append(timed(big_sd, args.reps))
        t_asd.append(timed(big_asd, args.reps))
    a, b = big_a.cpu().numpy()[0, 0] == 3, big_b.cpu().numpy()[0, 0] == 3
    w_hd, w_q = calc_HD_host(a, b, spacing)
    rec['large_lists'] = {'contour_voxels': [int(_label_contour(a).sum()), int(_label_contour(b).sum())],
                          'sd_call_ms': float(np.median(t_sd)), 'asd_call_ms': float(np.median(t_asd)),
                          'kernels_ms_surface_distances': kernel_table(big_sd, args.reps),
                          'kernels_ms_average_surface_distance': kernel_table(big_asd, args.reps),
                          'hd': g_hd, 'hd95': g_q, 'bit_equal_to_host': g_hd == w_hd and g_q == w_q}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
