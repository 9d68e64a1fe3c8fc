"""
Convergence diagnostics of scalar MCMC traces (host, numpy): split R-hat (BDA3 section 11.4) and the multi-chain bulk effective
sample size of split chains (BDA3 section 11.5) with Geyer's initial monotone sequence.  For the per-voxel R-hat maps of the
displacement and the warped image see SGLDSampler.convergence_diagnostics (CUDA kernels in csrc/irs_diagnostics.cu).

`draws` is (chains, N): N draws of one scalar per chain.  Each chain is split into its first and last floor(N/2) draws (the
middle one of an odd N is dropped): M = 2 chains sequences of n = floor(N/2) draws.
"""
import numpy as np


def split_chains(draws):
    """(chains, N) -> (2 chains, floor(N/2)): the first halves of every chain, then the last halves"""
    x = np.asarray(draws, dtype=np.float64)
    if x.ndim != 2:
        raise ValueError('draws must be (chains, N)')
    n = x.shape[1] // 2
    if n < 2:
        raise ValueError('split R-hat / ESS need N >= 4 draws per chain')
    return np.concatenate((x[:, :n], x[:, x.shape[1] - n:]), axis=0)


def split_rhat(draws):
    """
    potential scale reduction factor of split chains: W = mean within-sequence variance, B/n = variance of the sequence means,
    var+ = (n - 1)/n W + B/n, R-hat = sqrt(var+ / W).  Every draw identical (W = 0, B = 0): 1; W = 0 < B: +inf -- the rules of
    the device kernel (csrc/irs_diagnostics.cu).
    """
    s = split_chains(draws)
    M, n = s.shape
    means = s.mean(axis=1)
    W = s.var(axis=1, ddof=1).mean()
    B_n = means.var(ddof=1)
    if W == 0.0:
        return 1.0 if B_n == 0.0 else float('inf')
    return float(np.sqrt(((n - 1) / n * W + B_n) / W))


def ess(draws):
    """
    bulk effective sample size of split chains (BDA3 section 11.5): rho_t = 1 - V_t / (2 var+) with the variogram
    V_t = mean over sequences of mean_i (x_{i+t} - x_i)^2; the autocorrelations are summed in pairs (rho_2k + rho_2k+1, starting
    at rho_0 = 1) while the pair sums stay positive, each pair sum capped at the one before (Geyer's initial monotone sequence).
    ESS = M n / (-1 + 2 sum of the pair sums).  NaN when every draw is identical (var+ = 0).
    """
    s = split_chains(draws)
    M, n = s.shape
    W = s.var(axis=1, ddof=1).mean()
    var_plus = (n - 1) / n * W + s.mean(axis=1).var(ddof=1)
    if not var_plus > 0.0:
        return float('nan')
    # variogram of every lag through the autocovariance (FFT): V_t = (sum_i x_i^2 + x_{i+t}^2 - 2 x_i x_{i+t}) / (n - t)
    c = s - s.mean(axis=1, keepdims=True)
    f = np.fft.rfft(c, n=2 * n, axis=1)
    acov = np.fft.irfft(f * np.conj(f), n=2 * n, axis=1)[:, :n]          # sum_i c_i c_{i+t}
    sq = c ** 2
    head = np.cumsum(sq[:, ::-1], axis=1)[:, ::-1]                       # sum_{i >= t} c_i^2
    tail = np.cumsum(sq, axis=1)[:, ::-1]                                # sum_{i < n - t} c_i^2
    t = np.arange(n)
    V = ((head + tail - 2.0 * acov) / (n - t)).mean(axis=0)
    rho = 1.0 - V / (2.0 * var_plus)
    rho[0] = 1.0
    total, prev = 0.0, np.inf
    for k in range(0, n - 1, 2):
        p = rho[k] + rho[k + 1]
        if not p > 0.0:
            break
        p = min(p, prev)
        total += p
        prev = p
    tau = -1.0 + 2.0 * total
    return float(M * n / tau)
