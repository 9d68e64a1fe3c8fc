"""
fp64 numpy restatement of the landmark posterior (irsgmcmc_b200/csrc/irs_landmark.cuh, irs_landmark.cu):
  predict / tre    utils.util.landmark_predict_host / landmark_tre_host (bit-equal to the kernel), and plain per-landmark
                   loops of the same definition that the tests hold them against;
  accumulate       the Welford recurrence of irs_landmark_welford over stacked samples, every operation rounded on its own
                   (bit-equal to the kernel);
  two_pass         mean and co-moments of the stacked samples in two passes, the independent check of accumulate;
  posterior        the (P,16) table of irs_landmark_finish through np.linalg.eigvalsh and np.linalg.solve.
"""
import math

import numpy as np

from irsgmcmc_b200.utils.util import landmark_predict_host, landmark_tre_host

PAIRS = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]


def predict_loops(T, p):
    """(C,P,3) by plain loops: floor, clamp to [0, n - 2], three lerps per axis order x, y, z, then ((g + 1)(n - 1)) / 2"""
    T = np.asarray(T, dtype=np.float32)
    C, _, D, H, W = T.shape
    n = (W, H, D)
    out = np.empty((C, len(p), 3))
    for c in range(C):
        for i, pt in enumerate(np.asarray(p, dtype=np.float64)):
            base, frac = [], []
            for a in range(3):
                fl = math.floor(pt[a]) if math.isfinite(pt[a]) else (0 if math.isnan(pt[a]) else (n[a] - 2 if pt[a] > 0 else 0))
                i0 = min(max(int(fl), 0), n[a] - 2)
                base.append(i0)
                frac.append(pt[a] - i0)
            x0, y0, z0 = base
            for ch in range(3):
                v = lambda dz, dy, dx: float(T[c, ch, z0 + dz, y0 + dy, x0 + dx])
                lerp = lambda a, b, f: a + f * (b - a)
                c0 = lerp(lerp(v(0, 0, 0), v(0, 0, 1), frac[0]), lerp(v(0, 1, 0), v(0, 1, 1), frac[0]), frac[1])
                c1 = lerp(lerp(v(1, 0, 0), v(1, 0, 1), frac[0]), lerp(v(1, 1, 0), v(1, 1, 1), frac[0]), frac[1])
                g = lerp(c0, c1, frac[2])
                out[c, i, ch] = ((g + 1.0) * (n[ch] - 1)) * 0.5
    return out


def tre_loops(pred, q, s):
    out = np.empty(pred.shape[:2])
    for c in range(pred.shape[0]):
        for i in range(pred.shape[1]):
            acc = 0.0
            for a in range(3):
                d = s[a] * (pred[c, i, a] - q[i][a])
                acc = acc + d * d
            out[c, i] = math.sqrt(acc)
    return out


predict = landmark_predict_host
tre = landmark_tre_host


def accumulate(pred, tre_, acc=None, count_before=0):
    """(P, 11) accumulators after folding pred (N,P,3) / tre (N,P) in sample order into acc (zeros by default)"""
    N, P = tre_.shape
    acc = np.zeros((P, 11)) if acc is None else acc.copy()
    for k in range(N):
        kk = float(count_before + k + 1)
        m = pred[k]
        d = m - acc[:, :3]
        acc[:, :3] = acc[:, :3] + d / kk
        e = m - acc[:, :3]
        for j, (a, b) in enumerate(PAIRS):
            acc[:, 3 + j] = acc[:, 3 + j] + d[:, a] * e[:, b]
        dt = tre_[k] - acc[:, 9]
        acc[:, 9] = acc[:, 9] + dt / kk
        acc[:, 10] = acc[:, 10] + dt * (tre_[k] - acc[:, 9])
    return acc


def two_pass(pred, tre_):
    """(P, 11) from the stacked samples: mean, sum of (x - mean)_a (x - mean)_b, TRE mean and sum of squared deviations"""
    mean = pred.mean(0)
    d = pred - mean
    out = np.empty((pred.shape[1], 11))
    out[:, :3] = mean
    for j, (a, b) in enumerate(PAIRS):
        out[:, 3 + j] = (d[..., a] * d[..., b]).sum(0)
    out[:, 9] = tre_.mean(0)
    out[:, 10] = ((tre_ - out[:, 9]) ** 2).sum(0)
    return out


def covariance(acc, n, s):
    """(P, 3, 3) covariance in mm^2"""
    s = np.asarray(s, dtype=np.float64)
    S = np.empty((acc.shape[0], 3, 3))
    for j, (a, b) in enumerate(PAIRS):
        S[:, a, b] = S[:, b, a] = s[a] * s[b] * acc[:, 3 + j] / (n - 1)
    return S


def posterior(acc, n, q, s):
    """(P, 16) table of irs_landmark_posterior through numpy's eigvalsh / solve"""
    q, s = np.asarray(q, dtype=np.float64), np.asarray(s, dtype=np.float64)
    P = acc.shape[0]
    out = np.full((P, 16), np.nan)
    out[:, :3] = acc[:, :3]
    out[:, 3] = np.sqrt((((acc[:, :3] - q) * s) ** 2).sum(1))
    out[:, 4] = acc[:, 9]
    if n < 2:
        return out
    out[:, 5] = np.sqrt(acc[:, 10] / (n - 1))
    S = covariance(acc, n, s)
    for j, (a, b) in enumerate(PAIRS):
        out[:, 6 + j] = S[:, a, b]
    ev = np.linalg.eigvalsh(S)[:, ::-1]
    out[:, 12:15] = np.sqrt(np.maximum(ev, 0.0))
    r = (q - acc[:, :3]) * s
    for i in range(P):
        try:
            np.linalg.cholesky(S[i])
            out[i, 15] = float(r[i] @ np.linalg.solve(S[i], r[i]))
        except np.linalg.LinAlgError:
            out[i, 15] = np.inf
    return out
