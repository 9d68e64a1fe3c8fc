"""
fp64 reference of one scaling-and-squaring step and of its adjoint that takes the kernels' own fp32 decisions.

A trilinear gradient is piecewise constant in the sampling position, so an fp64 oracle that computes the position in
fp64 disagrees with any fp32 kernel by O(1) wherever a 1-ulp difference moves a sample across a cell face.  This
reference removes those kinks instead of tolerating them.  From the input field u (fp32, as the kernels read it) it
takes exactly the decisions the kernels take (csrc/irs_bodies.cuh, csrc/irs_common.cuh, csrc/irs_svf.cu):

  * position        p = fl32(x + u in_scale), clamped to [0, n - 1]       (u in_scale is exact: in_scale = 2^-k)
  * cell            floor(p), the fraction p - floor(p) (exact in fp32), inside(p) = 0 < p < n - 1 before the clamp
  * source offset   c = clamp(u in_scale, -s, n - 1 - s)                  (the transpose, in the kernels' offset form)

and evaluates everything after them in fp64.  A kernel result can then be held to a per-voxel rounding bound with no
exceptions.  Given fp64 input the same code makes fp64 decisions, i.e. it is the exact operation (test_svf_step_ref.py
checks it against the oracle's ATen pipeline at that precision).

Rounding bounds (u = 2^-24, first order; SO = 1 + 2^-10 covers the second-order terms: every m u below is < 2^-10)
--------------------------------------------------------------------------------------------------------------------
Forward, out = u s + s trilinear[u](p) per component.  The fractions are exact, so only the arithmetic rounds.  A lerp
a + f (b - a) of values bounded by M rounds the difference (2uM, scaled by f <= 1), the product (2uM, none with an
FMA) and the sum (uM): 5uM per level, and a level passes on its inputs' errors as a convex combination.  Three levels
give 15uM; the final add of u s rounds once more, u (|u s| + s M):

    |out_kernel - out| <= u SO (|u s| + 16 s M),   M = max |u| over the 8 corners of the cell (raw, unscaled)

Adjoint, out(t) = o_s [ g(t) + inside(t) s sum_k g_k(t) grad trilinear[u_k](p(t)) + sum_s w(s, t) g(s) ], o_s = out_scale.
  * position term: the corner values W = sum_k g_k U_k (or the three per-component gradients) round by <= 3uA with
    A = sum_k |g_k(t)| M_k(t); the lerps and differences of the gradient add 5u per lerp level on values <= 2A and one
    rounding per difference, 28uA in total = 14u P with P = 2 s inside A, the bound on the term's magnitude.
  * transpose: a weight is the product of three hats; each hat 1 - |c + o| (or max(c, 0)) is off by <= u in absolute
    terms, and the two products round relatively (2u w).  The body kernels (global gathers, the scatter companion, the
    host emulation) use the position form hat(fl(s + c) - t) instead of the offset form: fl(s + c) is off by
    <= ulp(n) / 2 <= n u per axis.  Both absolute errors together: 3 (n + 1) u |g(s)| per source s in the support.
  * the sum: every accumulation (FMA or add, in any order, atomics included) rounds once by <= u times the sum of the
    magnitudes of the terms, S(t) = |g(t)| + P(t) + sum_s w(s, t) |g(s)|; there are at most K(t) = |supp(t)| + 2
    non-zero terms (sources whose hat weight may be non-zero in either form, the direct and the position term).

    |out_kernel - out| <= o_s u SO [ (K + 16) S + 3 (n + 1) G ],   G(t) = sum_{s in supp(t)} |g(s)|,
    supp(t) = { s : |s_a + c_a - t_a| < 1 + n u on every axis a }

When the incoming gradient itself carries an error bound b (compose), |g| is replaced by |g| + b in S and G and the
step adds the exact propagation of b through the step with absolute values, o_s [ b + |position| b + |transpose| b ].

Layout helpers: max_abs / cell_map give what the forward pass leaves in its maxabs block (irs_svf_maxabs_floats):
n_steps global maxima of |u_k|, then n_steps cell maps (C, nz, ny, nx) of 32 x 8 x 8 voxels (csrc/irs_svf.cu make_cells).
"""
import math

import torch
import torch.nn.functional as F

from tests.util import smooth_field as _smooth_field

U24 = 2.0 ** -24
SO = 1.0 + 2.0 ** -10
CELL_X, CELL_Y, CELL_Z = 32, 8, 8


def _coords(shape, device, dtype):
    C, _, D, H, W = shape
    z, y, x = torch.meshgrid(torch.arange(D, device=device), torch.arange(H, device=device), torch.arange(W, device=device),
                             indexing='ij')
    return [t.reshape(1, -1).to(dtype) for t in (x, y, z)]


class Step:
    """the decisions of one step on input u (C, 3, D, H, W) with in_scale; fwd() and bwd() evaluate from them in fp64"""

    def __init__(self, u, in_scale):
        C, _, D, H, W = u.shape
        self.shape, self.C, self.V = u.shape, C, D * H * W
        self.dims = (W, H, D)                      # axis a = 0 (x, W), 1 (y, H), 2 (z, D)
        self.stride = (1, W, W * H)
        self.s = float(in_scale)
        self.n = max(D, H, W)
        V = self.V
        us = u * in_scale                          # exact: in_scale is a power of two
        self.u64 = u.double().reshape(C, 3, V)
        self.us64 = us.double().reshape(C, 3, V)
        xyz = _coords(u.shape, u.device, u.dtype)
        self.inside, self.i0, self.i1, self.f = [], [], [], []
        self.t0, self.ft = [], []
        for a in range(3):
            n, ua = self.dims[a], us[:, a].reshape(C, V)
            q = xyz[a] + ua                        # fl(x + u s) in the input's precision
            self.inside.append(((q > 0) & (q < n - 1)).double())
            p = q.clamp(0, n - 1)
            fl = torch.floor(p)
            self.f.append((p - fl).double())       # exact
            i0 = fl.long()
            self.i0.append(i0)
            self.i1.append((i0 + 1).clamp(max=n - 1))   # far border: stride 0 (that corner has weight 0)
            c = torch.maximum(torch.minimum(ua, (n - 1) - xyz[a]), -xyz[a])   # clamp(u s, -s, n - 1 - s), exact
            qs = xyz[a].double() + c.double()      # s + c, exact in fp64
            t0 = torch.floor(qs)
            self.t0.append(t0.long())
            self.ft.append(qs - t0)
        self._corners = None

    # ---- target side: the cell of p(t) ----
    def corners(self):
        """[(bits, index (C, V), weight (C, V))] for the 8 corners of every voxel's cell"""
        if self._corners is None:
            out = []
            for b in range(8):
                bits = (b & 1, (b >> 1) & 1, b >> 2)
                idx, w = 0, 1.0
                for a in range(3):
                    idx = idx + (self.i1[a] if bits[a] else self.i0[a]) * self.stride[a]
                    w = w * (self.f[a] if bits[a] else 1.0 - self.f[a])
                out.append((bits, idx, w))
            self._corners = out
        return self._corners

    def _gather(self, field, idx):
        return torch.gather(field, 2, idx.unsqueeze(1).expand(-1, field.shape[1], -1))

    def fwd(self):
        """(out, bound) of the step, (C, 3, D, H, W) fp64"""
        interp = torch.zeros_like(self.u64)
        M = torch.zeros_like(self.u64)
        for _, idx, w in self.corners():
            vals = self._gather(self.u64, idx)
            interp += w.unsqueeze(1) * vals
            M = torch.maximum(M, vals.abs())
        out = self.us64 + self.s * interp
        bound = U24 * SO * (self.us64.abs() + 16.0 * self.s * M)
        return out.view(self.shape), bound.view(self.shape)

    # ---- source side: the interpolation transpose in offset form ----
    def _scatter(self, vals, offsets=(0, 1), weighted=True):
        """sum over sources s of w(s, t) vals(s) (weighted) or of [t in supp(s)] vals(s); vals (C, k, V)"""
        C, k, V = vals.shape
        src = vals.permute(0, 2, 1).reshape(C * V, k)
        out = torch.zeros_like(src)
        base = (torch.arange(C, device=vals.device) * V).view(C, 1)
        delta = self.n * U24
        for oz in offsets:
            for oy in offsets:
                for ox in offsets:
                    o = (ox, oy, oz)
                    idx, w = base, torch.ones_like(self.ft[0])
                    for a in range(3):
                        t = self.t0[a] + o[a]
                        ok = (t >= 0) & (t < self.dims[a])
                        if weighted:
                            wa = self.ft[a] if o[a] == 1 else 1.0 - self.ft[a]
                        else:
                            wa = torch.ones_like(self.ft[a])
                            if o[a] == -1:
                                ok = ok & (self.ft[a] < delta)
                            elif o[a] == 2:
                                ok = ok & (self.ft[a] > 1.0 - delta)
                        w = w * wa * ok
                        idx = idx + t.clamp(0, self.dims[a] - 1) * self.stride[a]
                    out.index_add_(0, idx.reshape(-1), src * w.reshape(-1, 1))
        return out.view(C, V, k).permute(0, 2, 1)

    def bwd(self, g, out_scale, g_err=None):
        """(out, bound) of the adjoint step for incoming gradient g (C, 3, D, H, W); g_err: a bound on g's own error"""
        C, V = self.C, self.V
        g = g.double().reshape(C, 3, V)
        b = torch.zeros_like(g) if g_err is None else g_err.double().reshape(C, 3, V)
        ga = g.abs() + b
        # position term: d trilinear[u_k] / d p_a at p(t), raw corner values
        grad = [torch.zeros_like(g) for _ in range(3)]     # grad[a][:, k] = d_a trilinear[u_k]
        M = torch.zeros_like(g)
        for bits, idx, _ in self.corners():
            vals = self._gather(self.u64, idx)
            M = torch.maximum(M, vals.abs())
            for a in range(3):
                w = 1.0 if bits[a] else -1.0
                for e in range(3):
                    if e != a:
                        w = w * (self.f[e] if bits[e] else 1.0 - self.f[e])
                grad[a] += w.unsqueeze(1) * vals
        A = (ga * M).sum(1)
        pos = torch.stack([self.inside[a] * self.s * (g * grad[a]).sum(1) for a in range(3)], 1)
        pos_b = torch.stack([self.inside[a] * self.s * (b * grad[a].abs()).sum(1) for a in range(3)], 1)
        P = torch.stack([2.0 * self.s * self.inside[a] * A for a in range(3)], 1)
        tr = self._scatter(torch.cat([g, ga, b], 1))
        tr_g, tr_ga, tr_b = tr[:, 0:3], tr[:, 3:6], tr[:, 6:9]
        sup = self._scatter(torch.cat([ga, torch.ones_like(ga[:, :1])], 1), offsets=(-1, 0, 1, 2), weighted=False)
        G, K = sup[:, 0:3], sup[:, 3:4] + 2.0
        S = ga + P + tr_ga
        out = out_scale * (g + pos + tr_g)
        bound = out_scale * (U24 * SO * ((K + 16.0) * S + 3.0 * (self.n + 1) * G) + b + pos_b + tr_b)
        return out.view(self.shape), bound.view(self.shape), (out_scale * S).view(self.shape)


def fwd_step(u, in_scale):
    """(out64, bound): one squaring step u + s trilinear[u](clamp(x + u s)), decisions from u's own precision"""
    return Step(u, in_scale).fwd()


def bwd_step(u, in_scale, g, out_scale, g_err=None):
    """(g_out64, bound): the adjoint of one step (direct + position term + interpolation transpose) times out_scale"""
    out, bound, _ = Step(u, in_scale).bwd(g, out_scale, g_err)
    return out, bound


def abs_sum(u, in_scale, g, out_scale):
    """S(t): the adjoint step's sum taken over the magnitudes of its terms (times out_scale)"""
    return Step(u, in_scale).bwd(g, out_scale)[2]


def compose(v, hist, g, n_steps):
    """the whole adjoint over a GIVEN forward history (hist[k] = output of step k); returns (g_v64, propagated bound)"""
    b = None
    scale0 = 2.0 ** -n_steps
    for k in range(n_steps - 1, -1, -1):
        u, s = (v, scale0) if k == 0 else (hist[k - 1], 1.0)
        g, b = bwd_step(u, s, g, s, b)
    return g, b


# ---- the maxabs block ----------------------------------------------------------------------------------------------------
def cells_shape(D, H, W):
    return math.ceil(D / CELL_Z), math.ceil(H / CELL_Y), math.ceil(W / CELL_X)


def maxabs_floats(C, D, H, W, n_steps):
    nz, ny, nx = cells_shape(D, H, W)
    return n_steps * (1 + C * nz * ny * nx)


def split_maxabs(block, n_steps, C, D, H, W):
    """views (globals (n_steps,), maps (n_steps, C, nz, ny, nx)) of a maxabs block"""
    nz, ny, nx = cells_shape(D, H, W)
    return block[:n_steps], block[n_steps:].view(n_steps, C, nz, ny, nx)


def max_abs(u, in_scale):
    """max |u in_scale| over every chain, voxel and component, as the fp32 value the forward kernels leave"""
    return (u.float() * in_scale).abs().amax()


def cell_map(u, in_scale):
    """(C, nz, ny, nx) fp32 maxima of |u in_scale| over cells of 32 x 8 x 8 voxels"""
    C, _, D, H, W = u.shape
    nz, ny, nx = cells_shape(D, H, W)
    a = (u.float() * in_scale).abs().amax(dim=1)
    a = F.pad(a, (0, nx * CELL_X - W, 0, ny * CELL_Y - H, 0, nz * CELL_Z - D))
    return a.view(C, nz, CELL_Z, ny, CELL_Y, nx, CELL_X).amax(dim=(2, 4, 6))


def gather_radius(m):
    """svf_gather_radius: floor(m + 1e-3) + 1 evaluated in fp32"""
    import numpy as np
    return int(np.floor(np.float32(m) + np.float32(1e-3))) + 1


def worst(out, ref, bound):
    """(number of voxels outside the bound, index of the worst one, its |difference| / bound) for failure messages"""
    d = (out.double() - ref.double()).abs()
    bad = ~(d <= bound)   # NaN counts as outside
    ratio = torch.where(bad & ~(d < float('inf')), float('inf'), d / bound.clamp_min(1e-300))
    i = int(torch.argmax(ratio))
    return int(bad.sum()), tuple(int(x) for x in torch.unravel_index(torch.tensor(i), out.shape)), float(ratio.flatten()[i])


# ---- test inputs ---------------------------------------------------------------------------------------------------------
def threshold_field(n, C, seed=0):
    """U with |U| < 0.7 plus, at voxels on tile edges (x = 0, 31, 32, n - 1; y = 7, 8, 15, 16), the values where the
    kernels decide: the TMA forward's 0.999 fallback, the 1 and 2 voxel windows, integers, halves, and positions landing
    exactly on 0 or n - 1 or rounding onto n - 1 in fp32"""
    U = _smooth_field((C, 3, n, n, n), 0.7, seed)
    vals = [0.999, -0.999, 0.9989999, -0.9989999, 1.0, -1.0, 1.999, -1.999, 2.0, -2.0, 3.0, -3.0, 0.5, -0.5, 0.0]
    xs = sorted({0, 1, min(31, n - 1), min(32, n - 1), n - 2, n - 1})
    ys = sorted({0, min(7, n - 1), min(8, n - 1), min(15, n - 1), min(16, n - 1), n - 1})
    i = 0
    for c in range(C):
        for z in (0, n // 2, n - 1):
            for y in ys:
                for x in xs:
                    a = i % 3
                    U[c, a, z, y, x] = vals[(i * 7 + c) % len(vals)]
                    i += 1
        for x in range(n):   # p = 0 and p = n - 1 exactly along x
            U[c, 0, 1, 2, x] = -float(x)
            U[c, 0, 2, 3, x] = float(n - 1 - x)
        for z in range(n):   # the same along z
            U[c, 2, z, 4, 5] = -float(z) if c == 0 else float(n - 1 - z)
        # fl32(n - 2 + (1 - 2^-23)) rounds onto n - 1: inside() turns false although x + u < n - 1
        U[c, 1, 5, n - 2, 6] = 1.0 - 2.0 ** -23
        U[c, 0, 6, 7, n - 2] = 1.0 - 2.0 ** -23
        U[c, 2, n - 2, 8, 9] = 1.0 - 2.0 ** -23
        U[c, 0, 7, 9, 1] = -(1.0 - 2.0 ** -23)   # fl32(1 - (1 - 2^-23)) = 2^-23: exact, stays inside
    return U.float().contiguous()
